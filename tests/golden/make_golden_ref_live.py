"""Writes tests/golden/ref_live_balm.npz and tests/golden/ref_live_system.npz: what the reference's own source returns for every case
of the ref_* functions in tests/test_ref_pin.py and tests/test_ref_system_pin.py.  Those tests hold the oracles, the C++ port and
the device passes against these files, so they run without the reference.

The calls need oracle/_ref/ (the reference's sources compiled where they lie, oracle/Makefile `make ref`):
    LVBA_REFERENCE=<checkout of the original Global-LVBA sources> python __graft_entry__.py
    python tests/golden/make_golden_ref_live.py

The cases run in the order the tests run: LvbaSystem keeps its eigen-ratio array process-wide (bavoxel.hpp:17), so a call
sees what the calls before it set.
"""
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]


def store(out, tag, result):
    for k, v in result.items():
        out[f"{tag}__{k}"] = np.asarray(v)


def generate():
    import test_ref_pin as rp
    import test_ref_system_pin as rs
    from oracle import balm_ref, lvba_system_ref
    assert balm_ref.available() and lvba_system_ref.available(), "oracle/_ref/ is missing: build with LVBA_REFERENCE set"
    balm = {}
    for W, V, seed in rp.HESSIAN_CASES:
        store(balm, f"hessian_{seed}", rp.ref_hessian(W, V, seed))
    for seed, voxel_size in rp.VOXEL_MAP_CASES:
        store(balm, f"voxel_map_{seed}", rp.ref_voxel_map(seed, voxel_size))
    system = {}
    for seed, W, win, use_rel, stage1, _ in rs.RAGGED_CASES:
        store(system, f"lidar_ba_{seed}", rs.ref_lidar_ba(seed, W, win, use_rel, stage1))
    store(system, "container_order", rs.ref_container_order())
    store(system, "colmap_db_reader", rs.ref_colmap_db_reader())
    store(system, "dataset_loader", rs.ref_dataset_loader())
    store(system, "track_helpers", rs.ref_track_helpers())
    for seed, kw in rs.FUSION_CASES:
        store(system, f"build_tracks_{seed}", rs.ref_build_tracks(seed, kw))
    for seed, F, M, size in rs.DEPTH_CASES:
        store(system, f"depth_{seed}", rs.ref_depth(seed, F, M, size))
    store(system, "colmap_export", rs.ref_colmap_export())
    store(system, "lidar_ba_41", rs.ref_lidar_ba(41, 6, 10, False, True, window_stage=False))
    store(system, "bucket_counts", rs.ref_bucket_counts())
    return {rp.LIVE: balm, rs.LIVE: system}


if __name__ == "__main__":
    for path, arrays in generate().items():
        np.savez_compressed(path, **arrays)
        print(f"{path.name}: {len(arrays)} arrays, {path.stat().st_size} bytes")
