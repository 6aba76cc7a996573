"""The stage oracles, pinned against the REFERENCE'S PIPELINE SOURCE (src/lvba_system.cpp; SURVEY.md §8c, §8f N1-N4).

tests/golden/ref_system.npz holds seeded inputs and what LvbaSystem's own member functions computed from them — runWindowBA,
runLidarBA, buildGridMapFromOptimized, updateCameraPosesFromLidar, generateDepthWithVoxel, BuildTracksAndFuse3D and the Ceres problem
optimizeCameraPoses builds — with the whole of src/lvba_system.cpp compiled where it lies (oracle/ref_system_driver.cpp) on the
stand-in library headers of oracle/ref_shim/ (own code; what that leaves open: ref_shim/mini_eigen.h, DESIGN.md §2).  Without a GPU:

  L  the oracle chain the offline tool is tested against (voxel map + damping_iter per window with the 3-voxels-per-pose skip rule,
     anchor clouds, relative poses, two global stages, pose of every frame from its anchor) reproduces the reference's runLidarBA
  D  the numpy restatement of the camera-pose correction and oracle/depth_oracle.py reproduce the reference's camera poses and its
     depth images BIT FOR BIT; the device's depth passes, run through the host policy, do too
  F  oracle/fuse_oracle.py reproduces BuildTracksAndFuse3D track for track — same track order, observation order, inlier order,
     points to 1e-12 — once it is told the order the reference's three `for (auto& kv : unordered_map)` loops run in.  C++ leaves
     that order open; with g++ it is libstdc++'s, restated in fuse_oracle.libstdcxx_order and held against the real container here.
     The ABI of this repo documents ASCENDING image id instead; on this scene the two orders give 70 vs 63 tracks — the choice matters,
     and it is a property of the reference's container, not of the restatement (DESIGN.md §4.5)
  P  the problem the reference hands to Ceres: camera 0 constant (q and t), EigenQuaternionManifold on every camera, no loss function,
     sigma 0.5 px / 0.01 m, 50 iterations DENSE_SCHUR, default tolerances; the points that enter are exactly the usable tracks with a
     valid plane, their planes those of the voxel oracle on the oracle's anchor clouds (live test: the scene is rebuilt, not stored)

The tests named *_live_* / *differential* / *reference_reader* / *reference_loader* / *real_container* / *reference_writer* compare with
what the reference source computed from their inputs, stored in tests/golden/ref_live_system.npz by tests/golden/make_golden_ref_live.py
(the ref_* functions below make those calls).  Where oracle/_ref/liblvba_system_ref.so is built, ref_system.npz is also regenerated and
must come out bit for bit.
"""
import os
import sys
import tempfile
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "tests"))

from oracle import anchor_oracle as ao, depth_oracle as dep, fuse_oracle as fo, lidar_oracle as lo, lvba_system_ref as sr, synth, visual_oracle as vis, voxel_oracle as vox  # noqa: E402
import test_depth_emu  # noqa: E402

G = np.load(ROOT / "tests" / "golden" / "ref_system.npz")
LIVE = ROOT / "tests" / "golden" / "ref_live_system.npz"
needs_ref = pytest.mark.skipif(not sr.available(), reason="oracle/_ref/liblvba_system_ref.so is built only where the original sources are readable")


def recorded(tag):
    """What the ref_* function of case `tag` returned when the fixture was written."""
    with np.load(LIVE) as f:
        return {k[len(tag) + 2:]: f[k] for k in f.files if k.startswith(tag + "__")}


def flat(arrays):
    """A list of arrays as (concatenation, CSR pointer)."""
    return np.concatenate(arrays), np.r_[0, np.cumsum([len(a) for a in arrays])]


def split(flat, ptr):
    return [flat[ptr[i]:ptr[i + 1]] for i in range(len(ptr) - 1)]


def lex(a):
    return a[np.lexsort(a.T[::-1])]


# ------------------------------------------------------------------------------------------------ L
def lidar_chain(use_rel, scans=None, start=None, win=None, leaf=None, s1=None, s2=None, stage1=True):
    """runWindowBA (src/lvba_system.cpp:204-302) + runLidarBA (:304-409) out of the stage oracles.  Defaults: section L of the fixture."""
    if scans is None:
        scans = split(G["L_xyz"], G["L_scan_ptr"]); start = G["L_poses"]; win = int(G["L_window"]); leaf = float(G["L_anchor_leaf"])
        s1 = (float(G["L_s1_voxel"]), G["L_s1_ratio"]); s2 = (float(G["L_s2_voxel"]), G["L_s2_ratio"])
    W = len(scans)
    win_ptr = list(range(0, W, win)) + [W]
    anchor_index = np.full(W, -1, np.int32); rel = np.zeros((W, 12)); rel[:, [0, 4, 8]] = 1.0      # IMUST(): identity, zero
    anchors, clouds = [], []
    for w in range(len(win_ptr) - 1):
        a, b = win_ptr[w], win_ptr[w + 1]
        vp, pi, cl, _ = vox.voxelize(scans[a:b], start[a:b], s1[0], vox.EIGEN_RATIO_DEFAULT)                # :247-258: stage-1 SIZE, but the plane test reads
        #                                       the process-wide array, which still holds bavoxel.hpp:17's default here (the configured arrays are set at :358, later)
        if len(vp) - 1 < 3 * (b - a):                                                                      # :259-263
            continue
        x_win, _ = lo.damping_iter(vp, pi, cl, start[a:b])                                                 # :264
        aligned = start[a:b].copy()
        if use_rel:                                                                                        # :267-279
            R_align = start[a, :9].reshape(3, 3) @ x_win[0, :9].reshape(3, 3).T
            p_align = start[a, 9:] - R_align @ x_win[0, 9:]
            for j in range(b - a):
                aligned[j, :9] = (R_align @ x_win[j, :9].reshape(3, 3)).ravel(); aligned[j, 9:] = R_align @ x_win[j, 9:] + p_align
        r = rel_to(start[a], aligned)                                                                      # :283-289: anchor = the ODOMETRY pose of frame 0
        rel[a:b] = r; anchor_index[a:b] = len(anchors)
        clouds.append(ao.anchor_clouds(scans[a:b], r, np.array([0, b - a]), leaf)[0])
        anchors.append(start[a])
    anchors = np.array(anchors)
    for vs_, er in ([s1] if stage1 else []) + [s2]:                                                        # :355-389 (stage 1 only if BALM_stage1/enable)
        vp, pi, cl, _ = vox.voxelize(clouds, anchors, vs_, er)
        anchors, _ = lo.damping_iter(vp, pi, cl, anchors)
    final = start.copy()
    for i in range(W):                                                                                     # :393-403
        k = anchor_index[i]
        if k < 0:
            continue
        A = anchors[k, :9].reshape(3, 3)
        final[i, :9] = (A @ rel[i, :9].reshape(3, 3)).ravel(); final[i, 9:] = A @ rel[i, 9:] + anchors[k, 9:]
    return anchor_index, rel, clouds, final


def rel_to(anchor, poses):
    """rel.R = anchor.R^T x.R ; rel.p = anchor.R^T (x.p - anchor.p)  (:286-289)."""
    Ra = anchor[:9].reshape(3, 3); out = np.zeros_like(poses)
    for j in range(len(poses)):
        out[j, :9] = (Ra.T @ poses[j, :9].reshape(3, 3)).ravel(); out[j, 9:] = Ra.T @ (poses[j, 9:] - anchor[9:])
    return out


def test_window_stage_anchor_bookkeeping_equals_reference_source():
    idx, rel, clouds, _ = lidar_chain(False)
    assert np.array_equal(idx, G["L_anchor_index"]) and idx.tolist() == [0, 0, 0, -1, -1, -1, 1, 1, 1]      # the middle window is skipped
    assert np.abs(rel - G["L_rel_poses"]).max() <= 1e-12
    ref_clouds = split(G["L_anchor_clouds_sorted"], G["L_anchor_cloud_ptr"])
    assert len(clouds) == len(ref_clouds) == 2
    for c, r in zip(clouds, ref_clouds):
        assert np.array_equal(lex(c), r)                                                                   # float32 points, bit for bit
    # use_window_ba_rel: the relative poses now carry the window solves themselves (damping_iter per window, aligned to the anchor)
    _, rel_w, clouds_w, _ = lidar_chain(True)
    assert np.abs(rel_w - G["L_rel_poses_rel"]).max() <= 1e-10 and np.abs(G["L_rel_poses_rel"] - G["L_rel_poses"]).max() > 1e-3
    assert np.array_equal(rel_w[3:6], np.tile(np.r_[np.eye(3).ravel(), np.zeros(3)], (3, 1)))               # skipped window: IMUST() stays
    got = np.concatenate([lex(c) for c in clouds_w])
    assert got.shape == G["L_anchor_clouds_rel_sorted"].shape
    assert np.mean(np.all(got == G["L_anchor_clouds_rel_sorted"], axis=1)) > 0.99                           # float32 of poses equal to 1e-11: a last-bit flip here and there
    assert np.array_equal(G["L_anchor_poses"], G["L_poses"][[0, 6]])                                        # anchors keep the odometry pose (:283)


@pytest.mark.parametrize("use_rel", [False, True])
def test_lidar_half_equals_reference_source(use_rel):
    _, _, _, final = lidar_chain(use_rel)
    ref = G["L_final_poses_rel"] if use_rel else G["L_final_poses"]
    assert np.abs(final - ref).max() <= 1e-9
    assert np.array_equal(ref[3:6], G["L_poses"][3:6])                    # frames of the skipped window keep their odometry pose (:396)
    assert np.abs(ref - G["L_poses"]).max() > 1e-3                        # the others moved
    if use_rel:
        assert np.abs(G["L_final_poses_rel"] - G["L_final_poses"]).max() > 1e-5       # the switch does something


RAGGED_CASES = [(31, 10, 4, False, True, [0, 0, 0, 0, 1, 1, 1, 1, 2, 2]), (32, 10, 4, True, True, [0, 0, 0, 0, 1, 1, 1, 1, 2, 2]),
                (33, 7, 3, True, False, [0, 0, 0, 1, 1, 1, -1])]
S1R = np.array([0.3, 0.1, 0.06, 0.03], np.float32)
S2R = np.array([0.08] * 4, np.float32)


def noisy_scan_scene(seed, W):
    scans, poses = synth.make_scan_scene(seed, W=W, n_per_scan=2500)
    rng = np.random.default_rng(seed)
    noisy = poses.copy()
    for i in range(W):
        noisy[i, :9] = (noisy[i, :9].reshape(3, 3) @ synth.so3_exp(rng.normal(0, 0.004, (1, 3)))[0]).ravel(); noisy[i, 9:] += rng.normal(0, 0.01, 3)
    return scans, noisy


def ref_lidar_ba(seed, W, win, use_rel, stage1, window_stage=True):
    """The reference's runLidarBA on noisy_scan_scene(seed, W)."""
    scans, noisy = noisy_scan_scene(seed, W)
    sr.set_eigen_ratio_array(S1R)                                  # a fresh process: bavoxel.hpp:17
    S = sr.System()
    S.set_lidar(scans, noisy)
    S.set_stages(window_stage, win, 0.1, use_rel, stage1, 1.0, S1R, 0.5, S2R)
    out = S.run_lidar_ba()
    S.close()
    return dict(poses=out)


@pytest.mark.parametrize("seed,W,win,use_rel,stage1,index", RAGGED_CASES)
def test_lidar_half_live_ragged_windows_and_stage_switches(seed, W, win, use_rel, stage1, index):
    """A last window shorter than the others, a last window of ONE frame (no voxel can see two poses: skipped, its frame keeps the odometry pose),
    BALM_stage1/enable = false, both settings of use_window_ba_rel: the reference's runLidarBA against the oracle chain."""
    scans, noisy = noisy_scan_scene(seed, W)
    out = recorded(f"lidar_ba_{seed}")["poses"]
    idx, _, _, final = lidar_chain(use_rel, scans, noisy, win, 0.1, (1.0, S1R), (0.5, S2R), stage1)
    assert idx.tolist() == index
    assert np.abs(out - final).max() <= 1e-9 and np.abs(out - noisy).max() > 1e-3


# ------------------------------------------------------------------------------------------------ D
def camera_chain():
    """updateCameraPosesFromLidar (:412-446) and the extrinsics of initFromDatasetIO (:497-503) / generateDepthWithVoxel (:861-862)."""
    opt, before, ts = G["D_poses"], G["D_poses_before"], G["D_frame_ts"]
    body = np.zeros_like(G["D_image_poses"])
    for i, t_img in enumerate(G["D_image_ts"]):
        it = int(np.searchsorted(ts, t_img, side="left"))                 # std::lower_bound
        idx = len(ts) - 1 if it == len(ts) else it
        if 0 < it < len(ts) and abs(ts[idx - 1] - t_img) < abs(ts[idx] - t_img):
            idx -= 1
        Ro, po = opt[idx, :9].reshape(3, 3), opt[idx, 9:]; Rb, pb = before[idx, :9].reshape(3, 3), before[idx, 9:]
        Rd = Ro @ Rb.T; pd = Ro @ (-(Rb.T @ pb)) + po                     # T_opt * T_orig^-1
        Rc, pc = G["D_image_poses"][i, :9].reshape(3, 3), G["D_image_poses"][i, 9:]
        body[i, :9] = (Rd @ Rc).ravel(); body[i, 9:] = Rd @ pc + pd
    Rli = G["D_Ril"].T; tli = -Rli @ G["D_til"]
    Rci = G["D_Rcl"] @ Rli; tci = G["D_Rcl"] @ tli + G["D_tcl"]
    cams = np.zeros_like(body)
    for i in range(len(body)):
        Rcw = Rci @ body[i, :9].reshape(3, 3).T
        cams[i, :9] = Rcw.ravel(); cams[i, 9:] = -Rcw @ body[i, 9:] + tci
    return body, cams


def test_camera_poses_from_the_lidar_result_equal_reference_source():
    body, cams = camera_chain()
    assert np.abs(body - G["D_camera_body_poses"]).max() <= 1e-12
    assert np.abs(cams - G["D_cams"]).max() <= 1e-12
    assert np.abs(G["D_cams"] - G["D_cams_odometry"]).max() > 1e-3        # the LiDAR correction moved the cameras


def depth_scene():
    return dict(scans=split(G["D_xyz"], G["D_scan_ptr"]), poses=G["D_poses"], frame_ts=G["D_frame_ts"], cams=G["D_cams"], image_ts=G["D_image_ts"],
                intr=G["D_intr"], width=int(G["D_size"][0]), height=int(G["D_size"][1]))


@pytest.mark.parametrize("literal", [False, True])
def test_depth_images_equal_reference_source_bit_for_bit(literal):
    s = depth_scene()
    fn = dep.render_literal if literal else dep.render
    img = fn(s["scans"], s["poses"], s["frame_ts"], s["cams"], s["image_ts"], s["intr"], s["width"], s["height"])
    assert np.array_equal(img, G["D_depth"]) and int((G["D_depth"] > 0).sum()) > 5000


def test_device_depth_passes_equal_reference_source_bit_for_bit(tmp_path_factory):
    import ctypes
    import subprocess
    so = tmp_path_factory.mktemp("emu_ref_sys") / "libdepth_emu.so"
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", str(ROOT / "tests" / "emu" / "depth_emu.cpp"), "-o", str(so)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rc, img, info = test_depth_emu.emu_render(ctypes.CDLL(str(so)), depth_scene())
    assert rc == 0 and info["pairs"] > 0
    assert np.array_equal(img, G["D_depth"])


# ------------------------------------------------------------------------------------------------ F
def fuse_inputs():
    kp_ptr, kp_uv = G["F_kp_ptr"], G["F_kp_uv"]
    Xw, valid = dep.backproject(list(G["F_depth"]), G["F_cams"], G["F_intr"], kp_ptr, kp_uv)
    return kp_ptr, kp_uv, G["F_matches"], G["F_cams"], G["F_intr"], Xw, valid


def test_track_fusion_equals_reference_source_under_its_container_order():
    tr = fo.fuse(*fuse_inputs(), map_order=fo.libstdcxx_order)
    assert len(tr) == len(G["F_Xw"]) == 70
    for k, t in enumerate(tr):
        ob = G["F_obs"][G["F_obs_ptr"][k]:G["F_obs_ptr"][k + 1]]
        assert np.array_equal(t["obs"], ob), k                                                  # same component, same member order
        assert list(t["kept"]) == G["F_inl"][G["F_inl_ptr"][k]:G["F_inl_ptr"][k + 1]].tolist(), k     # same inliers in the same order
        assert np.abs(t["Xw"] - G["F_Xw"][k]).max() <= 1e-12, k


def test_device_fusion_pass_equals_reference_source_under_its_container_order(tmp_path_factory):
    """csrc/fuse_pipeline.h (host component walk + rounds + the per-component device functor) through the host policy with
    map_order = LVBA_FUSE_ORDER_LIBSTDCXX against what the reference's own BuildTracksAndFuse3D produced."""
    import ctypes
    import subprocess
    import test_fuse_emu
    so = tmp_path_factory.mktemp("emu_ref_fuse") / "libfuse_emu.so"
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", str(ROOT / "tests" / "emu" / "fuse_emu.cpp"), "-o", str(so)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = ctypes.CDLL(str(so)); lib.fuse_emu_run.restype = ctypes.c_longlong
    kp_ptr, kp_uv, matches, cams, intr, Xw, valid = fuse_inputs()
    got = test_fuse_emu.run_emu(lib, dict(kp_ptr=kp_ptr, kp_uv=kp_uv, matches=matches, cams=cams, intr=intr, kp_Xw=Xw, kp_valid=valid), map_order=1)
    assert len(got["seed"]) == len(G["F_Xw"]) == 70
    for k in range(70):
        a, b = got["obs_ptr"][k], got["obs_ptr"][k + 1]
        ob = G["F_obs"][G["F_obs_ptr"][k]:G["F_obs_ptr"][k + 1]]
        assert np.array_equal(np.column_stack([got["img"][a:b], got["kp"][a:b]]), ob), k
        inl = np.zeros(b - a, bool); inl[G["F_inl"][G["F_inl_ptr"][k]:G["F_inl_ptr"][k + 1]]] = True
        assert np.array_equal(got["inlier"][a:b].astype(bool), inl), k
        assert np.abs(got["Xw"][k] - G["F_Xw"][k]).max() <= 1e-9, k
    asc = test_fuse_emu.run_emu(lib, dict(kp_ptr=kp_ptr, kp_uv=kp_uv, matches=matches, cams=cams, intr=intr, kp_Xw=Xw, kp_valid=valid), map_order=0)
    assert len(asc["seed"]) == 63                                                  # the documented default order: another answer on this scene


def test_ascending_order_is_a_different_but_documented_choice():
    """The ABI's library-independent alternative (LVBA_FUSE_ORDER_ASCENDING) against what the reference's container does under g++ (the default): same
    logic, other visiting order."""
    tr = fo.fuse(*fuse_inputs(), map_order=fo.ascending_order)
    ref = {tuple(map(tuple, G["F_obs"][G["F_obs_ptr"][k]:G["F_obs_ptr"][k + 1]].tolist())) for k in range(len(G["F_Xw"]))}
    mine = {tuple(map(tuple, sorted(t["obs"].tolist()))) for t in tr}
    assert len(tr) == 63 and mine <= {tuple(sorted(r)) for r in ref}                            # every ascending-order track is a reference track


def container_order_cases():
    rng = np.random.default_rng(0)
    for _ in range(2000):
        res = int(rng.integers(1, 60))
        yield res, rng.choice(90, size=int(rng.integers(1, min(res, 40) + 1)), replace=False).tolist()


def ref_container_order():
    """The order std::unordered_map (reserve(res), then the keys inserted) visits its keys in, for every case."""
    order, ptr = flat([np.array(sr.unordered_map_order(res, keys), np.int8) for res, keys in container_order_cases()])
    return dict(order=order, ptr=ptr)


def test_libstdcxx_order_restatement_equals_the_real_container():
    R = recorded("container_order")
    for k, (res, keys) in enumerate(container_order_cases()):
        assert R["order"][R["ptr"][k]:R["ptr"][k + 1]].tolist() == fo.libstdcxx_order(res, keys), (res, keys)
    assert k + 1 == len(R["ptr"]) - 1


# ------------------------------------------------------------------------------------------------ P
def test_problem_handed_to_ceres():
    assert G["P_cam_const"].tolist() == [3] + [0] * 7                     # q AND t of camera 0 constant (:1582-1583), nothing else
    assert np.all(G["P_cam_manifold"] == 1)                               # EigenQuaternionManifold on every camera, also the constant one (:1579)
    assert not G["P_obs_loss"].any() and not G["P_pl_loss"].any()         # the two HuberLoss objects are created (:1585-1586) and never passed (:1630, :1639)
    assert np.all(G["P_obs_sigma"] == 0.5) and np.all(G["P_pl_sigma"] == 0.01)
    assert G["P_options"].tolist() == [50.0, 3.0, 1e-6, 1e-10, 1e-8]       # max_num_iterations, DENSE_SCHUR, function / gradient / parameter tolerance
    assert np.all(G["P_obs_intr"] == G["F_intr"][None])
    assert np.array_equal(G["P_pl_pt"], np.arange(len(G["P_X"])))         # one plane residual per point block, in order
    assert np.all(np.diff(G["P_obs_pt"]) >= 0) and set(G["P_obs_pt"].tolist()) == set(range(len(G["P_X"])))
    n = np.linalg.norm(G["P_pl_nd"][:, :3], axis=1)
    assert np.abs(n - 1).max() <= 1e-12
    # the parameter blocks start from the cameras / fused points of the stages before
    q = G["P_q"]; R = vis.quat_to_rot(q)
    assert np.abs(R.reshape(-1, 9) - G["F_cams"][:, :9]).max() <= 1e-12 and np.abs(G["P_t"] - G["F_cams"][:, 9:]).max() == 0
    assert np.abs(np.linalg.norm(q, axis=1) - 1).max() <= 1e-15           # q_eig.normalize() (:1515); the sign of q is the library's branch, no result depends on it
    # every point block is a fused track, every observation one of its INLIERS with the keypoint's pixel as the measurement
    for j, X in enumerate(G["P_X"]):
        k = int(np.nonzero(np.all(G["F_Xw"] == X, axis=1))[0][0])
        ob = G["F_obs"][G["F_obs_ptr"][k]:G["F_obs_ptr"][k + 1]]; inl = G["F_inl"][G["F_inl_ptr"][k]:G["F_inl_ptr"][k + 1]]
        rows = np.nonzero(G["P_obs_pt"] == j)[0]
        assert G["P_obs_cam"][rows].tolist() == ob[inl, 0].tolist()
        uv = np.array([G["F_kp_uv"][G["F_kp_ptr"][c] + kp] for c, kp in ob[inl]], np.float64)
        assert np.array_equal(G["P_obs_uv"][rows], uv)


def test_points_and_planes_of_the_problem_against_the_oracle_chain_live():
    """Rebuilds the scene (2.9 MB of scans, not stored): usable tracks (:1432-1438), anchor clouds (:1471-1490), surf map under the eigen-ratio array
    in force (:1498-1506), recompute_local_planes (:1529-1566) out of the stage oracles vs what the reference recorded."""
    import visual_scene as vs
    g = vs.make(Path(tempfile.mkdtemp()), seed=3, W=8)
    win, leaf = int(G["P_window"]), float(G["P_anchor_leaf"])
    win_ptr = np.array(list(range(0, 8, win)) + [8])
    rel = ao.rel_poses(g["poses"], win_ptr)
    clouds = ao.anchor_clouds(g["scans"], rel, win_ptr, leaf)
    roots = vox.build_tree_literal(clouds, g["poses"][win_ptr[:-1]], float(G["P_voxel"]), G["P_ratio"])
    usable = [k for k in range(len(G["F_Xw"])) if G["F_obs_ptr"][k + 1] - G["F_obs_ptr"][k] >= 3 and np.all(np.isfinite(G["F_Xw"][k])) and not np.all(np.abs(G["F_Xw"][k]) <= 1e-12)]
    nd = vox.plane_lookup_literal(roots, G["F_Xw"][usable], float(G["P_voxel"]))
    has = vis.valid_tracks(nd)
    assert np.array_equal(G["F_Xw"][np.array(usable)[has]], G["P_X"])                            # the same tracks enter, in the same order
    sgn = np.sign(np.einsum("ij,ij->i", nd[has][:, :3], G["P_pl_nd"][:, :3]))
    assert np.abs(nd[has] * sgn[:, None] - G["P_pl_nd"]).max() <= 1e-9                          # plane (n, d) up to the eigenvector's sign


# ------------------------------------------------------------------------------------------------ the file itself
@needs_ref
def test_fixture_is_what_the_reference_pipeline_source_computes_bit_for_bit():
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    import make_golden_ref_system
    fresh = make_golden_ref_system.generate()
    assert sorted(fresh) == sorted(G.files)
    exact = True
    for k in G.files:
        a, b = np.asarray(fresh[k]), G[k]
        if a.dtype.kind in "iub":
            assert np.array_equal(a, b), k                                  # counts, keys, indices, flags: always
        elif a.shape != b.shape:                                            # a down-sampled cloud behind an LM solve: a tie may fall the other way
            assert a.ndim == b.ndim and abs(len(a) - len(b)) <= max(2, len(b) // 200), k
            exact = False
        else:
            same = np.array_equal(a, b, equal_nan=True)
            exact = exact and same
            if not same:                                                    # another host CPU (libm / BLAS kernels pick FMA variants at run time)
                if k.endswith("_sorted"):
                    assert np.mean(np.all(a == b, axis=1)) > 0.99, k
                else:
                    assert np.allclose(a, b, rtol=1e-9, atol=1e-11, equal_nan=True), k
    assert exact or os.environ.get("LVBA_ALLOW_OTHER_HOST", "1") == "1"     # on the machine that wrote the file the regeneration is bit for bit


@needs_ref
def test_live_fixtures_are_what_the_reference_source_computes():
    """tests/golden/ref_live_balm.npz and ref_live_system.npz, which the *_live_* / differential / reader / loader / writer tests of this file
    and of tests/test_ref_pin.py compare with, recomputed from the reference source by tests/golden/make_golden_ref_live.py."""
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    import make_golden_ref_live
    for path, fresh in make_golden_ref_live.generate().items():
        with np.load(path) as stored:
            assert sorted(fresh) == sorted(stored.files), path.name
            for k in stored.files:
                a, b = np.asarray(fresh[k]), stored[k]
                if a.dtype.kind in "iubU":
                    assert np.array_equal(a, b), k                          # counts, keys, indices, flags, text: always
                else:                                                       # another host CPU may round the last bits differently
                    assert a.shape == b.shape and np.allclose(a, b, rtol=1e-9, atol=1e-11, equal_nan=True), k


# ------------------------------------------------------------------------------------------------ N4: the COLMAP database reader
def colmap_db_scene(root):
    import visual_scene as vs
    return vs.make(root, seed=5, W=6, n_per_scan=4000, n_landmarks=120)


def ref_colmap_db_reader():
    import visual_scene as vs
    root = Path(tempfile.mkdtemp())
    g = colmap_db_scene(root)
    S = sr.System()
    S.set_lidar(g["scans"][:1], g["poses"][:1], g["ts"][:1])
    S.set_camera(g["width"], g["height"], g["intr"], vs.RCL.ravel(), vs.PCL, np.eye(3).ravel(), np.zeros(3), np.array(g["image_ts"]), g["image_poses"])
    ok, kp_ptr, kp_uv, m = S.load_colmap_db(str(root) + "/", root / "Colmap" / "colmap.db")
    S.close()
    return dict(ok=ok, kp_ptr=kp_ptr, kp_uv=kp_uv, matches=m)


def test_reference_reader_reads_the_database_the_dataset_writer_writes():
    """loadFromColmapDB (src/lvba_system.cpp:510-685, run from its own source against the system's SQLite) on the database
    oracle/dataset_writer.py wrote: database ids shuffled (so some pairs are stored with swapped columns, :655-660), one match with an
    out-of-range keypoint (dropped, :668-672).  It must hand back exactly the scene's keypoints and matches in the order
    BuildTracksAndFuse3D visits them — the same truth tests/test_visual_offline.py holds the product's own reader
    (global-lvba_b200/host/lvba_visual_offline.hpp) against."""
    g = colmap_db_scene(Path(tempfile.mkdtemp()))
    assert sorted(g["db_ids"]) != g["db_ids"]
    R = recorded("colmap_db_reader")
    ok, kp_ptr, kp_uv, m = bool(R["ok"]), R["kp_ptr"], R["kp_uv"], R["matches"]
    assert ok
    assert np.array_equal(np.diff(kp_ptr), [len(k) for k in g["keypoints"]]) and np.array_equal(kp_uv, np.concatenate(g["keypoints"]))
    M = len(g["keypoints"])
    want = [(a, ka, b, kb) for a in range(M) for b in range(a + 1, M) for (ka, kb) in g["pair"].get((a, b), [])
            if ka < len(g["keypoints"][a]) and kb < len(g["keypoints"][b])]
    dropped = sum(len(v) for v in g["pair"].values()) - len(want)
    assert dropped == 1 and np.array_equal(m, np.array(want, np.int32))


# ------------------------------------------------------------------------------------------------ N4: the dataset loader
def loader_dataset(root):
    """The dataset the loader test reads, written under root; returns what was written."""
    from oracle import dataset_writer as dw
    scans, poses = synth.make_scan_scene(3, W=7, n_per_scan=900)
    scans[4] = scans[4][:0]                                              # an empty scan file
    ts = dw.write_lidar_dataset(root, scans, poses)                       # binary, ascii and LZF-compressed PCD files in turn
    (root / "all_pcd_body" / "notes.txt").write_text("ignored")
    image_ts = [t + 0.013 for t in ts]
    image_poses = poses.copy(); image_poses[:, 9:] += np.random.default_rng(1).normal(0, 0.02, (7, 3))
    dw.write_image_set(root, image_ts, image_poses, extra_between=1)
    return scans, poses, ts, image_ts, image_poses


def ref_dataset_loader():
    """What DatasetIO's constructor read; its two paths with the dataset's directory taken off the front."""
    root = Path(tempfile.mkdtemp())
    loader_dataset(root)
    S = sr.System({"data_config/data_path": str(root) + "/", "data_config/colmap_db_path": "Colmap/colmap.db", "data_config/image_sample_step": 2,
                   "cam_model/cam_width": 160, "cam_model/cam_height": 128, "cam_model/scale": 0.5, "cam_model/cam_fx": 96.0, "cam_model/cam_fy": 96.3,
                   "cam_model/cam_cx": 79.7, "cam_model/cam_cy": 64.2})
    d = S.dataset()
    S.close()
    assert d["data_path"].startswith(str(root)) and d["db_path"].startswith(str(root))
    xyz, scan_ptr = flat(d.pop("scans"))
    return dict(d, scans_xyz=xyz, scan_ptr=scan_ptr, data_path=d["data_path"][len(str(root)):], db_path=d["db_path"][len(str(root)):])


def test_reference_loader_reads_the_dataset_the_dataset_writer_writes():
    """DatasetIO's constructor (src/dataset_io.cpp, run from its own source; PCD files through the stand-in reader of oracle/ref_shim/pcl/io/pcd_io.h)
    on the directory oracle/dataset_writer.py lays out — the layout
    tests/test_dataset_loader.py holds the product's loader (global-lvba_b200/host/lvba_dataset.hpp) against.  Pins: frame timestamps come from the
    file NAMES (:228-233), TUM lines with a comment, an empty and an unparsable line and un-normalised quaternions (:137-180), images = every
    image_sample_step-th file by timestamp and the same stride over the VALID pose lines (:118-121, :159), intrinsics scaled by cam_model/scale (:59-62),
    colmap_db_path appended to the data path (:65)."""
    from oracle import dataset_writer as dw
    scans, poses, ts, image_ts, image_poses = loader_dataset(Path(tempfile.mkdtemp()))
    d = recorded("dataset_loader")
    d["scans"] = split(d["scans_xyz"], d["scan_ptr"])
    assert str(d["data_path"]) == "/" and str(d["db_path"]) == "/Colmap/colmap.db"
    assert d["cam"][:6].tolist() == [80.0, 64.0, 48.0, 48.15, 39.85, 32.1] and d["cam"][10:].tolist() == [0.5, 2.0]
    assert np.array_equal(d["frame_ts"], np.array(ts))                   # from the names: the TUM file's own timestamps (0, 1, 2 ...) are ignored
    assert [len(s) for s in d["scans"]] == [len(s) for s in scans] and all(np.array_equal(a, b) for a, b in zip(d["scans"], scans))
    assert np.array_equal(d["intensity"], np.concatenate([np.arange(len(s)) % 7 for s in scans]).astype(np.float32))
    rt = lambda P: np.array([np.r_[dw.quat_to_R(dw.R_to_quat(p[:9].reshape(3, 3))).ravel(), p[9:]] for p in P])  # noqa: E731
    assert np.abs(d["frame_poses"] - rt(poses)).max() <= 1e-11            # 15-digit text, quaternion normalised on reading (:165-166)
    assert np.abs(d["image_ts"] - np.array(image_ts)).max() <= 1e-9 and len(d["image_ts"]) == 7      # 14 files, every second one
    assert np.abs(d["image_poses"] - rt(image_poses)).max() <= 1e-11      # the skipped lines carry poses 100 m away: none of them was taken


# ------------------------------------------------------------------------------------------------ B5: the per-track helpers on their own
def ref_track_helpers():
    import test_track_emu as tt
    p, cams, op, oc, uv, intr = tt._problem()
    Xr, mr, cr, okr = sr.track_helpers(op, oc, uv, cams, intr)
    _, m2, c2, ok2 = sr.track_helpers(op, oc, uv, cams, intr, Xw=np.ascontiguousarray(p["X_gt"] + 0.01), min_count=5)
    return dict(X=Xr, mean=mr, count=cr, ok=okr, mean_at_X=m2, count_at_X=c2, ok_at_X=ok2)


def test_dlt_and_mean_reprojection_equal_reference_source_live():
    """TriangulateTrackDLT (src/lvba_system.cpp:52-111) and ComputeMeanReproj (:8-50), called directly (they are file-scope functions of the
    included source), vs oracle/track_oracle.py and the device functors through the host policy (tests/emu/track_emu.cpp) on 400 tracks.
    The reference sums in its container's order and solves the 4x4 eigen-problem with the library's solver (here: the stand-in's Jacobi):
    agreement to 1e-9, not to the bit."""
    import ctypes
    import subprocess
    import test_track_emu as tt
    from oracle import track_oracle as tro
    p, cams, op, oc, uv, intr = tt._problem()
    T = len(op) - 1
    R = recorded("track_helpers")
    Xr, mr, cr, okr = R["X"], R["mean"], R["count"], R["ok"]
    so = Path(tempfile.mkdtemp()) / "libtrack_emu.so"
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", str(ROOT / "tests" / "emu" / "track_emu.cpp"), "-o", str(so)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    emu = ctypes.CDLL(str(so))
    Xe = np.zeros((T, 3)); me = np.zeros(T); ce = np.zeros(T, np.int32); oke = np.zeros(T, np.uint8)
    emu.emu_tracks_triangulate(ctypes.c_int64(T), tt._ptr(op, ctypes.c_int64), tt._ptr(oc, ctypes.c_int32), tt._ptr(uv, ctypes.c_float), ctypes.c_int32(40),
                               tt._ptr(cams, ctypes.c_double), tt._ptr(intr, ctypes.c_double), tt._ptr(Xe, ctypes.c_double), tt._ptr(me, ctypes.c_double),
                               tt._ptr(ce, ctypes.c_int32), oke.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)))
    assert np.array_equal(okr, oke.astype(bool)) and okr.sum() > 100 and not okr.all()
    assert np.array_equal(cr[okr], ce[okr])
    assert np.abs(Xr[okr] - Xe[okr]).max() <= 1e-9 * max(1.0, np.abs(Xr[okr]).max()) and np.abs(mr[okr] - me[okr]).max() <= 1e-9
    for t in np.nonzero(okr)[0][::9]:
        sel = list(range(op[t], op[t + 1]))
        o_ok, X, m, c = tro.triangulate_dlt(cams[oc[sel]], uv[sel], intr)
        assert o_ok and c == cr[t] and np.abs(X - Xr[t]).max() <= 1e-7 * max(1.0, np.abs(X).max()) and abs(m - mr[t]) <= 1e-7   # LAPACK eigh vs Jacobi on short baselines: the smallest eigenvector of A^T A is conditioned like 1e7
    X = np.ascontiguousarray(p["X_gt"] + 0.01)
    m2, c2, ok2 = R["mean_at_X"], R["count_at_X"], R["ok_at_X"]
    assert ok2.any() and not ok2.all()
    for t in range(0, T, 5):
        sel = list(range(op[t], op[t + 1]))
        o_ok, m, c = tro.mean_reproj(X[t], cams[oc[sel]], uv[sel], intr, 5)
        assert o_ok == bool(ok2[t]) and c == c2[t] and (not o_ok or abs(m - m2[t]) <= 1e-9)


# ------------------------------------------------------------------------------------------------ F, differential: many scenes, live
def _depth_images_for(s, width=640, height=512):
    """Depth images that hand every keypoint with a depth candidate (roughly) the camera-frame depth of that candidate: its four bilinear
    neighbours are set to z_c.  Overlapping neighbourhoods overwrite each other — both sides read the images, so that only varies the scene."""
    M = len(s["kp_ptr"]) - 1
    img = np.zeros((M, height, width), np.float32)
    for i in range(M):
        R = s["cams"][i, :9].reshape(3, 3); t = s["cams"][i, 9:]
        for g in range(int(s["kp_ptr"][i]), int(s["kp_ptr"][i + 1])):
            if not s["kp_valid"][g]:
                continue
            z = float((R @ s["kp_Xw"][g] + t)[2])
            u, v = float(s["kp_uv"][g, 0]), float(s["kp_uv"][g, 1])
            if z <= 0.1 or not (0 <= u < width - 1 and 0 <= v < height - 1):
                continue
            x, y = int(np.floor(u)), int(np.floor(v))
            img[i, y:y + 2, x:x + 2] = np.float32(z)
    return img


FUSION_CASES = [(0, {}), (1, dict(wrong=0.15)), (2, dict(no_depth=0.6)), (3, dict(bad_depth=0.3, px_noise=1.2)),
                (4, dict(n_images=30, n_points=300)), (7, dict(n_images=45, n_points=200, wrong=0.1)), (8, dict(n_images=20, n_points=150, wrong=0.3))]


def ref_build_tracks(seed, kw):
    import fuse_scene
    s = fuse_scene.make(seed=seed, **kw)
    S = sr.System()
    S.set_fusion_inputs(s["cams"], _depth_images_for(s), s["intr"], s["kp_ptr"], s["kp_uv"], s["matches"])
    T = S.build_tracks()
    S.close()
    return T


@pytest.mark.parametrize("seed,kw", FUSION_CASES)
def test_track_fusion_differential_reference_source_vs_oracle_and_device_pass(seed, kw, tmp_path_factory):
    """BuildTracksAndFuse3D from the reference's own source on the scenes of tests/test_fuse_emu.py (wrong matches that merge components, missing and
    wrong depth, up to 45 images: more keys than buckets in the reference's maps, failed components retried from other seeds) against
    oracle/fuse_oracle.py under the container order and against csrc/fuse_pipeline.h through the host policy with LVBA_FUSE_ORDER_LIBSTDCXX."""
    import ctypes
    import subprocess
    import fuse_scene
    import test_fuse_emu
    s = fuse_scene.make(seed=seed, **kw)
    depth = _depth_images_for(s)
    Xw, valid = dep.backproject(list(depth), s["cams"], s["intr"], s["kp_ptr"], s["kp_uv"])
    T = recorded(f"build_tracks_{seed}")
    tr = fo.fuse(s["kp_ptr"], s["kp_uv"], s["matches"], s["cams"], s["intr"], Xw, valid, map_order=fo.libstdcxx_order)
    assert len(tr) == len(T["Xw"]) > 0
    for k, t in enumerate(tr):
        assert np.array_equal(t["obs"], T["obs"][T["obs_ptr"][k]:T["obs_ptr"][k + 1]]), k
        assert list(t["kept"]) == T["inl"][T["inl_ptr"][k]:T["inl_ptr"][k + 1]].tolist(), k
        assert np.abs(t["Xw"] - T["Xw"][k]).max() <= 1e-7 * max(1.0, np.abs(T["Xw"][k]).max()), k      # DLT on short baselines: LAPACK eigh vs Jacobi
    so = tmp_path_factory.mktemp("emu_ref_fuse_diff") / "libfuse_emu.so"
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", str(ROOT / "tests" / "emu" / "fuse_emu.cpp"), "-o", str(so)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = ctypes.CDLL(str(so)); lib.fuse_emu_run.restype = ctypes.c_longlong
    got = test_fuse_emu.run_emu(lib, dict(s, kp_Xw=Xw, kp_valid=valid), map_order=1)
    assert len(got["seed"]) == len(T["Xw"])
    for k in range(len(T["Xw"])):
        a, b = got["obs_ptr"][k], got["obs_ptr"][k + 1]
        assert np.array_equal(np.column_stack([got["img"][a:b], got["kp"][a:b]]), T["obs"][T["obs_ptr"][k]:T["obs_ptr"][k + 1]]), k
        inl = np.zeros(b - a, bool); inl[T["inl"][T["inl_ptr"][k]:T["inl_ptr"][k + 1]]] = True
        assert np.array_equal(got["inlier"][a:b].astype(bool), inl), k
        assert np.abs(got["Xw"][k] - T["Xw"][k]).max() <= 1e-9 * max(1.0, np.abs(T["Xw"][k]).max()), k


# ------------------------------------------------------------------------------------------------ D, differential: more scenes, live
DEPTH_CASES = [(11, 5, 3, (64, 48)), (12, 9, 6, (120, 90)), (13, 4, 5, (200, 160))]


def depth_scene_for(seed, F, M, size):
    sc = synth.make_depth_scene(seed, F=F, n_per_scan=1800, M=M, width=size[0], height=size[1])
    img_ts = np.round(sc["image_ts"], 6)
    img_ts[0] = sc["frame_ts"][0] - 3.0                                   # nothing within +-0.5 s: an empty image
    return sc, img_ts


def ref_depth(seed, F, M, size):
    sc, img_ts = depth_scene_for(seed, F, M, size)
    body = np.zeros((M, 12))
    for k in range(M):                                                    # body poses whose cameras are sc["cams"]: Rcw = Rci Rwi^T with Rci = I, tci = 0
        Rcw = sc["cams"][k, :9].reshape(3, 3); tcw = sc["cams"][k, 9:]
        body[k, :9] = Rcw.T.ravel(); body[k, 9:] = -Rcw.T @ tcw
    S = sr.System()
    S.set_lidar(sc["scans"], sc["poses"], sc["frame_ts"])
    S.set_stages(False)
    S.set_camera(size[0], size[1], sc["intr"], np.eye(3).ravel(), np.zeros(3), np.eye(3).ravel(), np.zeros(3), img_ts, body)
    S.build_grid(); S.update_camera_poses()
    d, _, c1 = S.generate_depth()
    S.close()
    return dict(depth=d, cams=c1)


@pytest.mark.parametrize("seed,F,M,size", DEPTH_CASES)
def test_depth_rendering_differential_reference_source_vs_oracle(seed, F, M, size):
    """buildGridMapFromOptimized + generateDepthWithVoxel from the reference's own source on further scenes (image timestamps outside the scan range
    included: some images see no frame) — images equal to the oracle's bit for bit."""
    sc, img_ts = depth_scene_for(seed, F, M, size)
    R = recorded(f"depth_{seed}")
    d, c1 = R["depth"], R["cams"]
    assert np.abs(c1 - sc["cams"]).max() <= 1e-12
    img = dep.render(sc["scans"], sc["poses"], sc["frame_ts"], c1, img_ts, sc["intr"], size[0], size[1])
    assert np.array_equal(img, d) and not d[0].any() and (d[1:] > 0).sum() > 500


# ------------------------------------------------------------------------------------------------ N4: the COLMAP text model
def colmap_export_dataset(data):
    import visual_scene as vs
    from oracle import dataset_writer as dw
    g = vs.make(data, seed=4, W=6, n_per_scan=6000, n_landmarks=60)
    # one more image 5 s after the last scan: no LiDAR within +-0.5 s -> the reference lists it neither in images.txt nor in the points (:1994-1997)
    image_ts = list(g["image_ts"]) + [g["image_ts"][-1] + 5.0]
    image_poses = np.vstack([g["image_poses"], g["image_poses"][-1:]])
    dw.write_image_set(data, image_ts, image_poses, extra_between=1)
    dw.write_colmap_db(data / "Colmap" / "colmap.db", image_ts, g["keypoints"] + [np.zeros((0, 2), np.float32)], {k: np.array(v) for k, v in g["pair"].items() if k != (0, 1)})


def points3d_rows(text):
    return sorted(" ".join(ln.split()[1:]) for ln in text.splitlines())


def ref_colmap_export():
    """The reference's images.txt and the rows of its points3D.txt (point ids dropped, sorted) on colmap_export_dataset."""
    import visual_scene as vs
    data = Path(tempfile.mkdtemp()) / "data"
    colmap_export_dataset(data)
    F = vs.INTR_FULL
    S = sr.System({"data_config/data_path": str(data) + "/", "data_config/colmap_db_path": "Colmap/colmap.db", "data_config/image_sample_step": 2,
                   "cam_model/cam_width": vs.WIDTH_FULL, "cam_model/cam_height": vs.HEIGHT_FULL, "cam_model/scale": vs.SCALE, "cam_model/cam_fx": F[0],
                   "cam_model/cam_fy": F[1], "cam_model/cam_cx": F[2], "cam_model/cam_cy": F[3], "cam_model/cam_d0": F[4], "cam_model/cam_d1": F[5],
                   "cam_model/cam_d2": F[6], "cam_model/cam_d3": F[7], "extrin_calib/Rcl": vs.RCL.ravel(), "extrin_calib/Pcl": vs.PCL,
                   "extrin_calib/extrinsic_R": np.eye(3).ravel(), "extrin_calib/extrinsic_T": np.zeros(3)})
    d = S.init_from_dataset()
    S.build_grid(); S.update_camera_poses(); S.generate_depth()
    S.colmap_export(str(data) + "/")
    S.close()
    ref_dir = data / "Colmap" / "sparse"
    return dict(n_frames=len(d["frame_ts"]), n_images=len(d["image_ts"]), images_txt=(ref_dir / "images.txt").read_text(),
                points3d_rows="\n".join(points3d_rows((ref_dir / "points3D.txt").read_text())))


def test_colmap_export_equals_the_reference_writer(pkg, tmp_path):
    """VisualizeOptComparison (src/lvba_system.cpp:1932-2143), run from its own source on a dataset its own loader read (every image file = one grey value:
    there is no decoder on either side), against `lvba_offline --check --visual --points3d lidar` (host code of global-lvba_b200/host/lvba_visual_offline.hpp,
    no GPU): images.txt line for line, points3D.txt row for row as a set (the reference lists the thinned points in unordered_map order)."""
    import subprocess
    data = tmp_path / "data"
    colmap_export_dataset(data)
    exe = tmp_path / "lvba_offline"
    cmd = ["g++", "-std=c++17", "-O2", "-I", str(ROOT / "include"), str(ROOT / "tools" / "lvba_offline.cpp"), "-o", str(exe),
           str(pkg.LIB_PATH), f"-Wl,-rpath,{pkg.LIB_PATH.parent}", "-L/usr/local/cuda/lib64", "-lcudart", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    mine = tmp_path / "mine"
    r = subprocess.run([str(exe), "--data", str(data), "--config", str(data / "config.yaml"), "--check", "--visual", "--points3d", "lidar", "--sparse-dir", str(mine)],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    R = recorded("colmap_export")
    assert int(R["n_frames"]) == 6 and int(R["n_images"]) == 7
    ref_images = str(R["images_txt"])
    assert (mine / "images.txt").read_text() == ref_images
    assert len(ref_images.splitlines()) == 12                                     # six of the seven images: the late one is left out on both sides
    a, b = points3d_rows((mine / "points3D.txt").read_text()), str(R["points3d_rows"]).split("\n")
    assert len(a) == len(b) > 2000 and a == b
    assert all(ln.endswith("128 128 128 0") for ln in a[:50])


def test_lidar_half_live_without_the_window_stage():
    """window_ba/enable = false (:217-225): the global stages run on the frames themselves — the path `lvba_offline` takes without --window."""
    scans, noisy = noisy_scan_scene(41, 6)
    out = recorded("lidar_ba_41")["poses"]
    x = noisy
    for vs_, er in ((1.0, S1R), (0.5, S2R)):
        vp, pi, cl, _ = vox.voxelize(scans, x, vs_, er)
        x, _ = lo.damping_iter(vp, pi, cl, x)
    assert np.abs(out - x).max() <= 1e-9 and np.abs(out - noisy).max() > 1e-3


def bucket_count_ns():
    return list(range(0, 300)) + [p + d for p in fo._PRIMES if p < 3_000_000 for d in (-1, 0, 1)]


def ref_bucket_counts():
    return dict(n=np.array(bucket_count_ns(), np.int64), bucket_count=np.array([sr.bucket_count_after_reserve(n) for n in bucket_count_ns()], np.int64))


def test_bucket_count_table_equals_the_real_container(tmp_path_factory):
    """stl_bucket_count (csrc/fuse_pipeline.h) and the table of oracle/fuse_oracle.py against std::unordered_map::reserve(n) / bucket_count() of the
    library the reference is compiled with: every n up to 300, then every table entry below 3e6 and its two neighbours."""
    import ctypes
    import subprocess
    so = tmp_path_factory.mktemp("emu_bkt") / "libfuse_emu.so"
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", str(ROOT / "tests" / "emu" / "fuse_emu.cpp"), "-o", str(so)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    lib = ctypes.CDLL(str(so)); lib.emu_stl_bucket_count.restype = ctypes.c_uint
    R = recorded("bucket_counts")
    ns = bucket_count_ns()
    assert R["n"].tolist() == ns
    for n, real in zip(ns, R["bucket_count"].tolist()):
        assert lib.emu_stl_bucket_count(ctypes.c_uint(n)) == real, n
        if n >= 14:
            assert next(p for p in fo._PRIMES if p >= n) == real, n
