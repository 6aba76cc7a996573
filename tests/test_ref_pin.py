"""The oracles, pinned against the REFERENCE'S OWN SOURCE (SURVEY.md §8c).

tests/golden/ref_balm.npz holds seeded inputs and what /root/reference/include/BALM/{tools,bavoxel}.hpp and
/root/reference/include/utils.hpp computed from them, compiled where they lie (oracle/ref_driver.cpp, `make -C oracle ref`)
on top of stand-ins for Eigen / PCL / OpenCV / Ceres / Sophus (oracle/ref_shim/, own code: the 3x3 eigen-solver, the sparse
LDL^T and the dual numbers under the reference's lines are ours, every line of the reference's arithmetic and control flow
is the reference's).  Here, without a GPU:

  1. the numpy oracles (oracle/*.py) reproduce the file            -> the restatements equal the source they restate
  2. the C++ port oracle/cpu_ref.cpp (the bench's CPU arm) does too  -> the timed CPU arm computes what the reference does
  3. the device passes, run through the host policy (tests/emu/), do too (voxel map, anchor clouds, >128-pose voxel pass)
  4. further seeded problems, at sizes the fixture does not hold, against what the reference source computed from them
     (tests/golden/ref_live_balm.npz, written by tests/golden/make_golden_ref_live.py); where oracle/_ref/libbalm_ref.so is
     built, the fixture is also regenerated and must come out bit for bit.

The CUDA path is held against the same file in tests/test_zzz_ref_gpu.py.  Tolerances: integer / key / count data exact;
float64 sums whose order differs 1e-12 relative; quantities behind the eigen-decomposition of P/N - v v^T (lambda_0, g, H:
a difference of O(1e2..1e4) terms, SURVEY.md Q7) 1e-9 relative — observed 1e-11; LM end poses 1e-9 (observed 2e-11).
"""
import os
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT / "tests"))

from oracle import anchor_oracle as ao, balm_ref, depth_oracle as dep, lidar_oracle as lo, synth, visual_oracle as vis, voxel_oracle as vox  # noqa: E402
import test_anchor_emu, test_big_voxel_emu, test_voxel_emu  # noqa: E402,E401

G = np.load(ROOT / "tests" / "golden" / "ref_balm.npz")
LIVE = ROOT / "tests" / "golden" / "ref_live_balm.npz"

needs_ref = pytest.mark.skipif(not balm_ref.available(), reason="oracle/_ref/libbalm_ref.so is built only where the original sources are readable")


def recorded(tag):
    """What the ref_* function below returned for case `tag` when the fixture was written."""
    with np.load(LIVE) as f:
        return {k[len(tag) + 2:]: f[k] for k in f.files if k.startswith(tag + "__")}


def csr(tag):
    return G[f"{tag}_vox_ptr"], G[f"{tag}_pose_idx"], G[f"{tag}_clusters"], G[f"{tag}_poses"]


def split(flat, ptr):
    return [flat[ptr[i]:ptr[i + 1]] for i in range(len(ptr) - 1)]


def lex(a):
    return a[np.lexsort(a.T[::-1])]


# ------------------------------------------------------------------------------------------------ 1. numpy oracles
@pytest.mark.parametrize("tag", ["L1", "L2", "L3"])
def test_numpy_hessian_equals_reference_source(tag):
    vp, pi, cl, ps = csr(tag)
    W = len(ps)
    keep = np.diff(vp) >= 2                                       # push_voxel (bavoxel.hpp:45-54): the oracle takes kept voxels
    assert int(keep.sum()) == int(G[f"{tag}_kept"])
    if not keep.all():
        sel = np.concatenate([np.arange(vp[a], vp[a + 1]) for a in np.nonzero(keep)[0]])
        vp = np.concatenate([[0], np.cumsum(np.diff(vp)[keep])]); pi = pi[sel]; cl = cl[sel]
    r, g, blocks = lo.acc_evaluate2(vp, pi, cl, ps, W)
    H = lo.assemble_dense(blocks, W)
    assert abs(r - G[f"{tag}_residual_sum"]) <= 1e-9 * abs(G[f"{tag}_residual_sum"])
    assert np.abs(g - G[f"{tag}_g"]).max() <= 1e-9 * np.abs(G[f"{tag}_g"]).max()
    assert np.abs(H - G[f"{tag}_H"]).max() <= 1e-9 * np.abs(G[f"{tag}_H"]).max()
    Hr = G[f"{tag}_H"]
    off = np.kron(1 - np.eye(W), np.ones((6, 6))) > 0              # bavoxel.hpp:171-173 mirrors the off-diagonal BLOCKS (exactly);
    assert np.array_equal(Hr[off], Hr.T[off])                      # a diagonal block is symmetric up to rounding only
    assert np.abs(Hr - Hr.T).max() <= 1e-12 * np.abs(Hr).max()


@pytest.mark.parametrize("tag", ["L1", "L2"])
def test_divide_thread_is_the_same_sum_averaged(tag):
    """BALM2::divide_thread (16 private Hessians, bavoxel.hpp:597-639): sum / kept (AVG_THR) of what one call accumulates."""
    kept = int(G[f"{tag}_kept"])
    assert abs(G[f"{tag}_residual_avg_threads"] * kept - G[f"{tag}_residual_sum"]) <= 1e-12 * abs(G[f"{tag}_residual_sum"])
    assert np.abs(G[f"{tag}_g_threads"] - G[f"{tag}_g"]).max() <= 1e-12 * np.abs(G[f"{tag}_g"]).max()


@pytest.mark.parametrize("tag", ["L1", "L2"])
def test_numpy_residual_and_damping_iter_equal_reference_source(tag):
    vp, pi, cl, ps = csr(tag)
    r_gt = lo.only_residual(vp, pi, cl, G[f"{tag}_poses_gt"])
    assert abs(r_gt - G[f"{tag}_residual_gt"]) <= 1e-9 * abs(G[f"{tag}_residual_gt"])
    poses, info = lo.damping_iter(vp, pi, cl, ps)
    assert np.abs(poses - G[f"{tag}_lm_poses"]).max() <= 1e-9
    assert np.abs(G[f"{tag}_lm_poses"] - ps).max() > 1e-3          # the solve moved the poses: the comparison is not vacuous
    assert abs(info["r_last"] * (len(vp) - 1) - G[f"{tag}_lm_residual_sum"]) <= 1e-8 * abs(G[f"{tag}_lm_residual_sum"])


def test_numpy_exp_equals_reference_source():
    assert np.abs(lo.so3_exp(G["E_w"]) - G["E_R"]).max() <= 1e-15
    assert np.array_equal(G["E_R"][0], np.eye(3)) and np.array_equal(G["E_R"][1], np.eye(3))     # below the 1e-11 switch (tools.hpp:66)


def map_scene():
    return split(G["M_xyz"], G["M_scan_ptr"]), G["M_poses"]


def ref_map():
    meta = dict(key=G["M_key"], layer=G["M_layer"], path=[tuple(int(x) for x in p if x >= 0) for p in G["M_path"]],
                centre=G["M_centre"], direct=G["M_direct"], eigenvalues=G["M_eigenvalues"])
    return G["M_vox_ptr"], G["M_pose_idx"], G["M_clusters"], meta


@pytest.mark.parametrize("literal", [True, False])
def test_numpy_voxel_map_equals_reference_source(literal):
    scans, poses = map_scene()
    fn = vox.voxelize_literal if literal else vox.voxelize
    vp, pi, cl, meta = fn(scans, poses, float(G["M_voxel_size"]), G["M_eigen_ratio"])
    rvp, rpi, rcl, rmeta = ref_map()
    assert np.array_equal(vp, rvp) and np.array_equal(pi, rpi)
    assert np.array_equal(meta["key"], rmeta["key"]) and np.array_equal(meta["layer"], rmeta["layer"]) and list(meta["path"]) == rmeta["path"]
    assert np.abs(cl - rcl).max() <= 1e-12 * np.abs(rcl).max()     # (equal to the bit on the machine that wrote the file: numpy's small matmul adds in the same order)
    assert np.abs(meta["centre"] - rmeta["centre"]).max() <= 1e-12
    assert np.abs(meta["eigenvalues"] - rmeta["eigenvalues"]).max() <= 1e-12
    assert np.all(np.abs(np.einsum("ij,ij->i", meta["direct"], rmeta["direct"])) >= 1 - 1e-9)   # eigenvector sign is the library's


def ref_lookup_nd():
    """The (n, d) step of recompute_local_planes (src/lvba_system.cpp:1552-1563) on the node the reference's findCorrespondPoint found."""
    st, d, c = G["M_lookup_state"], G["M_lookup_direct"], G["M_lookup_centre"]
    nd = np.zeros((len(st), 4))
    for i in np.nonzero(st == 2)[0]:
        if np.all(np.isfinite(d[i])) and np.linalg.norm(d[i]) >= 1e-6 and np.all(np.isfinite(c[i])):
            n = d[i] / np.linalg.norm(d[i]); nd[i, :3] = n; nd[i, 3] = -n @ c[i]
    return nd


def test_numpy_plane_lookup_equals_reference_source():
    scans, poses = map_scene()
    roots = vox.build_tree_literal(scans, poses, float(G["M_voxel_size"]), G["M_eigen_ratio"])
    nd = vox.plane_lookup_literal(roots, G["M_lookup_X"], float(G["M_voxel_size"]))
    ref = ref_lookup_nd()
    assert 50 < int((ref != 0).any(1).sum()) < len(ref)           # hits and misses both present
    assert np.all(G["M_lookup_state"][[7, 8, 9]] == -1)            # NaN / inf / far away: no root voxel
    test_voxel_emu.compare_lookup(nd, ref)
    sgn = np.sign(np.einsum("ij,ij->i", nd[:, :3], ref[:, :3])); sgn[sgn == 0] = 1
    assert np.abs(nd * sgn[:, None] - ref).max() <= 1e-11


def test_numpy_window_lm_on_the_map_equals_reference_source():
    vp, pi, cl, _ = ref_map()
    poses, _ = lo.damping_iter(vp, pi, cl, G["M_poses"])
    assert np.abs(poses - G["M_lm_poses"]).max() <= 1e-9
    assert np.abs(G["M_lm_poses"] - G["M_poses"]).max() > 1e-4


def test_numpy_anchor_cloud_equals_reference_source():
    scans, _ = map_scene()
    win_ptr = np.array([0, len(scans)])
    for fn in (ao.anchor_clouds_literal, ao.anchor_clouds):
        got = fn(scans, G["A_rel"], win_ptr, float(G["A_leaf"]))[0]
        assert np.array_equal(lex(got), G["A_cloud_sorted"])       # the reference's order is its unordered_map's: compared as sets


def visual_rows():
    trk = np.repeat(np.arange(len(G["V_obs_ptr"]) - 1), np.diff(G["V_obs_ptr"]))
    return G["V_q"][G["V_obs_cam"]], G["V_t"][G["V_obs_cam"]], G["V_X"][trk]


def test_numpy_cost_functors_equal_reference_source():
    """Residuals with T = double, Jacobians with T = Jet (what AutoDiffCostFunction hands the solver) vs the oracle's analytic ones."""
    q, t, X = visual_rows()
    r, Jq, Jt, JX = vis.reproj_eval(q, t, X, G["V_obs_uv"], G["V_intr"], float(G["V_sigma_px"]))
    assert np.abs(r - G["V_reproj_r"]).max() <= 1e-10 * np.abs(G["V_reproj_r"]).max()
    J = G["V_reproj_J"]
    Jq_ref = J[:, :, :4] @ vis.plus_jacobian(q / np.linalg.norm(q, axis=1, keepdims=True))      # ambient (w,x,y,z) -> the manifold's tangent
    for mine, ref in ((Jq, Jq_ref), (Jt, J[:, :, 4:7]), (JX, J[:, :, 7:])):
        assert np.abs(mine - ref).max() <= 1e-12 * np.abs(ref).max()
    r, Jp = vis.plane_eval(G["V_X"], G["V_plane_nd"], float(G["V_sigma_plane"]))
    assert np.abs(r - G["V_plane_r"]).max() <= 1e-10 * np.abs(G["V_plane_r"]).max()
    assert np.abs(Jp - G["V_plane_J"]).max() <= 1e-12 * np.abs(G["V_plane_J"]).max()


def test_numpy_cost_functor_edge_cases_equal_reference_source():
    """Points behind the camera and z_c <= 1e-8 give zero residual AND zero Jacobian (utils.hpp:78); a scaled quaternion is
    normalised by QuaternionRotatePoint (the residual does not change, the ambient Jacobian loses its radial part)."""
    q, t, X, uv = G["V_edge_q"], G["V_edge_t"], G["V_edge_X"], G["V_edge_uv"]
    r_ref, J_ref = G["V_edge_r"], G["V_edge_J"]
    dead = [0, 1, 2, 3, 8, 9]
    assert np.all(r_ref[dead] == 0) and np.all(J_ref[dead] == 0) and np.all(np.abs(r_ref[10]) > 0)
    r, Jq, Jt, JX = vis.reproj_eval(q, t, X, uv, G["V_intr"], float(G["V_sigma_px"]))
    assert np.all(r[dead] == 0) and np.all(Jt[dead] == 0) and np.all(JX[dead] == 0) and np.all(Jq[dead] == 0)
    live = [i for i in range(12) if i not in dead and i != 10]      # row 10 sits at z_c = 2e-8: |r| ~ 1e3 px, conditioning 1e8
    assert np.abs(r[live] - r_ref[live]).max() <= 1e-10 * np.abs(r_ref[live]).max()
    assert np.abs(r[10] - r_ref[10]).max() <= 1e-6 * np.abs(r_ref[10]).max()
    assert np.abs(Jt[live] - J_ref[live][:, :, 4:7]).max() <= 1e-12 * np.abs(J_ref[live]).max()
    qs = q[4:8]                                                     # scaled by 1.7: J_ambient . q = 0 (no radial sensitivity)
    assert np.abs(np.einsum("nak,nk->na", J_ref[4:8, :, :4], qs)).max() <= 1e-9 * np.abs(J_ref[4:8, :, :4]).max()


def test_numpy_camera_helpers_equal_reference_source():
    ok, uu, vv = dep.project(G["C_Xc"], G["C_intr"])
    assert np.array_equal(ok, G["C_proj_ok"]) and not ok[:13].any() and ok[13:].all()
    assert np.array_equal(uu[ok], G["C_proj_uv"][ok, 0]) and np.array_equal(vv[ok], G["C_proj_uv"][ok, 1])     # bit for bit
    assert np.array_equal(G["C_Xc"][ok, 2], G["C_proj_z"][ok])
    res = [dep.undistort_pixel(G["C_intr"], float(a), float(b)) for a, b in G["C_und_uv"]]
    ok = np.array([r[0] for r in res]); xy = np.array([[r[1], r[2]] for r in res])
    assert np.array_equal(ok, G["C_und_ok"]) and not ok[3] and np.array_equal(xy[ok], G["C_und_xy"][ok])
    kp = G["C_kp"]
    Xw, valid = dep.backproject([G["C_depth"]], G["C_cam"][None], G["C_intr"], np.array([0, len(kp)]), kp)
    assert np.array_equal(valid.astype(bool), G["C_cand_ok"] == 3) and 100 < int(valid.sum()) < len(kp)
    assert np.array_equal(Xw, G["C_cand_Xw"])                      # fetchDepthBilinear (float32) -> back-projection -> camToWorld: bit for bit
    for i in np.nonzero(G["C_cand_ok"] & 1)[0][:50]:
        ok1, d = dep.fetch_depth_bilinear(G["C_depth"], kp[i, 0], kp[i, 1])
        assert ok1 and d == G["C_cand_d"][i]


# ------------------------------------------------------------------------------------------------ 2. the C++ port (CPU arm of bench.py)
@pytest.mark.parametrize("tag", ["L1", "L2"])
def test_cpp_port_equals_reference_source(tag):
    from oracle import cpu_ref
    vp, pi, cl, ps = csr(tag)
    W = len(ps)
    for threads in (1, 4):
        r, g, br_, bc, bl = cpu_ref.lidar_build(vp, pi, cl, ps, threads=threads)
        H = np.zeros((6 * W, 6 * W))
        for k in range(len(br_)):
            i, j = int(br_[k]), int(bc[k])
            H[6 * i:6 * i + 6, 6 * j:6 * j + 6] = bl[k]
            H[6 * j:6 * j + 6, 6 * i:6 * i + 6] = bl[k].T
        # the port returns the same quantity divide_thread returns or its sum: accept either convention, pin the value
        ref_sum = float(G[f"{tag}_residual_sum"])
        assert min(abs(r - ref_sum), abs(r * int(G[f"{tag}_kept"]) - ref_sum)) <= 1e-9 * abs(ref_sum)
        assert np.abs(g - G[f"{tag}_g"]).max() <= 1e-9 * np.abs(G[f"{tag}_g"]).max()
        assert np.abs(H - G[f"{tag}_H"]).max() <= 1e-9 * np.abs(G[f"{tag}_H"]).max()
    assert abs(cpu_ref.lidar_residual(vp, pi, cl, G[f"{tag}_poses_gt"]) - G[f"{tag}_residual_gt"]) <= 1e-9 * abs(G[f"{tag}_residual_gt"])
    poses, info = cpu_ref.lidar_lm(vp, pi, cl, ps, threads=4)
    assert np.abs(poses - G[f"{tag}_lm_poses"]).max() <= 1e-9


# ------------------------------------------------------------------------------------------------ 3. the device passes through the host policy
def test_device_voxel_passes_equal_reference_source(request):
    emu = request.getfixturevalue("voxel_emu_lib")
    scans, poses = map_scene()
    m = test_voxel_emu.EmuMap(emu, scans, poses, float(G["M_voxel_size"]), G["M_eigen_ratio"])
    assert m.rc == 0
    test_voxel_emu.compare_with_oracle(m.export(), ref_map())
    test_voxel_emu.compare_lookup(m.lookup(G["M_lookup_X"]), ref_lookup_nd())
    m.close()


def test_device_anchor_pass_equals_reference_source(request):
    emu = request.getfixturevalue("anchor_emu_lib")
    scans, _ = map_scene()
    rc, got = test_anchor_emu.run(emu, scans, G["A_rel"], np.array([0, len(scans)]), float(G["A_leaf"]))
    assert rc == 0 and np.array_equal(lex(got[0]), G["A_cloud_sorted"])


@pytest.mark.parametrize("tag", ["L1", "L2"])
def test_device_wide_voxel_pass_equals_reference_source(request, tag):
    """csrc/lidar_big.h (the accumulation pass for voxels seen from more than 128 poses) run on ordinary voxels."""
    emu = request.getfixturevalue("big_emu_lib")
    vp, pi, cl, ps = csr(tag)
    W = len(ps)
    r, g, lower = test_big_voxel_emu.run(emu, dict(vox_ptr=vp, pose_idx=pi, clusters=cl, poses=ps), W)
    mask = np.kron(np.tril(np.ones((W, W))), np.ones((6, 6))) > 0
    assert abs(r - G[f"{tag}_residual_sum"]) <= 1e-8 * abs(G[f"{tag}_residual_sum"])
    assert np.abs(g - G[f"{tag}_g"]).max() <= 1e-7 * np.abs(G[f"{tag}_g"]).max()
    assert np.abs(lower - G[f"{tag}_H"] * mask).max() <= 1e-7 * np.abs(G[f"{tag}_H"]).max()


@pytest.fixture(scope="module")
def voxel_emu_lib(tmp_path_factory):
    return _compile("voxel_emu.cpp", tmp_path_factory)


@pytest.fixture(scope="module")
def anchor_emu_lib(tmp_path_factory):
    return _compile("anchor_emu.cpp", tmp_path_factory)


@pytest.fixture(scope="module")
def big_emu_lib(tmp_path_factory):
    lib = _compile("big_emu.cpp", tmp_path_factory)
    import ctypes
    lib.emu_big_accumulate.restype = ctypes.c_double
    return lib


def _compile(src, tmp_path_factory):
    import ctypes
    import subprocess
    so = tmp_path_factory.mktemp("emu_ref") / ("lib" + src.replace(".cpp", ".so"))
    r = subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared", str(ROOT / "tests" / "emu" / src), "-o", str(so)],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return ctypes.CDLL(str(so))


# ------------------------------------------------------------------------------------------------ 4. live, where the reference can be compiled
@needs_ref
def test_fixture_is_what_the_reference_source_computes_bit_for_bit():
    sys.path.insert(0, str(ROOT / "tests" / "golden"))
    import make_golden_ref
    fresh = make_golden_ref.generate()
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


# The ref_* functions run the reference source on one case; tests/golden/make_golden_ref_live.py stores what they return.
HESSIAN_CASES = [(6, 40, 1), (50, 1500, 2), (120, 3000, 3)]
VOXEL_MAP_CASES = [(31, 1.0), (32, 0.5), (33, 2.0)]
H_FULL_MAX_W = 6         # a larger H is stored as H Z, its diagonal blocks and 200 of the others: the whole of it would not fit the file.
#                          The stored blocks are checked entry by entry at the tolerance; an entry outside them only through H Z, which
#                          misses an error in a single entry below about sum|Z[:, j]| / |Z[i, j]| (some 6W) times the tolerance.


def hessian_problem(W, V, seed):
    p = synth.make_problem(W, V, 0, seed=seed, visual=False)
    return p["vox_ptr"], p["pose_idx"], p["clusters"], p["poses"]


def hessian_probe(W, seed):
    """The fixed test matrix Z and the (i, j), i > j, of the off-diagonal blocks kept of a Hessian too large to store whole."""
    rng = np.random.default_rng(1000 + seed)
    Z = rng.standard_normal((6 * W, 8))
    lower = np.array([(i, j) for i in range(W) for j in range(i)])
    return Z, lower[np.sort(rng.choice(len(lower), size=min(len(lower), 200), replace=False))]


def blocks_at(H, ij):
    return np.array([H[6 * i:6 * i + 6, 6 * j:6 * j + 6] for i, j in ij])


def ref_hessian(W, V, seed):
    a = hessian_problem(W, V, seed)
    res, g, H, kept = balm_ref.lidar_hessian(*a, threads=(seed % 2 == 0))
    out = dict(res=res, g=g, kept=kept, lm_poses=balm_ref.lidar_damping_iter(*a))
    if W <= H_FULL_MAX_W:
        out["H"] = H
    else:
        Z, pick = hessian_probe(W, seed)
        out.update(HZ=H @ Z, H_absmax=np.abs(H).max(), H_diag=blocks_at(H, [(i, i) for i in range(W)]), H_pick=blocks_at(H, pick))
    return out


@pytest.mark.parametrize("W,V,seed", HESSIAN_CASES)
def test_live_hessian_and_lm_reference_source_vs_numpy(W, V, seed):
    a = hessian_problem(W, V, seed)
    R = recorded(f"hessian_{seed}")
    res, g, kept = float(R["res"]), R["g"], int(R["kept"])
    r, g_o, blocks = lo.acc_evaluate2(*a, W)
    H_o = lo.assemble_dense(blocks, W)
    res_sum = res * kept if seed % 2 == 0 else res
    tol = 1e-9 * np.abs(H_o).max()
    assert kept == V and abs(res_sum - r) <= 1e-9 * abs(r)
    assert np.abs(g - g_o).max() <= 1e-9 * np.abs(g_o).max()
    if "H" in R:
        assert np.abs(R["H"] - H_o).max() <= tol
    else:
        Z, pick = hessian_probe(W, seed)
        assert abs(float(R["H_absmax"]) - np.abs(H_o).max()) <= tol
        assert np.all(np.abs(R["HZ"] - H_o @ Z) <= tol * np.abs(Z).sum(0))      # implied by every entry within tol, not the converse
        assert np.abs(R["H_diag"] - blocks_at(H_o, [(i, i) for i in range(W)])).max() <= tol
        assert np.abs(R["H_pick"] - blocks_at(H_o, pick)).max() <= tol
    poses, _ = lo.damping_iter(*a)
    assert np.abs(R["lm_poses"] - poses).max() <= 1e-9


def scan_scene(seed):
    return synth.make_scan_scene(seed, W=6, n_per_scan=2000)


def ref_voxel_map(seed, voxel_size):
    scans, poses = scan_scene(seed)
    m = balm_ref.Map(scans, poses, voxel_size)
    vp, pi, cl, meta = m.export()
    m.close()
    path = np.full((len(meta["path"]), max([1] + [len(p) for p in meta["path"]])), -1, np.int64)
    for k, p in enumerate(meta["path"]):
        path[k, :len(p)] = p
    rel = ao.rel_poses(poses, np.array([0, len(scans)]))
    return dict(vox_ptr=vp, pose_idx=pi, clusters=cl, key=meta["key"], layer=meta["layer"], path=path,
                anchor_cloud_sorted=lex(balm_ref.anchor_cloud(scans, rel, 0.2)))


@pytest.mark.parametrize("seed,voxel_size", VOXEL_MAP_CASES)
def test_live_voxel_map_reference_source_vs_numpy(seed, voxel_size):
    scans, poses = scan_scene(seed)
    R = recorded(f"voxel_map_{seed}")
    ovp, opi, ocl, ometa = vox.voxelize_literal(scans, poses, voxel_size)
    assert np.array_equal(R["vox_ptr"], ovp) and np.array_equal(R["pose_idx"], opi) and np.abs(R["clusters"] - ocl).max() <= 1e-12 * np.abs(ocl).max()
    path = [tuple(int(x) for x in p if x >= 0) for p in R["path"]]
    assert np.array_equal(R["key"], ometa["key"]) and path == [tuple(p) for p in ometa["path"]] and np.array_equal(R["layer"], ometa["layer"])
    win_ptr = np.array([0, len(scans)])
    rel = ao.rel_poses(poses, win_ptr)
    assert np.array_equal(R["anchor_cloud_sorted"], lex(ao.anchor_clouds_literal(scans, rel, win_ptr, 0.2)[0]))
