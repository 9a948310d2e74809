"""The restated oracles against the REFERENCE'S OWN CODE.

oracle/_ref/libbalm_ref.so is the reference's src/benchmark/bavoxel.hpp + include/tools.hpp ($BALM_REFERENCE_DIR) compiled where
they lie (oracle/Makefile, oracle/ref_harness.cpp) against stand-ins for the absent Eigen / PCL / ROS headers
(oracle/ref_stubs: generic dense arithmetic, nothing of the reference). These tests pin
  oracle/balm_oracle.c       against  VOX_HESS::{push_voxel, left_evaluate_acc2, evaluate_only_residual},
                                      BALM2::{divide_thread_left, damping_iter}, Exp / Log, the LM solve line
  tests/assoc_ref.py         against  cut_voxel + OCTO_TREE_NODE::{recut, tras_opt} and OCTO_TREE_ROOT::marginalize
so a transcription error in a restatement shows up as a difference from the reference's source, not only from its
description. (What the stand-ins restate is Eigen's eigen-solver and pivoted LDLT; those agree with any correct
implementation to rounding, and H, g, r are invariant to the eigenvector signs.)"""
import os

import numpy as np
import pytest

import assoc_ref
import scenes
from oracle import oracle_py as orc
from oracle import ref_py as ref

pytestmark = pytest.mark.skipif(not ref.available(), reason="oracle/_ref/libbalm_ref.so not built (needs BALM_REFERENCE_DIR)")


def _pose_err(a, b):
    rot = max(np.linalg.norm(orc.log_so3(scenes.unpack_pose(x)[0].T @ scenes.unpack_pose(y)[0])) for x, y in zip(a, b))
    tra = max(np.linalg.norm(x[9:] - y[9:]) for x, y in zip(a, b))
    return rot, tra


def test_exp_log_match_the_reference():
    rng = np.random.default_rng(0)
    for phi in list(rng.normal(size=(6, 3))) + [np.zeros(3), np.array([1e-12, 0, 0]), np.array([0, 3.0, 0.5])]:
        assert np.abs(ref.exp_so3(phi) - orc.exp_so3(phi)).max() <= 1e-15
        R = orc.exp_so3(phi)
        assert np.abs(ref.log_so3(R) - orc.log_so3(R)).max() <= 1e-12


@pytest.mark.parametrize("n_poses,n_planes,drop,with_fix", [(6, 40, 0.0, False), (9, 60, 0.4, False), (8, 30, 0.3, True), (25, 80, 0.0, False),
                                                            (2, 20, 0.0, False), (3, 20, 0.0, True)])
def test_evaluators_match_the_reference(n_poses, n_planes, drop, with_fix):
    sc = scenes.make_scene(n_poses=n_poses, n_planes=n_planes, seed=17, drop=drop, with_fix=with_fix, pts_size=12)
    # the reference's push_voxel derives coe = sum of N itself (bavoxel.hpp:42-44): the scene's coe must be that
    coe = np.array([sc["obs10"][a:b, 9].sum() for a, b in zip(sc["row_ptr"][:-1], sc["row_ptr"][1:])])
    p = ref.Problem(n_poses, sc["row_ptr"], sc["pose_idx"], sc["obs10"], sc["fix10"])
    assert p.pushed() == n_planes and np.array_equal(p.coeffs(), coe)
    o = orc.Oracle(n_poses, sc["row_ptr"], sc["pose_idx"], sc["obs10"], coe, sc["fix10"])
    for x in (sc["poses_init"], sc["poses_gt"]):
        Hr, gr, rr = p.left_evaluate_acc2(x)
        Ho, go, ro = o.evaluate(x)                           # bavoxel.hpp's evaluator ignores the fix cluster (:325)
        assert abs(rr - ro) <= 1e-11 * abs(rr)
        assert np.abs(gr - go).max() <= 1e-10 * np.abs(gr).max()
        assert np.abs(Hr - Ho).max() <= 1e-10 * np.abs(Hr).max()
        assert abs(p.evaluate_only_residual(x) - o.residual(x)) <= 1e-11 * abs(rr)   # includes the fix cluster (:441)
    # voxel range semantics and the 4-thread split with its ordered reduction
    Hr, gr, rr = p.left_evaluate_acc2(sc["poses_init"], 3, 17)
    Ho, go, ro = o.evaluate(sc["poses_init"], 3, 17)
    assert abs(rr - ro) <= 1e-11 * abs(rr) and np.abs(Hr - Ho).max() <= 1e-10 * np.abs(Hr).max()
    Hr, gr, rr = p.divide_thread_left(sc["poses_init"])
    Ho, go, ro = o.evaluate_threads(sc["poses_init"], threads=4)
    assert abs(rr - ro) <= 1e-11 * abs(rr) and np.abs(gr - go).max() <= 1e-10 * np.abs(gr).max()
    assert np.abs(Hr - Ho).max() <= 1e-10 * np.abs(Hr).max()


def test_lm_solve_line_and_damping_iter_match_the_reference():
    sc = scenes.make_scene(n_poses=24, n_planes=600, seed=18, pts_size=10)       # >= 20 planes per pose (bavoxel.hpp:1079)
    coe = np.array([sc["obs10"][a:b, 9].sum() for a, b in zip(sc["row_ptr"][:-1], sc["row_ptr"][1:])])
    p = ref.Problem(24, sc["row_ptr"], sc["pose_idx"], sc["obs10"])
    o = orc.Oracle(24, sc["row_ptr"], sc["pose_idx"], sc["obs10"], coe)
    H, g, r = o.evaluate_threads(sc["poses_init"], threads=4)
    for u in (0.01, 1.0):
        dxr = ref.lm_solve(H, g, u)                          # D.diagonal() = Hess.diagonal(); (Hess + u*D).ldlt().solve(-JacT)
        dxo, _, _ = o.lm_step(H, g, u, sc["poses_init"])
        assert np.abs(dxr - dxo).max() <= 1e-9 * max(1e-3, np.abs(dxr).max())
    poses_r = p.damping_iter(sc["poses_init"])               # the reference's whole loop, gauge step included
    st, poses_o, tr, _ = o.damping_iter(sc["poses_init"], gauge_mode=0)
    assert st == 0 and len(tr) >= 3
    rot, tra = _pose_err(poses_r, poses_o)
    assert rot <= 1e-8 and tra <= 1e-8, (rot, tra)


def _session_from_scans(pts, frs, poses12, n, **kw):
    s = ref.Session(n, kw["voxel_size"], kw["layer_limit"], kw["min_ps"], kw["eigen_value_array"])
    for i in range(n):                                        # benchmark_realworld.cpp:187-188
        s.cut_voxel(pts[frs == i], poses12[i], i)
    s.recut(n)                                                # :196-197
    return s


@pytest.mark.parametrize("kw", [
    dict(voxel_size=2.0, layer_limit=2, min_ps=15, eigen_value_array=(1 / 16, 1 / 16, 1 / 16)),
    dict(voxel_size=2.0, layer_limit=2, min_ps=15, eigen_value_array=(1 / 16, 1 / 16, 1 / 9)),      # benchmark_realworld.cpp:183-185
    dict(voxel_size=1.0, layer_limit=1, min_ps=10, eigen_value_array=(1 / 16, 1 / 16, 1 / 16)),
])
def test_association_restatement_matches_the_reference_octree(kw):
    n = 8
    pts, frs, poses = assoc_ref.synthetic_scans(n_poses=n, pts_per_scan=4000, seed=21)
    poses12 = scenes.pack_poses([r for r, _ in poses], [p for _, p in poses])
    s = _session_from_scans(pts.astype(np.float32), frs, poses12, n, **kw)
    keys, rp, pi, ob, fx, co = s.export(n)                    # tras_opt -> push_voxel (:198)
    rp0, pi0, ob0, co0, keys0 = assoc_ref.cut_voxels(pts, frs, poses, **kw)
    assert len(keys) > 50
    assert np.array_equal(keys, keys0) and np.array_equal(rp, rp0) and np.array_equal(pi, pi0) and np.array_equal(co, co0)
    assert np.all(np.abs(ob - ob0) <= 1e-11 * np.abs(ob0).max(axis=0))
    assert not fx.any()


def test_marginalisation_restatement_matches_the_reference_octree():
    n, mg = 8, 2
    kw = dict(voxel_size=2.0, layer_limit=2, min_ps=15, eigen_value_array=(1 / 16, 1 / 16, 1 / 16))
    pts, frs, poses = assoc_ref.synthetic_scans(n_poses=n, pts_per_scan=4000, seed=22)
    poses12 = scenes.pack_poses([r for r, _ in poses], [p for _, p in poses])
    s = _session_from_scans(pts.astype(np.float32), frs, poses12, n, **kw)
    keys, rp, pi, ob, fx, co = s.export(n)
    rng = np.random.default_rng(1)                            # "optimised" poses: the retired clusters are re-transformed by them
    opt = poses12.copy()
    opt[:, 9:] += rng.normal(0, 0.01, (n, 3))
    s.marginalize(mg, opt, n)                                 # OCTO_TREE_ROOT::marginalize on every root (consistency.cpp:131-135)
    keys1, rp1, pi1, ob1, fx1, co1 = s.export(n - mg)         # the window now holds n - mg scans
    r_rp, r_pi, r_ob, r_fx, r_co = assoc_ref.marginalize_ref(n, rp, pi, ob, None, opt, mg, kw["min_ps"])
    assert np.array_equal(rp1, r_rp) and np.array_equal(pi1, r_pi) and np.array_equal(co1, r_co)
    assert np.array_equal(ob1, r_ob)
    assert np.abs(fx1 - r_fx).max() <= 1e-12 * np.abs(r_fx).max()


def test_append_restatement_matches_the_reference_octree_on_the_voxels_it_keeps():
    """balm_append_scan's contract (include/balm_b200.h) against the reference's persistent octree: after the window
    shifted, the NEW scan is cut into the tree (cut_voxel with fnum = its window slot, benchmark_realworld.cpp:187-188) and
    every node re-judged (recut :196-197). The device path only joins plane leaves that already exist -- it does not grow
    new roots or split a leaf that stopped being planar -- so: every voxel it keeps is a voxel the reference pushes, with
    identical observation rows; what the reference pushes beyond that are nodes that did not exist as plane leaves before."""
    n, mg = 8, 2
    kw = dict(voxel_size=2.0, layer_limit=2, min_ps=15, eigen_value_array=(1 / 16, 1 / 16, 1 / 16))
    pts, frs, poses = assoc_ref.synthetic_scans(n_poses=n + 1, pts_per_scan=4000, seed=23)
    poses12 = scenes.pack_poses([r for r, _ in poses], [p for _, p in poses])
    win = frs < n
    s = _session_from_scans(pts[win].astype(np.float32), frs[win], poses12[:n], n, **kw)
    keys, rp, pi, ob, fx, co, lay = s.export(n, with_layers=True)
    rp0, pi0, ob0, co0, keys0, lay0 = assoc_ref.cut_voxels(pts[win], frs[win], poses[:n], with_layers=True, **kw)
    assert np.array_equal(keys, keys0) and np.array_equal(lay, lay0)
    assert ((keys & 63) == 63).sum() > (lay == 0).sum()        # octant-7 leaves whose key digits look like "not split"
    s.marginalize(mg, poses12[:n], n)
    keys1, rp1, pi1, ob1, fx1, co1, lay1 = s.export(n - mg, with_layers=True)
    slot = n - mg
    shifted = np.vstack([poses12[mg:n], poses12[n:n + 1], poses12[n:n + 1]])
    new = pts[frs == n]
    s.cut_voxel(new.astype(np.float32), shifted[slot], slot)
    s.recut(slot + 1)
    keys2, rp2, pi2, ob2, fx2, co2, lay2 = s.export(slot + 1, with_layers=True)
    k, l, r_rp, r_pi, r_ob, r_fx, r_co, matched = assoc_ref.append_scan_ref(
        keys1, lay1, rp1, pi1, ob1, fx1, co1, new, shifted, slot, **kw)
    assert matched > 0.3 * len(new) and (r_pi == slot).sum() > 20
    where = {(int(a), int(b)): i for i, (a, b) in enumerate(zip(keys2, lay2))}
    for a in range(len(k)):
        i = where[(int(k[a]), int(l[a]))]                     # KeyError: a voxel the reference does not push
        assert np.array_equal(pi2[rp2[i]:rp2[i + 1]], r_pi[r_rp[a]:r_rp[a + 1]])
        assert np.array_equal(co2[i], r_co[a])
        assert np.all(np.abs(ob2[rp2[i]:rp2[i + 1]] - r_ob[r_rp[a]:r_rp[a + 1]]) <= 1e-11 * np.abs(r_ob).max(axis=0))
        assert np.abs(fx2[i] - r_fx[a]).max() <= 1e-12 * max(1.0, np.abs(r_fx[a]).max())
    before = {(int(a), int(b)) for a, b in zip(keys1, lay1)}
    kept = {(int(a), int(b)) for a, b in zip(k, l)}
    extra = [kl for kl in where if kl not in kept]
    assert all(kl not in before for kl in extra)              # nothing that WAS a plane leaf is pushed by the reference only
    assert len(kept) > 0.6 * len(where)


def test_repeated_marginalisation_matches_the_reference_octree():
    """Two window shifts in a row: after the first one many fix clusters hold >= 50 points, so the second exercises the
    rule that such a leaf no longer absorbs retired scans (to_margi, bavoxel.hpp:790) next to leaves that still do."""
    n, mg = 10, 2
    kw = dict(voxel_size=2.0, layer_limit=2, min_ps=15, eigen_value_array=(1 / 16, 1 / 16, 1 / 16))
    pts, frs, poses = assoc_ref.synthetic_scans(n_poses=n, pts_per_scan=3000, seed=24)
    poses12 = scenes.pack_poses([r for r, _ in poses], [p for _, p in poses])
    s = _session_from_scans(pts.astype(np.float32), frs, poses12, n, **kw)
    keys, rp, pi, ob, fx, co = s.export(n)
    rng = np.random.default_rng(2)
    cur = (rp, pi, ob, None)
    win, x = n, poses12.copy()
    for step in range(2):
        x = x.copy()
        x[:, 9:] += rng.normal(0, 0.005, x.shape[0:1] + (3,))
        s.marginalize(mg, x, win)                             # x: the window's optimised poses (x_poses)
        k1, rp1, pi1, ob1, fx1, co1 = s.export(win - mg)
        r_rp, r_pi, r_ob, r_fx, r_co = assoc_ref.marginalize_ref(win, cur[0], cur[1], cur[2], cur[3], x, mg, kw["min_ps"])
        assert np.array_equal(rp1, r_rp) and np.array_equal(pi1, r_pi) and np.array_equal(co1, r_co)
        assert np.array_equal(ob1, r_ob)
        assert np.abs(fx1 - r_fx).max() <= 1e-12 * np.abs(r_fx).max()
        if step == 0:
            big = fx1[:, 9] >= 50
            assert big.any() and (~big).any()                 # both kinds of leaves go into the second shift
        cur = (rp1, pi1, ob1, fx1)
        x = np.vstack([x[mg:], np.tile(x[-1], (mg, 1))])      # the window shifts (consistency.cpp:137-140); the tail is unused
        win -= mg


REALWORLD = os.path.join(os.environ.get("BALM_REFERENCE_DIR", "/nonexistent"), "datas", "benchmark_realworld")


@pytest.mark.skipif(not os.path.exists(os.path.join(REALWORLD, "alidarPose.csv")), reason="BALM_REFERENCE_DIR does not name a checkout with the dataset")
def test_association_restatement_matches_the_reference_octree_on_its_own_dataset():
    """The first 16 scans of datas/benchmark_realworld (every 4th point), re-anchored to pose 0 and cut with the constants
    of benchmark_realworld.cpp:163-185 (voxel_size 2, eigen ratios {1/16, 1/16, 1/9} stored as float): real lidar data has
    heavy-tailed leaves, negative coordinates and ratios that land close to the thresholds."""
    from balm_b200 import io
    n = 16
    R, p, t, scans = io.read_realworld_dir(REALWORLD, max_scans=n)
    R0, p0 = R[0].copy(), p[0].copy()
    poses = [(R0.T @ R[i], R0.T @ (p[i] - p0)) for i in range(n)]          # :163-168
    poses12 = scenes.pack_poses([r for r, _ in poses], [q for _, q in poses])
    pts = np.concatenate([sc[::4] for sc in scans]).astype(np.float32)
    frs = np.concatenate([np.full(len(sc[::4]), i, dtype=np.int32) for i, sc in enumerate(scans)])
    kw = dict(voxel_size=2.0, layer_limit=2, min_ps=15, eigen_value_array=(1 / 16, 1 / 16, 1 / 9))
    s = _session_from_scans(pts, frs, poses12, n, **kw)
    keys, rp, pi, ob, fx, co, lay = s.export(n, with_layers=True)
    rp0, pi0, ob0, co0, keys0, lay0 = assoc_ref.cut_voxels(pts.astype(np.float64), frs, poses, with_layers=True, **kw)
    assert len(keys) > 200 and len(np.unique(lay)) == 3
    assert np.array_equal(keys, keys0) and np.array_equal(lay, lay0)
    assert np.array_equal(rp, rp0) and np.array_equal(pi, pi0) and np.array_equal(co, co0)
    assert np.all(np.abs(ob - ob0) <= 1e-11 * np.abs(ob0).max(axis=0))


@pytest.mark.parametrize("fixture", ["realworld_voxels.npz", "realworld_c5_177.npz"])
def test_golden_fixtures_are_outputs_of_the_reference_code(fixture):
    """tests/golden/*.npz (plane voxels cut from the reference's dataset; what the GPU tests are held to per iteration) were
    written with the oracle's outputs. The reference's own VOX_HESS / BALM2 on the same inputs give the same residual,
    gradient, Hessian diagonal and final poses -- to rounding -- so the golden vectors ARE reference outputs."""
    d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", fixture))
    n = int(d["n_poses"])
    p = ref.Problem(n, d["row_ptr"], d["pose_idx"], d["obs10"])
    assert p.pushed() == len(d["coe"]) and np.array_equal(p.coeffs(), d["coe"])
    H, g, r = p.divide_thread_left(d["poses_init"])
    assert abs(r - float(d["oracle_residual0"])) <= 1e-13 * r
    assert np.abs(g - d["oracle_g0"]).max() <= 1e-12 * np.abs(g).max()
    assert np.abs(np.diag(H) - d["oracle_Hdiag0"]).max() <= 1e-12 * np.abs(np.diag(H)).max()
    assert abs(np.linalg.norm(H) - float(d["oracle_H0_fro"])) <= 1e-12 * np.linalg.norm(H)
    rot, tra = _pose_err(p.damping_iter(d["poses_init"]), d["oracle_poses"])   # BALM2::damping_iter, the whole loop
    assert rot <= 1e-10 and tra <= 1e-10, (rot, tra)


def test_restatement_fixture_is_output_of_the_reference_code():
    """tests/golden/restatement_outputs.npz (what tests/test_gpu_vs_restatement.py holds the GPU to) was written with the
    oracle and tests/assoc_ref.py. The reference's own VOX_HESS / BALM2 / octree on the same inputs give the same values."""
    import restated_cases as rc
    d = rc.load()
    for k, (n_poses, n_planes, drop, with_fix) in enumerate(rc.EVAL_SCENES):
        sc = rc.eval_scene(n_poses, n_planes, drop, with_fix)
        p = ref.Problem(n_poses, sc["row_ptr"], sc["pose_idx"], sc["obs10"], sc["fix10"])
        assert p.pushed() == n_planes and np.array_equal(p.coeffs(), rc.coe_of(sc))
        for name in ("poses_init", "poses_gt"):
            H, g, r = p.divide_thread_left(sc[name])
            assert abs(r - float(d[f"eval{k}_{name}_r"])) <= 1e-11 * abs(r)
            assert np.abs(g - d[f"eval{k}_{name}_g"]).max() <= 1e-10 * np.abs(g).max()
            assert np.abs(np.diag(H) - d[f"eval{k}_{name}_Hdiag"]).max() <= 1e-10 * np.abs(np.diag(H)).max()
            assert rc.probes_close(H, d[f"eval{k}_{name}_Hprobes"], 1e-10)
            assert abs(p.evaluate_only_residual(sc[name]) - float(d[f"eval{k}_{name}_residual"])) <= 1e-11 * abs(r)
        H, g, r = p.left_evaluate_acc2(sc["poses_init"], *rc.eval_range(n_planes))
        assert abs(r - float(d[f"eval{k}_range_r"])) <= 1e-11 * abs(r)
        assert rc.probes_close(H, d[f"eval{k}_range_Hprobes"], 1e-10)
    sc = rc.lm_scene()
    p = ref.Problem(24, sc["row_ptr"], sc["pose_idx"], sc["obs10"])
    rot, tra = _pose_err(p.damping_iter(sc["poses_init"]), d["lm_poses"])
    assert rot <= 1e-8 and tra <= 1e-8, (rot, tra)
    n, mg, kw = rc.ASSOC_N, rc.ASSOC_MG, rc.ASSOC_KW
    pts, frs, poses, poses12, opt = rc.assoc_inputs()
    s = _session_from_scans(pts.astype(np.float32), frs, poses12, n, **kw)
    keys, rp, pi, ob, fx, co, lay = s.export(n, with_layers=True)
    assert np.array_equal(keys, d["assoc_keys"]) and np.array_equal(lay, d["assoc_layers"])
    assert np.array_equal(rp, d["assoc_row_ptr"]) and np.array_equal(pi, d["assoc_pose_idx"])
    assert np.array_equal(co, d["assoc_coe"]) and rc.probes_close(ob, d["assoc_obs_probes"], 1e-11)
    s.marginalize(mg, opt, n)
    keys1, rp1, pi1, ob1, fx1, co1 = s.export(n - mg)
    assert np.array_equal(keys1, d["marg_keys"]) and np.array_equal(rp1, d["marg_row_ptr"])
    assert np.array_equal(pi1, d["marg_pose_idx"]) and np.array_equal(co1, d["marg_coe"])
    assert rc.probes_close(ob1, d["marg_obs_probes"], 1e-11) and rc.probes_close(fx1, d["marg_fix_probes"], 1e-12)


@pytest.mark.parametrize("n_poses,n_planes,drop,with_fix", [(6, 40, 0.0, False), (9, 60, 0.4, True)])
def test_right_update_restatement_matches_the_reference(n_poses, n_planes, drop, with_fix):
    """tests/numpy_acc2.py (the second reference-side pin of residual and gradient, used on the oracle and on the GPU path)
    against the reference's actual VOX_HESS::acc_evaluate2 (bavoxel.hpp:53-158)."""
    import numpy_acc2 as na
    sc = scenes.make_scene(n_poses=n_poses, n_planes=n_planes, seed=17, drop=drop, with_fix=with_fix, pts_size=12)
    coe = np.array([sc["obs10"][a:b, 9].sum() for a, b in zip(sc["row_ptr"][:-1], sc["row_ptr"][1:])])
    p = ref.Problem(n_poses, sc["row_ptr"], sc["pose_idx"], sc["obs10"], sc["fix10"])
    for x in (sc["poses_init"], sc["poses_gt"]):
        Hr, gr, rr = p.acc_evaluate2(x)
        g, r = na.acc_evaluate2(n_poses, sc["row_ptr"], sc["pose_idx"], sc["obs10"], coe, x, sc["fix10"])
        assert abs(r - rr) <= 1e-12 * abs(rr)
        assert np.abs(g - gr).max() <= 1e-12 * np.abs(gr).max()


# ---------------- the consistency experiment (src/simulation/BAs_left.hpp, toolss.hpp) ----------------
sim = pytest.mark.skipif(not ref.sim_available(), reason="oracle/_ref/libbalm_ref_sim.so not built (needs BALM_REFERENCE_DIR)")


@sim
def test_cluster_covariance_matches_the_reference_push():
    import numpy_cov as nc
    rng = np.random.default_rng(5)
    pts = rng.normal(size=(23, 3)) * [1.5, 0.4, 2.0] + [0.5, -1.0, 2.0]
    o10, cc = ref.sim_push_points(pts, 0.03)                 # PointCluster::push under POINT_NOISE (toolss.hpp:311-343)
    P = pts.T @ pts
    assert np.allclose(o10[:6], [P[0, 0], P[0, 1], P[0, 2], P[1, 1], P[1, 2], P[2, 2]], rtol=1e-13) and o10[9] == 23
    assert np.abs(nc.cluster_cov_isotropic(o10, 0.03) - cc).max() <= 1e-12 * np.abs(cc).max()


@sim
@pytest.mark.parametrize("drop,with_fix", [(0.0, False), (0.4, True)])
def test_covariance_jacobian_restatement_matches_the_reference(drop, with_fix):
    import numpy_cov as nc
    sc = scenes.make_scene(n_poses=6, n_planes=14, seed=9, drop=drop, with_fix=with_fix, pts_size=15)
    x = sc["poses_init"]
    cc = np.stack([nc.cluster_cov_isotropic(o10, 0.02) for o10 in sc["obs10"]])
    p = ref.SimProblem(6, sc["row_ptr"], sc["pose_idx"], sc["obs10"], sc["fix10"], cc)
    R_ref = p.left_jacobian_point(x)                         # VOX_HESS::left_jacobian_point (BAs_left.hpp:342-473), coe = 1
    ones = np.ones(len(sc["coe"]))
    R_np = nc.left_jacobian_point(6, sc["row_ptr"], sc["pose_idx"], sc["obs10"], ones, x, sc["fix10"], c_cov=cc)
    assert np.abs(R_ref - R_np).max() <= 1e-10 * np.abs(R_ref).max()
    half = nc.left_jacobian_point(6, sc["row_ptr"], sc["pose_idx"], sc["obs10"], ones, x, sc["fix10"], c_cov=cc, beg=3, end=11)
    assert np.abs(p.left_jacobian_point(x, 3, 11) - half).max() <= 1e-10 * np.abs(half).max()
    # the sim's evaluator keeps the fix cluster in C (BAs_left.hpp:183-185): the oracle's include_fix variant
    o = orc.Oracle(6, sc["row_ptr"], sc["pose_idx"], sc["obs10"], ones, sc["fix10"])
    Hr, gr, rr = p.left_evaluate_acc2(x)
    Ho, go, ro = o.evaluate(x, include_fix=True)
    assert abs(rr - ro) <= 1e-11 * abs(rr) and np.abs(gr - go).max() <= 1e-10 * np.abs(gr).max()
    assert np.abs(Hr - Ho).max() <= 1e-10 * np.abs(Hr).max()
