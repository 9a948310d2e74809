#!/usr/bin/env python
"""Writes tests/golden/restatement_outputs.npz: what the CPU oracle (oracle/balm_oracle.c) and the association
restatement (tests/assoc_ref.py) compute on the seeded inputs of tests/restated_cases.py. These are restatements of the
reference, not the reference's own output; tests/test_reference_pin.py compares the stored values with the reference's
compiled code wherever oracle/_ref is built. Large arrays are stored as probes (tests/restated_cases.probes)."""
import os
import sys

import numpy as np

TESTS = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.dirname(TESTS), TESTS]
import assoc_ref  # noqa: E402
import restated_cases as rc  # noqa: E402
from oracle import oracle_py as orc  # noqa: E402


def main():
    out = {}
    for k, (n_poses, n_planes, drop, with_fix) in enumerate(rc.EVAL_SCENES):
        sc = rc.eval_scene(n_poses, n_planes, drop, with_fix)
        o = orc.Oracle(n_poses, sc["row_ptr"], sc["pose_idx"], sc["obs10"], rc.coe_of(sc), sc["fix10"])
        for name in ("poses_init", "poses_gt"):
            H, g, r = o.evaluate_threads(sc[name], threads=4)               # divide_thread_left: 4 ranges, ordered sum
            out[f"eval{k}_{name}_r"] = r
            out[f"eval{k}_{name}_g"] = g
            out[f"eval{k}_{name}_Hdiag"] = np.diag(H).copy()
            out[f"eval{k}_{name}_Hprobes"] = rc.probes(H)
            out[f"eval{k}_{name}_residual"] = o.residual(sc[name])          # evaluate_only_residual: fix cluster included
        H, g, r = o.evaluate(sc["poses_init"], *rc.eval_range(n_planes))     # left_evaluate_acc2 on one voxel range
        out[f"eval{k}_range_r"] = r
        out[f"eval{k}_range_Hprobes"] = rc.probes(H)
    sc = rc.lm_scene()
    o = orc.Oracle(24, sc["row_ptr"], sc["pose_idx"], sc["obs10"], rc.coe_of(sc))
    st, poses, tr, _ = o.damping_iter(sc["poses_init"], gauge_mode=0)       # BALM2::damping_iter, gauge step included
    assert st == 0
    out["lm_poses"] = poses
    n, mg, kw = rc.ASSOC_N, rc.ASSOC_MG, rc.ASSOC_KW
    pts, frs, poses, poses12, opt = rc.assoc_inputs()
    rp, pi, ob, co, keys, lay = assoc_ref.cut_voxels(pts, frs, poses, with_layers=True, **kw)
    out.update(assoc_keys=keys, assoc_layers=lay, assoc_row_ptr=rp, assoc_pose_idx=pi, assoc_coe=co,
               assoc_obs_probes=rc.probes(ob))
    rp1, pi1, ob1, fx1, co1 = assoc_ref.marginalize_ref(n, rp, pi, ob, None, opt, mg, kw["min_ps"])
    kept = [a for a in range(len(co)) if (pi[rp[a]:rp[a + 1]] >= mg).sum() >= 2
            and ob[rp[a]:rp[a + 1]][pi[rp[a]:rp[a + 1]] >= mg, 9].sum() >= kw["min_ps"]]
    assert len(kept) == len(co1)
    out.update(marg_keys=keys[kept], marg_row_ptr=rp1, marg_pose_idx=pi1, marg_coe=co1, marg_obs_probes=rc.probes(ob1),
               marg_fix_probes=rc.probes(fx1))
    np.savez_compressed(rc.GOLDEN, **out)
    print("wrote", os.path.getsize(rc.GOLDEN), "bytes")


if __name__ == "__main__":
    main()
