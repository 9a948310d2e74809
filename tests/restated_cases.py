"""Seeded inputs of tests/test_gpu_vs_reference.py and the stored restatement outputs on them.

tests/golden/restatement_outputs.npz (written by tests/golden/make_restatement_fixture.py) holds what the CPU oracle and
tests/assoc_ref.py compute on these inputs. tests/test_gpu_vs_restatement.py holds the CUDA path to those values on any
B200; tests/test_reference_pin.py checks them against the reference's own compiled code wherever oracle/_ref is built."""
import os

import numpy as np

import assoc_ref
import scenes

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "restatement_outputs.npz")
EVAL_SCENES = [(6, 40, 0.0, False), (37, 64, 0.0, False), (20, 200, 0.4, False), (12, 50, 0.3, True)]
ASSOC_KW = dict(voxel_size=2.0, layer_limit=2, min_ps=15, eigen_value_array=(1 / 16, 1 / 16, 1 / 16))
ASSOC_N, ASSOC_MG = 8, 2


def load():
    d = np.load(GOLDEN)
    return {k: d[k] for k in d.files}


def coe_of(sc):  # the reference's push_voxel derives the weight itself: sum of N over the voxel (bavoxel.hpp:42-44)
    return np.array([sc["obs10"][a:b, 9].sum() for a, b in zip(sc["row_ptr"][:-1], sc["row_ptr"][1:])])


def probes(A):
    """Column sums and a fixed weighted sum over the rows of a 2-D array (H, obs10, fix10)."""
    A = np.asarray(A, dtype=np.float64)
    return np.stack([A.sum(0), np.cos(np.arange(len(A)) * 0.7) @ A])


def probes_close(A, stored, tol):
    """A's probes against stored ones, relative to max |A| times the row count."""
    return np.abs(probes(A) - stored).max() <= tol * np.abs(A).max() * len(A)


def eval_scene(n_poses, n_planes, drop, with_fix):
    return scenes.make_scene(n_poses=n_poses, n_planes=n_planes, seed=31, drop=drop, with_fix=with_fix, pts_size=12)


def eval_range(n_planes):
    return n_planes // 5, n_planes // 2                      # voxel range of one worker thread


def lm_scene():
    return scenes.make_scene(n_poses=24, n_planes=600, seed=18, pts_size=10)   # >= 20 planes per pose (bavoxel.hpp:1079)


def assoc_inputs():
    """-> scan points, frame of each point, poses (R, p), the same packed, the "optimised" poses the window retires with."""
    pts, frs, poses = assoc_ref.synthetic_scans(n_poses=ASSOC_N, pts_per_scan=4000, seed=22)
    poses12 = scenes.pack_poses([r for r, _ in poses], [p for _, p in poses])
    rng = np.random.default_rng(1)
    opt = poses12.copy()
    opt[:, 9:] += rng.normal(0, 0.01, (ASSOC_N, 3))
    return pts, frs, poses, poses12, opt
