"""Host-side readers of the reference's on-disk formats (balm_b200/io.py; SURVEY 8f row N4). CPU only."""
import os

import numpy as np
import pytest

import scenes
from balm_b200 import drivers, io


def test_pcd_roundtrip_binary_and_ascii(tmp_path):
    rng = np.random.default_rng(1)
    xyz = rng.normal(0, 10, (257, 3)).astype(np.float32)
    inten = rng.uniform(0, 255, 257).astype(np.float32)
    for binary in (True, False):
        f = tmp_path / ("b.pcd" if binary else "a.pcd")
        io.write_pcd(f, xyz, inten, binary=binary)
        got, gi = io.read_pcd(f, want_intensity=True)
        assert got.dtype == np.float32 and np.array_equal(got, xyz) and np.array_equal(gi, inten)
    io.write_pcd(tmp_path / "e.pcd", np.zeros((0, 3)))
    assert io.read_pcd(tmp_path / "e.pcd").shape == (0, 3)


def test_pcd_other_layouts_and_errors(tmp_path):
    # x y z only, float64 z, an integer ring field in between
    n = 5
    dt = np.dtype([("x", np.float32), ("ring", np.uint16), ("y", np.float32), ("z", np.float64)])
    rec = np.zeros(n, dtype=dt)
    rec["x"], rec["y"], rec["z"], rec["ring"] = np.arange(n), -np.arange(n), 0.5 * np.arange(n), 7
    hdr = (f"VERSION 0.7\nFIELDS x ring y z\nSIZE 4 2 4 8\nTYPE F U F F\nCOUNT 1 1 1 1\nWIDTH {n}\nHEIGHT 1\n"
           f"POINTS {n}\nDATA binary\n")
    f = tmp_path / "m.pcd"
    f.write_bytes(hdr.encode() + rec.tobytes())
    got = io.read_pcd(f)
    assert np.array_equal(got, np.stack([rec["x"], rec["y"], rec["z"].astype(np.float32)], axis=1))
    f.write_bytes(hdr.encode() + rec.tobytes()[:-3])
    with pytest.raises(ValueError):
        io.read_pcd(f)
    f.write_bytes(hdr.replace("DATA binary", "DATA binary_compressed").encode() + rec.tobytes())
    with pytest.raises(ValueError):
        io.read_pcd(f)


def test_pose_csv_roundtrip_and_layout(tmp_path):
    rng = np.random.default_rng(2)
    R = np.stack([scenes.exp_so3(rng.normal(0, 0.5, 3)) for _ in range(6)])
    p = rng.normal(0, 3, (6, 3))
    t = np.arange(6) * 0.1
    f = tmp_path / "alidarPose.csv"
    io.write_pose_csv(f, R, p, t)
    lines = f.read_text().strip().splitlines()
    assert len(lines) == 24
    first = [float(x) for x in lines[0].split(",")]            # line 1 of a pose = first ROW of [R p]
    assert np.allclose(first, [R[0][0, 0], R[0][0, 1], R[0][0, 2], p[0][0]])
    f.write_text(f.read_text() + "1,2,3,4\n")                   # an incomplete trailing group is ignored
    R2, p2, t2 = io.read_pose_csv(f)
    assert np.array_equal(R2, R) and np.array_equal(p2, p) and np.array_equal(t2, t)


def test_pose_packing_and_rsme():
    rng = np.random.default_rng(3)
    R = np.stack([scenes.exp_so3(rng.normal(0, 0.5, 3)) for _ in range(4)])
    p = rng.normal(0, 3, (4, 3))
    P = drivers.pack_poses(R, p)
    assert np.array_equal(P, scenes.pack_poses(list(R), list(p)))
    R2, p2 = drivers.unpack_poses(P)
    assert np.array_equal(R2, R) and np.array_equal(p2, p)
    w = np.array([0.01, -0.02, 0.03])
    Rn = np.stack([r @ scenes.exp_so3(w) for r in R])
    rot, tran = drivers.rsme(drivers.pack_poses(Rn, p + 0.1), P)
    assert abs(rot - np.linalg.norm(w)) < 1e-9 and abs(tran - 0.1 * np.sqrt(3)) < 1e-12


REALWORLD = os.path.join(os.environ.get("BALM_REFERENCE_DIR", "/nonexistent"), "datas", "benchmark_realworld")


@pytest.mark.skipif(not os.path.isdir(REALWORLD), reason="BALM_REFERENCE_DIR does not name a checkout with the dataset")
def test_reads_the_reference_dataset():
    d = REALWORLD
    R, p, t = io.read_pose_csv(os.path.join(d, "alidarPose.csv"))
    assert len(R) == 177 and np.allclose(np.einsum("nij,nkj->nik", R, R), np.eye(3), atol=1e-5)  # the csv stores six decimals
    xyz = io.read_pcd(os.path.join(d, "full0.pcd"))
    assert xyz.dtype == np.float32 and xyz.shape[1] == 3 and len(xyz) > 10000 and np.isfinite(xyz).all()


def test_down_sampling_voxel_matches_the_sequential_definition():
    rng = np.random.default_rng(5)
    xyz = rng.normal(0, 0.2, (3000, 3)).astype(np.float32)
    vs = 0.05
    got = drivers.down_sampling_voxel(xyz, vs)
    cells = {}
    for q in xyz:  # tools.hpp:209-234, literally (float32 state)
        loc = q / np.float32(vs)
        loc = np.where(loc < 0, loc - np.float32(1.0), loc)
        k = tuple(int(x) for x in np.trunc(loc))
        if k not in cells:
            cells[k] = [q.copy(), np.float32(1.0)]
        else:
            m, c = cells[k]
            cells[k] = [(m * c + q) / (c + np.float32(1.0)), c + np.float32(1.0)]
    want = np.array([cells[k][0] for k in sorted(cells)])
    assert got.shape == want.shape and np.abs(got - want).max() < 2e-6
    assert drivers.down_sampling_voxel(xyz, 0.0).shape == xyz.shape          # below 1 mm: untouched (:205)


def test_data_show_reanchors_and_concatenates():
    R = np.stack([scenes.exp_so3(np.array([0.0, 0.0, 0.3 * i])) for i in range(3)])
    p = np.array([[1.0, 2.0, 3.0], [2.0, 2.0, 3.0], [3.0, 2.0, 3.0]])
    scans = [np.array([[1.0, 0.0, 0.0]], dtype=np.float32)] * 3
    cloud, path = drivers.data_show(drivers.pack_poses(R, p), scans)
    assert cloud.shape == (3, 3) and path.shape == (3, 3)
    assert np.allclose(path[0], 0) and np.allclose(path[2], [2, 0, 0], atol=1e-6)
    assert np.allclose(cloud[0], [1, 0, 0], atol=1e-6)
    assert np.allclose(cloud[1], R[1] @ [1, 0, 0] + [1, 0, 0], atol=1e-6)
