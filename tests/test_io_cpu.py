"""CPU: the thin host-side loaders (3dgs-to-pc_b200/gauss_dataloader.py, transform_dataloader.py) — self-consistency and
equality with the reference's own parsers on generated COLMAP / transforms.json files (their outputs are stored in
tests/golden/transforms.npz by tests/golden/make_golden.py)."""
import json
import os
import struct

import numpy as np
import pytest
import torch


def write_gaussian_ply(path, sc, sh_degree=3):
    """A 3DGS-style binary PLY from a g2pc.synth scene (inverse of load_ply_data)."""
    n = sc["xyz"].shape[0]
    k = (sh_degree + 1) ** 2
    names = ["x", "y", "z", "nx", "ny", "nz", "f_dc_0", "f_dc_1", "f_dc_2"] + [f"f_rest_{i}" for i in range(3 * (k - 1))] + \
            ["opacity", "scale_0", "scale_1", "scale_2", "rot_0", "rot_1", "rot_2", "rot_3"]
    arr = np.zeros(n, dtype=[(nm, "<f4") for nm in names])
    xyz = sc["xyz"].numpy()
    arr["x"], arr["y"], arr["z"] = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    shs = sc["shs"].numpy()
    for c in range(3):
        arr[f"f_dc_{c}"] = shs[:, c, 0]
    rest = shs[:, :, 1:k].reshape(n, -1)
    for i in range(rest.shape[1]):
        arr[f"f_rest_{i}"] = rest[:, i]
    o = sc["opacities"].double().numpy()
    arr["opacity"] = np.log(o / (1 - o))
    for i in range(3):
        arr[f"scale_{i}"] = sc["scales"].numpy()[:, i]
    for i in range(4):
        arr[f"rot_{i}"] = sc["rots"].numpy()[:, i]
    with open(path, "wb") as f:
        f.write(("ply\nformat binary_little_endian 1.0\n" + f"element vertex {n}\n" +
                 "".join(f"property float {nm}\n" for nm in names) + "end_header\n").encode())
        f.write(arr.tobytes())


def write_transforms_json(path, cams, intr):
    frames = [{"file_path": f"images/frame_{i:04d}.png", "transform_matrix": c.tolist()} for i, c in enumerate(cams)]
    json.dump({"w": intr[0][0], "h": intr[0][1], "fl_x": intr[0][2], "fl_y": intr[0][3], "frames": frames}, open(path, "w"))


def test_ply_roundtrip(tmp_path):
    import gauss_dataloader as gd
    from g2pc import synth
    sc = synth.make_scene(500, seed=3, sh_degree=3)
    p = str(tmp_path / "scene.ply")
    write_gaussian_ply(p, sc)
    xyz, scales, rots, colours, opac, shs = gd.load_ply_data(p, max_sh_degree=3, device="cpu")
    assert xyz.dtype == torch.float32 and scales.dtype == torch.float64 and opac.dtype == torch.float32
    assert torch.equal(xyz, sc["xyz"])
    assert float((scales - sc["scales"]).abs().max()) < 1e-6
    assert float((opac - sc["opacities"]).abs().max()) < 1e-6
    assert shs.shape == (500, 3, 16) and float((shs - sc["shs"]).abs().max()) < 1e-6
    assert float((colours - sc["colours"]).abs().max()) < 1e-6
    assert float((rots.norm(dim=1) - 1).abs().max()) < 1e-9


def test_save_ply_layout(tmp_path):
    import gauss_dataloader as gd
    n = 1234
    g = torch.Generator().manual_seed(0)
    pts = torch.randn(n, 3, generator=g)
    nrm = torch.randn(n, 3, generator=g)
    col = torch.rand(n, 3, generator=g) * 255
    p = str(tmp_path / "out.ply")
    gd.save_xyz_to_ply(pts, p, rgb_colors=col, normals_points=nrm, chunk_size=500, quiet=True)
    v = gd.read_ply_vertices(p)
    assert v.shape[0] == n and v.dtype.names == ("x", "y", "z", "nx", "ny", "nz", "red", "green", "blue")
    assert np.array_equal(np.stack([v["x"], v["y"], v["z"]], 1), pts.numpy())
    assert np.array_equal(np.stack([v["nx"], v["ny"], v["nz"]], 1), nrm.numpy())
    assert np.array_equal(np.stack([v["red"], v["green"], v["blue"]], 1), col.numpy().astype(np.uint8))


def _write_colmap(dirpath, cams_c2w, binary):
    """COLMAP images/cameras files whose parsed poses equal the given OpenGL c2w matrices is not required — only that
    both parsers read the same numbers; so arbitrary quaternions / translations are written."""
    os.makedirs(dirpath, exist_ok=True)
    rng = np.random.default_rng(1)
    recs = []
    for i in range(len(cams_c2w)):
        q = rng.normal(size=4)
        q /= np.linalg.norm(q)
        recs.append((i + 1, *q, *rng.normal(size=3), 1, f"img_{i:03d}.jpg"))
    if binary:
        with open(os.path.join(dirpath, "cameras.bin"), "wb") as f:
            f.write(struct.pack("<Q", 1))
            f.write(struct.pack("<iiQQdddd", 1, 1, 1920, 1080, 1600.0, 1590.0, 960.0, 540.0))
        with open(os.path.join(dirpath, "images.bin"), "wb") as f:
            f.write(struct.pack("<Q", len(recs)))
            for r in recs:
                f.write(struct.pack("<idddddddi", r[0], *r[1:8], r[8]))
                f.write(r[9].encode() + b"\x00")
                f.write(struct.pack("<Q", 2))
                f.write(struct.pack("<ddqddq", 1.0, 2.0, -1, 3.0, 4.0, -1))
    else:
        with open(os.path.join(dirpath, "cameras.txt"), "w") as f:
            f.write("# Camera list\n1 PINHOLE 1920 1080 1600.0 1590.0 960.0 540.0\n")
        with open(os.path.join(dirpath, "images.txt"), "w") as f:
            f.write("# Image list\n")
            for r in recs:
                f.write(" ".join(str(v) for v in r) + "\n")
                f.write("1.0 2.0 -1 3.0 4.0 -1\n")


def write_transform_files(dirpath, kind):
    """The camera file(s) of one loader kind for 7 synthetic cameras; returns the path to load."""
    from g2pc import synth
    cams, intr = synth.make_cameras(7)
    if kind == "json":
        path = os.path.join(dirpath, "transforms.json")
        write_transforms_json(path, cams, intr)
    else:
        path = os.path.join(dirpath, kind)
        _write_colmap(path, cams, binary=(kind == "colmap_bin"))
    return path


@pytest.mark.parametrize("kind", ["json", "colmap_txt", "colmap_bin"])
def test_transform_loaders_match_reference(tmp_path, kind):
    import transform_dataloader as td
    from g2pc import synth
    from util import GOLDEN
    cams, intr = synth.make_cameras(7)
    path = write_transform_files(str(tmp_path), kind)
    g = np.load(os.path.join(GOLDEN, "transforms.npz"))
    for skip in (0, 2):
        tr, ik = td.load_transform_data(path, skip_rate=skip)
        assert len(tr) >= 1 and set(tr.keys()) <= set(ik.keys())
        for k, m in tr.items():
            assert np.asarray(m).shape == (4, 4)
        rnames = [str(v) for v in g[f"{kind}_skip{skip}_names"]]
        rc2w, rik = g[f"{kind}_skip{skip}_c2w"], g[f"{kind}_skip{skip}_intrinsics"]
        assert list(tr.keys()) == rnames
        for i, k in enumerate(tr):
            assert np.allclose(np.asarray(tr[k], dtype=np.float64), rc2w[i], atol=1e-12)
            assert [float(v) for v in ik[k]] == [float(v) for v in rik[i]]
    if kind == "json":
        tr, ik = td.load_transform_data(path)
        assert np.allclose(np.asarray(tr["frame_0003"]), cams[3].numpy())
        assert ik["frame_0003"] == [1920, 1080, 1600.0, 1600.0]
