"""GPU: point-cloud cleaning (csrc/s9_knn.cu through the C ABI, g2pc/outliers.py, mesh_handler.clean_point_cloud and the
CLI's --clean_pointcloud) against the float64 oracle oracle/cleaning.py.

Tolerances: avg within 1e-6 relative (the kernel selects on float32 distances and recomputes the chosen ones in float64);
mean / std within 1e-9 relative; the keep mask identical except for points whose avg lies within 1e-6 relative of the
threshold (their count is printed; 0 expected)."""
import numpy as np
import pytest
import torch

from oracle import cleaning as oc

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _sampler_cloud(n_gauss, num_points, seed):
    """The sampler's own output on a synthetic scene (10 % floaters): (points, colours, normals) on the device."""
    import gauss_handler as gh
    import gauss_to_pc as g2p
    from g2pc import synth
    sc = synth.make_scene(n_gauss, seed=seed, sh_degree=0)
    d = {k: v.to(DEV) for k, v in sc.items()}
    G = gh.Gaussians(d["xyz"], d["scales"], d["rots"], d["colours"] * 255, d["opacities"])
    G.calculate_normals()
    G.validate_covariances()
    return g2p.generate_pointcloud(G, num_points, quiet=True)


def _cloud(name):
    g = torch.Generator().manual_seed(7)
    if name == "sampler":
        return _sampler_cloud(2000, 20000, 41)[0].cpu()
    if name == "identical":
        return torch.full((20000, 3), 1.25)
    if name == "two_clusters":
        return torch.cat([torch.randn(10000, 3, generator=g), 1e6 + torch.randn(10000, 3, generator=g)])
    if name == "line":
        return torch.rand(20000, 1, generator=g) * torch.tensor([[1.0, 2.0, -3.0]]) + 0.5
    if name == "plane":
        return torch.cat([torch.rand(20000, 2, generator=g) * 4.0, torch.zeros(20000, 1)], 1)
    if name == "offset":  # float32 spacing is 1.0 at 1e7: a lattice-like cloud far from the origin
        return 1e7 + torch.rand(20000, 3, generator=g) * 1e4
    if name == "duplicates":
        base = torch.randn(1500, 3, generator=g)
        return base[torch.randint(0, 1500, (20000,), generator=g)]
    if name == "n7":
        return torch.randn(7, 3, generator=g)
    if name == "n1":
        return torch.randn(1, 3, generator=g)
    if name == "n20013":
        return torch.randn(20013, 3, generator=g) * torch.tensor([[5.0, 1.0, 0.2]])
    raise KeyError(name)


CLOUDS = ["sampler", "identical", "two_clusters", "line", "plane", "offset", "duplicates", "n7", "n1", "n20013"]


def _check_avg(gpu, ref):
    gpu = gpu.cpu().numpy()
    assert np.isfinite(gpu).all()
    err = np.abs(gpu - ref)
    bad = err > 1e-6 * np.abs(ref)
    assert not bad.any(), f"{int(bad.sum())} rows off, worst rel {float((err / np.maximum(ref, 1e-300)).max()):.2e}"


@pytest.mark.parametrize("name", CLOUDS)
def test_knn_mean_distance_matches_brute_force(lib, name):
    from g2pc import outliers
    pts = _cloud(name).to(torch.float32).contiguous()
    avg = outliers.knn_mean_distance(pts.to(DEV), 20)
    _check_avg(avg, oc.knn_mean_distance(pts.numpy(), 20))


@pytest.mark.parametrize("k", [1, 5, 12, 25, 32])
def test_knn_other_k(lib, k):
    from g2pc import outliers
    pts = _cloud("n20013")
    _check_avg(outliers.knn_mean_distance(pts.to(DEV), k), oc.knn_mean_distance(pts.numpy(), k))


def _check_stats_and_mask(avg_ref, stats, index, std_ratio):
    mean, std, thr, keep = oc.outlier_stats(avg_ref, std_ratio)
    assert stats["mean"] == pytest.approx(mean, rel=1e-9) and stats["std"] == pytest.approx(std, rel=1e-9)
    got = np.zeros(avg_ref.shape[0], dtype=bool)
    got[index.cpu().numpy()] = True
    near = np.abs(avg_ref - thr) <= 1e-6 * thr
    print(f"[clean] n {avg_ref.shape[0]} kept {int(got.sum())} (oracle {int(keep.sum())}), threshold {thr:.6g}, "
          f"{int(near.sum())} points within 1e-6 of the threshold")
    assert ((got != keep) & ~near).sum() == 0


@pytest.mark.parametrize("name,std_ratio", [("sampler", 10.0), ("sampler", 1.0), ("duplicates", 3.0), ("n20013", 2.0)])
def test_stats_and_mask(lib, name, std_ratio):
    from g2pc import outliers
    pts = _cloud(name).to(torch.float32).contiguous()
    index, stats = outliers.remove_statistical_outliers(pts.to(DEV), 20, std_ratio)
    assert index.dtype == torch.int64 and bool((index[1:] > index[:-1]).all())
    _check_stats_and_mask(oc.knn_mean_distance(pts.numpy(), 20), stats, index, std_ratio)


def test_edge_clouds(lib):
    from g2pc import outliers
    for n in (0, 1):
        idx, _ = outliers.remove_statistical_outliers(torch.zeros((n, 3), device=DEV))
        assert idx.shape == (0,)
    idx, st = outliers.remove_statistical_outliers(_cloud("identical").to(DEV))
    assert idx.shape == (0,) and st["mean"] == 0.0
    bad = _cloud("n20013").to(DEV)
    bad[123, 1] = float("nan")
    with pytest.raises(Exception, match="non-finite"):
        outliers.remove_statistical_outliers(bad)
    with pytest.raises(Exception):
        outliers.remove_statistical_outliers(bad[:10].cpu())
    for kw in ({"nb_neighbors": 0}, {"nb_neighbors": 33}, {"std_ratio": 0.0}):
        with pytest.raises(Exception):
            outliers.remove_statistical_outliers(_cloud("n7").to(DEV), **kw)


def test_clean_point_cloud_outputs_and_reruns(lib):
    import mesh_handler
    pts, cols, nrm = _sampler_cloud(2000, 20000, 43)
    cols = cols.clone()
    cols[:7] = torch.tensor([-4.0, 255.7, 300.0], dtype=cols.dtype, device=DEV)  # out-of-range colours are clamped
    p1, c1, n1 = mesh_handler.clean_point_cloud(pts, cols, nrm)
    p2, c2, n2 = mesh_handler.clean_point_cloud(pts, cols, nrm)
    assert torch.equal(p1, p2) and torch.equal(c1, c2) and torch.equal(n1, n2)
    idx, _ = oc.remove_statistical_outliers(pts.cpu().numpy(), 20, 10.0)
    assert 0 < idx.shape[0] < pts.shape[0]
    assert p1.dtype == pts.dtype and n1.dtype == nrm.dtype and c1.dtype == torch.int32
    np.testing.assert_array_equal(p1.cpu().numpy(), pts.cpu().numpy()[idx])
    np.testing.assert_array_equal(n1.cpu().numpy(), nrm.cpu().numpy()[idx])
    np.testing.assert_array_equal(c1.cpu().numpy(), oc.convert_colours(cols.cpu())[idx])
    p3, c3, n3 = mesh_handler.clean_point_cloud(pts, cols, None)
    assert n3 is None and torch.equal(p3, p1) and torch.equal(c3, c1)


def test_ten_million_points_with_scattered_outliers(lib):
    """The C3 cloud size: generate_pointcloud on a 3M-Gaussian scene, plus 0.1 % points scattered over 100x the scene's
    extent.  avg of 2000 random rows and of every injected outlier against the oracle's subset query; the statistics
    against the oracle's reduction of the kernel's own avg (a full float64 kNN at 10M is out of reach on the CPU)."""
    from g2pc import outliers
    pts = _sampler_cloud(3_000_000, 10_000_000, 1236)[0]
    n0 = pts.shape[0]
    g = torch.Generator().manual_seed(11)
    ext = float((pts.max(0).values - pts.min(0).values).max())
    no = n0 // 1000
    scatter = ((torch.rand(no, 3, generator=g) * 2 - 1) * 50 * ext).to(DEV)  # a cube 100x the scene's extent
    cloud = torch.cat([pts, scatter]).contiguous()
    n = cloud.shape[0]
    avg = outliers.knn_mean_distance(cloud, 20)
    rows = np.concatenate([np.random.default_rng(12).choice(n0, 2000, replace=False), np.arange(n0, n)])
    host = cloud.cpu().numpy()
    ref = oc.knn_mean_distance(host, 20, queries=rows)
    _check_avg(avg[torch.as_tensor(rows, device=DEV)], ref)
    index, stats = outliers.remove_statistical_outliers(cloud, 20, 10.0)
    _check_stats_and_mask(avg.cpu().numpy(), stats, index, 10.0)
    kept_outliers = int((index >= n0).sum())
    print(f"[clean 10M] n {n}: kept {index.shape[0]}, injected outliers kept {kept_outliers} of {no}")
    index2, _ = outliers.remove_statistical_outliers(cloud, 20, 10.0)
    assert torch.equal(index, index2)


def test_cli_clean_pointcloud(lib, tmp_path):
    """main(--clean_pointcloud) writes the oracle-cleaned rows of the cloud the same seed gives without the flag;
    --generate_mesh is still rejected."""
    import gauss_dataloader as gd
    import gauss_to_pc as g2p
    from g2pc import sampler, synth
    from test_io_cpu import write_gaussian_ply, write_transforms_json
    sc = synth.make_scene(3000, seed=23, sh_degree=3)
    cams, intr = synth.make_cameras(3)
    ply, tj = str(tmp_path / "scene.ply"), str(tmp_path / "transforms.json")
    out_u, out_c = str(tmp_path / "raw.ply"), str(tmp_path / "clean.ply")
    write_gaussian_ply(ply, sc)
    write_transforms_json(tj, cams, intr)
    common = ["--input_path", ply, "--transform_path", tj, "--num_points", "30000", "--colour_quality", "tiny", "--quiet"]
    sampler.reset_call_counter(0)
    g2p.main(common + ["--output_path", out_u])
    sampler.reset_call_counter(0)
    g2p.main(common + ["--output_path", out_c, "--clean_pointcloud"])
    vu, vc = gd.read_ply_vertices(out_u), gd.read_ply_vertices(out_c)
    xyz = np.stack([vu["x"], vu["y"], vu["z"]], 1)
    idx, st = oc.remove_statistical_outliers(xyz, 20, 10.0)
    near = np.abs(st["avg"] - st["threshold"]) <= 1e-6 * st["threshold"]
    print(f"[clean cli] {vu.shape[0]} -> {vc.shape[0]} rows (oracle {idx.shape[0]}), {int(near.sum())} near the threshold")
    assert int(near.sum()) == 0
    assert vc.dtype == vu.dtype
    np.testing.assert_array_equal(vc, vu[idx])
    with pytest.raises(AttributeError):
        g2p.config_parser(["--input_path", ply, "--transform_path", tj, "--generate_mesh"])
