"""CPU: the statistical-outlier oracle (oracle/cleaning.py) on clouds whose answer is known by hand, the blocked kNN
search against the all-pairs one, and the parameter checks of the GPU entry points that fail before any launch."""
import numpy as np
import pytest
import torch

from oracle import cleaning as oc


def _lattice_with_spike():
    g = np.arange(10, dtype=np.float32)
    lat = np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3)
    spike = np.array([[4.5, 4.5, 104.5]], dtype=np.float32)  # 100 above the lattice's centre
    return np.concatenate([lat, spike])


def test_lattice_drops_only_the_spike():
    P = _lattice_with_spike()
    idx, st = oc.remove_statistical_outliers(P, 20, 10.0)
    assert idx.tolist() == list(range(1000))
    assert st["mean"] == pytest.approx(1.410, abs=5e-4)
    assert st["std"] == pytest.approx(2.828, abs=5e-4)
    assert st["threshold"] == pytest.approx(29.70, abs=5e-3)
    assert st["avg"][1000] > st["threshold"] > st["avg"][:1000].max()


def test_blocked_search_equals_all_pairs():
    rng = np.random.default_rng(3)
    clouds = [rng.random((3000, 3)).astype(np.float32),
              np.concatenate([rng.normal(size=(2500, 3)), 1e3 * rng.normal(size=(40, 3))]).astype(np.float32),
              np.repeat(rng.random((300, 3)), 7, axis=0).astype(np.float32),
              _lattice_with_spike()]
    for P in clouds:
        for k in (1, 20, 32):
            np.testing.assert_array_equal(oc.knn_mean_distance(P, k), oc.knn_mean_distance_all_pairs(P, k))
    q = rng.choice(3000, 50, replace=False)
    np.testing.assert_array_equal(oc.knn_mean_distance(clouds[0], 20, queries=q),
                                  oc.knn_mean_distance_all_pairs(clouds[0], 20)[q])


def test_exact_duplicates_have_zero_avg_but_count_in_valid():
    rng = np.random.default_rng(5)
    base = rng.random((200, 3)).astype(np.float32)
    dup = np.repeat(base[:1], 25, axis=0)  # 25 copies: their 20 nearest are all at distance 0
    P = np.concatenate([base[1:], dup])
    avg = oc.knn_mean_distance(P, 20)
    assert (avg[199:] == 0).all() and (avg[:199] > 0).all()
    idx, st = oc.remove_statistical_outliers(P, 20, 10.0)
    assert st["mean"] == pytest.approx(avg[avg > 0].sum() / P.shape[0], rel=1e-15)
    assert not np.isin(np.arange(199, 224), idx).any()
    assert idx.tolist() == sorted(idx.tolist())


def test_small_and_degenerate_clouds():
    assert oc.remove_statistical_outliers(np.zeros((0, 3), np.float32))[0].shape == (0,)
    idx, st = oc.remove_statistical_outliers(np.ones((1, 3), np.float32))
    assert idx.shape == (0,) and np.isnan(st["threshold"])
    assert oc.remove_statistical_outliers(np.full((50, 3), 2.5, np.float32))[0].shape == (0,)
    # N < k: every point averages over all N
    P = np.array([[0, 0, 0], [3, 0, 0], [0, 4, 0]], np.float32)
    avg = oc.knn_mean_distance(P, 20)
    np.testing.assert_allclose(avg, [(0 + 3 + 4) / 3, (0 + 3 + 5) / 3, (0 + 4 + 5) / 3], rtol=1e-15)


def test_parameter_errors():
    P = np.random.default_rng(1).random((10, 3)).astype(np.float32)
    for kw in ({"nb_neighbors": 0}, {"std_ratio": 0.0}, {"std_ratio": -1.0}):
        with pytest.raises(ValueError):
            oc.remove_statistical_outliers(P, **kw)


def test_colour_conversion():
    c = torch.tensor([[-3.0, 0.0, 0.99], [1.5, 254.999, 255.0], [300.0, 127.5, 12.0]], dtype=torch.float64)
    assert oc.convert_colours(c).tolist() == [[0, 0, 0], [1, 254, 255], [255, 127, 12]]
    assert oc.convert_colours(c).dtype == np.int32
    # the reference's /255 ... *255 round trip through Open3D is exact for every integer colour
    v = np.arange(256, dtype=np.int32)
    assert ((v / 255 * 255).astype(np.int32) == v).all()


def test_gpu_entry_points_reject_bad_parameters(lib):
    """Argument checks of the C ABI run on the host before any launch (no device needed)."""
    import ctypes
    from g2pc import capi
    fake = ctypes.c_void_p(256)  # never dereferenced: every call below fails its argument checks first
    for k in (0, 33, -1):
        assert lib.g2pc_knn_mean_distance(fake, 100, k, fake, fake, 1 << 30, None) == 1
    assert lib.g2pc_knn_mean_distance(fake, 1 << 31, 20, fake, fake, 1 << 62, None) == 1
    assert b"int32" in lib.g2pc_last_error()
    for r in (0.0, -1.0, float("nan")):
        assert lib.g2pc_outlier_mask(fake, 100, r, fake, fake, fake, 1 << 20, None) == 1
    assert lib.g2pc_outlier_mask(fake, 1 << 31, 10.0, fake, fake, fake, 1 << 20, None) == 1
    assert lib.g2pc_knn_workspace_bytes(1000, 20) > 1000 * 24 and lib.g2pc_knn_workspace_bytes(1000, 33) == 0
    with pytest.raises(capi.G2pcError):
        from g2pc import outliers
        outliers.knn_mean_distance(torch.zeros((4, 3)))  # a CPU tensor: no fallback
