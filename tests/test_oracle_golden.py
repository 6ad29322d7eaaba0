"""CPU: the oracle restatement against the committed golden vectors (outputs of the unmodified reference, generated
by tests/golden/make_golden.py)."""
import os

import numpy as np
import pytest
import torch

from util import GOLDEN


def _load(name):
    path = os.path.join(GOLDEN, name + ".npz")
    if not os.path.exists(path):
        pytest.skip(f"{path} missing")
    return np.load(path)


@pytest.mark.parametrize("name", ["sampling_a", "sampling_b"])
def test_sampling_oracle_matches_reference_golden(name):
    from g2pc import synth
    from oracle import gaussians as og, philox, sampling as osamp
    g = _load(name)
    n, scene_seed, num_points, exact, attempts, rng_seed = [int(v) for v in g["meta"]]
    sc = synth.make_scene(n, seed=scene_seed)
    cov0 = og.build_covariance(sc["scales"], sc["rots"])
    assert np.array_equal(cov0.numpy(), g["cov0"]), "covariance build differs from the reference (bit-exact on CPU)"
    nrm = og.calculate_normals(sc["scales"], sc["rots"])
    assert np.array_equal(nrm.numpy(), g["normals"])
    cov, keep = og.validate_covariances(cov0)
    assert np.array_equal(keep.numpy(), g["keep"])
    assert np.array_equal(cov.numpy(), g["cov"])
    mags = og.gaussian_magnitudes(cov, sc["opacities"])
    assert np.array_equal(mags.numpy(), g["magnitudes"])
    ppg = osamp.distribute_points(mags, num_points).to(torch.int32)
    assert np.array_equal(ppg.numpy(), g["ppg"])
    o = osamp.generate_pointcloud(sc["xyz"], cov, sc["colours"] * 255, nrm, mags, num_points, std=2.0,
                                  exact_num_points=bool(exact), num_sample_attempts=attempts,
                                  eps_fn=lambda gid, k, a: philox.draw_eps(gid, k, a, rng_seed, 0))
    assert o["points"].shape[0] == g["points"].shape[0], "emitted point count (integer output) must be exact"
    assert np.array_equal(o["points"].numpy(), g["points"]), "positions / order differ from the reference"
    assert np.array_equal(o["colours"].numpy().astype(np.float32), g["colours"])
    assert np.array_equal(o["normals"].numpy().astype(np.float32), g["point_normals"])
    # the sequence of MultivariateNormal calls (k, attempt, n') the reference made
    calls = []
    for (s, e, k, idx, tr) in o["bin_trace"]:
        if tr:
            calls += [(k - 1, a, len(todo)) for a, (todo, _, _, _) in enumerate(tr)]
    assert np.array_equal(np.array(calls, dtype=np.int64), g["mvn_calls"])


@pytest.mark.parametrize("name", ["colour_a", "colour_b"])
def test_colour_oracle_matches_reference_golden(name):
    """oracle/render.py against the unmodified reference renderer's outputs (tile parameters pinned to (60, 60000))."""
    from g2pc import synth
    from oracle import gaussians as og, render as orr
    g = _load(name)
    n, scene_seed, ncams, res = [int(v) for v in g["meta"]]
    sc = synth.make_scene(n, seed=scene_seed)
    cams, intr = synth.make_cameras(ncams)
    cov = og.build_covariance(sc["scales"], sc["rots"])
    for dense in (False, True):
        O = orr.PythonRendererOracle(sc["xyz"], sc["opacities"], sc["colours"], cov, dense=dense)
        for i, (c2w, k) in enumerate(zip(cams, intr)):
            img = O(orr.Camera(c2w, k, colour_resolution=res))
            assert np.abs(img - g["images"][i]).max() < 2e-6
        assert np.abs(O.gaussian_max_contribution - g["max_contribution"]).max() < 2e-6
        assert np.abs(O.gaussian_colours - g["colours"]).max() < 2e-6
        assert np.array_equal(O.gaussian_max_contribution > 0.05, g["visible"]), "visibility mask must be exact"


def _sh_inputs(n, seed):
    g = torch.Generator().manual_seed(seed)
    sh = (0.4 * torch.randn(n, 3, 16, generator=g)).float()
    d = torch.randn(n, 3, generator=g)
    return sh, (d / d.norm(dim=1, keepdim=True)).float()


def test_sh_colour_matches_reference_eval_sh():
    """oracle.render.sh_colour == clamp(eval_sh + 0.5, 0) of the reference (gauss_render.py:43-99), degrees 0-3:
    against the committed golden (outputs of the unmodified eval_sh)."""
    from oracle import render as orr
    g = np.load(os.path.join(GOLDEN, "sh_a.npz"))
    n, seed = [int(v) for v in g["meta"]]
    sh, d = _sh_inputs(n, seed)
    for deg in range(4):
        want = np.maximum(g[f"deg{deg}"] + np.float32(0.5), 0)
        got = orr.sh_colour(deg, sh[..., : (deg + 1) ** 2], d).numpy()
        assert np.abs(got - want).max() <= 2.4e-7, f"deg {deg}"  # same polynomial, fp32 association only


def test_philox_known_answers():
    """Random123 known-answer vectors for Philox4x32-10."""
    from oracle.philox import philox4x32_10
    z = np.uint32(0)
    f = np.uint32(0xFFFFFFFF)
    assert [int(v) for v in philox4x32_10(z, z, z, z, 0, 0)] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    assert [int(v) for v in philox4x32_10(f, f, f, f, 0xFFFFFFFF, 0xFFFFFFFF)] == [0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD]
    pi = philox4x32_10(np.uint32(0x243F6A88), np.uint32(0x85A308D3), np.uint32(0x13198A2E), np.uint32(0x03707344),
                       0xA4093822, 0x299F31D0)
    assert [int(v) for v in pi] == [0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1]


def test_eps_stream_statistics():
    from oracle.philox import draw_eps
    e = draw_eps(np.arange(4000), 64, 2, 42, 1)
    assert e.shape == (64, 4000, 3) and e.dtype == np.float32
    assert abs(float(e.mean())) < 5e-3 and abs(float(e.std()) - 1.0) < 5e-3
    acc = float((np.linalg.norm(e, axis=-1) <= 2.0).mean())
    assert abs(acc - 0.7385) < 5e-3  # P[chi_3 <= 2]
    # keyed by (gid, sample, attempt, call): independent of how the Gaussians are batched
    e2 = draw_eps(np.arange(1000, 1010), 64, 2, 42, 1)
    assert np.array_equal(e2, e[:, 1000:1010])


def test_live_reference_matches_oracle_small():
    """The oracle's generate_pointcloud with default arguments against the unmodified reference's (stored by
    tests/golden/make_golden.py: live_small), both drawing the same eps."""
    from g2pc import synth
    from oracle import gaussians as og, philox, sampling as osamp
    g = _load("live_small")
    n, scene_seed, num_points, rng_seed = [int(v) for v in g["meta"]]
    sc = synth.make_scene(n, seed=scene_seed)
    eps_fn = lambda gid, k, a: philox.draw_eps(gid, k, a, rng_seed, 0)
    cov, _ = og.validate_covariances(og.build_covariance(sc["scales"], sc["rots"]))
    nr = og.calculate_normals(sc["scales"], sc["rots"])
    o = osamp.generate_pointcloud(sc["xyz"], cov, sc["colours"] * 255, nr, og.gaussian_magnitudes(cov, sc["opacities"]),
                                  num_points, eps_fn=eps_fn)
    assert torch.equal(o["points"], torch.from_numpy(g["points"])) and torch.equal(o["colours"], torch.from_numpy(g["colours"]))
