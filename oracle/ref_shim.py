"""Run the UNMODIFIED reference (the checkout named by $G2PC_REFERENCE_ROOT) on CPU (TEST INFRASTRUCTURE).

Used by tests/golden/make_golden.py to produce the committed golden vectors that pin the oracle, and by bench.py's
reference legs; the tests compare against those vectors and never need the reference itself.

What the shim does (no reference source is edited or copied):
  * stubs the three import-time modules the container lacks (configargparse, imageio, plyfile);
  * redirects the reference's hard-coded "cuda" devices (gauss_handler.py:13,30,50,87; gauss_render.py:196,441,476)
    to CPU by wrapping torch factory functions, Tensor.to, Tensor.get_device and the torch.cuda memory queries;
  * pins the python renderer's memory-derived tile parameters (gauss_render.py:440-444) through the patched
    torch.cuda.mem_get_info / memory_allocated:  (60000*175000, 0) -> max_gaussians_per_tile 60000, max_tile 60;
  * injects the product's counter-based normal draws into MultivariateNormal.sample (gauss_to_pc.py:149) via a
    subclass placed in the gauss_to_pc module namespace.
"""
import contextlib
import importlib
import os
import sys
import types

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
# the reference's compiled CUDA extension (oracle/build_ref.py; git-ignored)
STAGED_EXT_ROOT = os.path.join(_HERE, "_ref")
REF_ROOT = os.environ.get("G2PC_REFERENCE_ROOT", "")

_FACTORIES = ["zeros", "ones", "full", "eye", "tensor", "arange", "empty", "zeros_like", "ones_like", "full_like",
              "empty_like", "linspace", "rand", "randn", "as_tensor"]


def available():
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, "gauss_to_pc.py"))


def _is_cuda_dev(d):
    if isinstance(d, int):
        return True
    if isinstance(d, str):
        return d.startswith("cuda")
    if isinstance(d, torch.device):
        return d.type == "cuda"
    return False


@contextlib.contextmanager
def cpu_redirect(pinned_tiles=(60, 60000)):
    """Context manager: inside it every 'cuda' device request lands on the CPU."""
    saved = {}
    for name in _FACTORIES:
        orig = getattr(torch, name)
        saved[name] = orig

        def make(orig):
            def wrapped(*a, **kw):
                if "device" in kw and _is_cuda_dev(kw["device"]):
                    kw["device"] = "cpu"
                return orig(*a, **kw)
            return wrapped
        setattr(torch, name, make(orig))

    orig_to = torch.Tensor.to
    orig_get_device = torch.Tensor.get_device
    orig_device_ctor = None

    def to(self, *a, **kw):
        if a and _is_cuda_dev(a[0]) and not isinstance(a[0], torch.dtype):
            a = ("cpu",) + tuple(a[1:])
        if "device" in kw and _is_cuda_dev(kw["device"]):
            kw["device"] = "cpu"
        return orig_to(self, *a, **kw)

    torch.Tensor.to = to
    torch.Tensor.get_device = lambda self: 0
    mgi, mal, emc = torch.cuda.mem_get_info, torch.cuda.memory_allocated, torch.cuda.empty_cache
    total = pinned_tiles[1] * 175000
    torch.cuda.mem_get_info = lambda *a, **k: (total, total)
    torch.cuda.memory_allocated = lambda *a, **k: 0
    torch.cuda.empty_cache = lambda *a, **k: None
    try:
        yield
    finally:
        for name, orig in saved.items():
            setattr(torch, name, orig)
        torch.Tensor.to = orig_to
        torch.Tensor.get_device = orig_get_device
        torch.cuda.mem_get_info, torch.cuda.memory_allocated, torch.cuda.empty_cache = mgi, mal, emc


def _stub_modules():
    for name in ("configargparse", "imageio", "plyfile"):
        if name in sys.modules:
            continue
        try:
            importlib.import_module(name)
        except Exception:
            m = types.ModuleType(name)
            if name == "plyfile":
                m.PlyData = m.PlyElement = object
            if name == "configargparse":
                import argparse
                m.ArgumentParser = argparse.ArgumentParser
            sys.modules[name] = m


_ref_ext = None


def _load_reference_extension():
    """The reference's OWN package `gaussian_pointcloud_rasterization` (its wrapper from REF_ROOT, _C built by
    oracle/build_ref.py), imported under a private module object — the product ships a package of the same name."""
    global _ref_ext
    if _ref_ext is not None:
        return _ref_ext
    import importlib.util
    src_dir = os.path.join(REF_ROOT, "gaussian-pointcloud-rasterization", "gaussian_pointcloud_rasterization")
    pkg_dir = os.path.join(STAGED_EXT_ROOT, "gaussian_pointcloud_rasterization")
    init = os.path.join(src_dir, "__init__.py")
    if not (os.path.isfile(init) and os.path.isdir(pkg_dir)):
        return None
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k == "gaussian_pointcloud_rasterization"
             or k.startswith("gaussian_pointcloud_rasterization.")}
    try:
        spec = importlib.util.spec_from_file_location("gaussian_pointcloud_rasterization", init,
                                                      submodule_search_locations=[src_dir, pkg_dir])
        mod = importlib.util.module_from_spec(spec)
        sys.modules["gaussian_pointcloud_rasterization"] = mod
        spec.loader.exec_module(mod)  # imports ._C from pkg_dir
        _ref_ext = {k: v for k, v in sys.modules.items() if k == "gaussian_pointcloud_rasterization"
                    or k.startswith("gaussian_pointcloud_rasterization.")}
    finally:
        for k in list(sys.modules):
            if k == "gaussian_pointcloud_rasterization" or k.startswith("gaussian_pointcloud_rasterization."):
                sys.modules.pop(k)
        sys.modules.update(saved)
    return _ref_ext


@contextlib.contextmanager
def reference_extension():
    """Inside the context `import gaussian_pointcloud_rasterization` (the reference imports it lazily: gauss_render.py:470,
    camera_handler.py:73) resolves to the REFERENCE's package, not the product's."""
    ext = _load_reference_extension()
    if ext is None:
        raise RuntimeError("reference CUDA extension not built (oracle/build_ref.py)")
    names = [k for k in sys.modules if k == "gaussian_pointcloud_rasterization"
             or k.startswith("gaussian_pointcloud_rasterization.")]
    saved = {k: sys.modules.pop(k) for k in names}
    sys.modules.update(ext)
    try:
        yield ext["gaussian_pointcloud_rasterization"]
    finally:
        for k in ext:
            sys.modules.pop(k, None)
        sys.modules.update(saved)


_loaded = None


def load():
    """Import the reference modules (unmodified) and return them in a namespace."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError("reference not found: set G2PC_REFERENCE_ROOT to its checkout")
    _stub_modules()
    # the reference modules are top-level scripts; import them under their own names from REF_ROOT only
    names = ["gauss_handler", "gauss_render", "camera_handler", "gauss_dataloader", "transform_dataloader",
             "mask_dataloader", "gauss_to_pc"]
    saved_mods = {n: sys.modules.pop(n) for n in names if n in sys.modules}
    sys.path.insert(0, REF_ROOT)
    try:
        mods = {n: importlib.import_module(n) for n in names}
    finally:
        sys.path.remove(REF_ROOT)
        for n in names:  # keep the reference modules out of sys.modules so the product's same-named modules import
            sys.modules.pop(n, None)
        sys.modules.update(saved_mods)
    _loaded = types.SimpleNamespace(**mods)
    return _loaded


class EpsInjector:
    """Makes the reference draw the product's eps: a MultivariateNormal subclass whose sample() uses
    eps_fn(gids, k, attempt) instead of torch's global generator.  Gaussians are identified by matching the
    `loc` rows against the scene's means (synthetic scenes have unique means)."""

    def __init__(self, ref, xyz_all, eps_fn, gid_offset=0):
        self.ref = ref
        self.eps_fn = eps_fn
        self.gid_offset = gid_offset
        x = np.ascontiguousarray(torch.as_tensor(xyz_all).numpy().astype(np.float32))
        self.lookup = {x[i].tobytes(): i for i in range(x.shape[0])}
        assert len(self.lookup) == x.shape[0], "means must be unique for eps injection"
        self.attempt = 0
        self.log = []

    def __enter__(self):
        inj = self
        g2p = self.ref.gauss_to_pc
        self._orig_mvn = g2p.MultivariateNormal
        self._orig_create = g2p.create_new_gaussian_points
        base = self._orig_mvn

        class InjectedMVN(base):
            def sample(self, sample_shape=torch.Size()):
                k = int(sample_shape[0])
                loc = np.ascontiguousarray(self.loc.numpy().astype(np.float32))
                gids = np.array([inj.lookup[loc[i].tobytes()] for i in range(loc.shape[0])], dtype=np.int64)
                eps = torch.as_tensor(inj.eps_fn(gids + inj.gid_offset, k, inj.attempt))
                inj.log.append((k, inj.attempt, gids))
                inj.attempt += 1
                # rsample arithmetic of torch 2.11 multivariate_normal.py:251-254, with the injected eps
                from torch.distributions.multivariate_normal import _batch_mv
                return self.loc + _batch_mv(self._unbroadcasted_scale_tril, eps)

        def create_wrapper(*a, **kw):
            inj.attempt = 0  # the attempt counter restarts for every bin (gauss_to_pc.py:189)
            return inj._orig_create(*a, **kw)

        g2p.MultivariateNormal = InjectedMVN
        g2p.create_new_gaussian_points = create_wrapper
        return self

    def __exit__(self, *exc):
        g2p = self.ref.gauss_to_pc
        g2p.MultivariateNormal = self._orig_mvn
        g2p.create_new_gaussian_points = self._orig_create
        return False
