#!/usr/bin/env python
"""Build the UNMODIFIED reference CUDA rasterizer for sm_100 into oracle/_ref/ (TEST INFRASTRUCTURE):

    G2PC_REFERENCE_ROOT=<reference checkout> python oracle/build_ref.py

  oracle/_ref/gaussian_pointcloud_rasterization/_C.cpython-*.so     the reference's compiled extension, nothing else

oracle/_ref/ is git-ignored and holds no reference source.  Only tests/golden/make_golden.py (the `ref_ext` vectors,
run on a GPU) and bench.py's reference legs load it; the product never does.

Build recipe of the extension (no source edit): copy gaussian-pointcloud-rasterization/ to a scratch dir and run its
own setup.py with  NVCC_APPEND_FLAGS="-include cstdint"  (rasterizer_impl.h:24,40-61 use std::uintptr_t / uint32_t
without <cstdint>; GCC 13 rejects that) and TORCH_CUDA_ARCH_LIST=10.0.
"""
import glob
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = os.environ.get("G2PC_REFERENCE_ROOT", "")
OUT = os.path.join(HERE, "_ref")
GPR = "gaussian-pointcloud-rasterization"


def _tree_hash(root):
    h = hashlib.sha256()
    for dp, dn, fn in sorted(os.walk(root)):
        if "third_party" in dp:
            continue
        for f in sorted(fn):
            if f.endswith((".cu", ".h", ".cpp", ".py")):
                h.update(f.encode())
                h.update(open(os.path.join(dp, f), "rb").read())
    return h.hexdigest()


def available():
    return bool(REF_ROOT) and os.path.isfile(os.path.join(REF_ROOT, GPR, "setup.py"))


def extension_path():
    """The built reference extension, or None."""
    so = glob.glob(os.path.join(OUT, "gaussian_pointcloud_rasterization", "_C*.so"))
    return so[0] if so else None


def build_extension(verbose=False):
    """Build the reference's CUDA extension for sm_100 with its own setup.py in a scratch copy."""
    pkg = os.path.join(OUT, "gaussian_pointcloud_rasterization")
    stamp = os.path.join(pkg, ".src_hash")
    want = _tree_hash(os.path.join(REF_ROOT, GPR))
    if extension_path() and os.path.exists(stamp) and open(stamp).read() == want:
        return extension_path()
    tmp = tempfile.mkdtemp(prefix="gpr_build_")
    src = os.path.join(tmp, "gpr")
    shutil.copytree(os.path.join(REF_ROOT, GPR), src)
    env = dict(os.environ)
    env["NVCC_APPEND_FLAGS"] = (env.get("NVCC_APPEND_FLAGS", "") + " -include cstdint").strip()
    env["TORCH_CUDA_ARCH_LIST"] = "10.0"
    env.setdefault("MAX_JOBS", "8")
    r = subprocess.run([sys.executable, "setup.py", "build_ext", "--inplace"], cwd=src, env=env,
                       stdout=None if verbose else subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0:
        raise RuntimeError("reference extension build failed:\n" + (r.stdout.decode()[-4000:] if r.stdout else ""))
    so = glob.glob(os.path.join(src, "gaussian_pointcloud_rasterization", "_C*.so"))
    if not so:
        raise RuntimeError("reference extension build produced no _C*.so")
    os.makedirs(pkg, exist_ok=True)
    for old in glob.glob(os.path.join(pkg, "_C*.so")):
        os.remove(old)
    dst = os.path.join(pkg, os.path.basename(so[0]))
    shutil.copyfile(so[0], dst)
    open(stamp, "w").write(want)
    shutil.rmtree(tmp, ignore_errors=True)
    return dst


def build(verbose=False):
    if not available():
        return None
    return build_extension(verbose)


if __name__ == "__main__":
    if not available():
        raise SystemExit("set G2PC_REFERENCE_ROOT to a checkout of the reference project")
    print(build(verbose="-v" in sys.argv))
