"""Build the UNMODIFIED reference CUDA extensions for sm_100a into oracle/_ref/.

TEST INFRASTRUCTURE ONLY.  Compiles the four reference extensions from the
sources where they lie under /root/reference (never copied into this repo):

    modules/radnerfs/raymarching/src/{raymarching.cu,bindings.cpp}   -> _raymarching_face
    modules/radnerfs/encoders/gridencoder/src/{gridencoder.cu,bindings.cpp} -> _gridencoder
    modules/radnerfs/encoders/shencoder/src/{shencoder.cu,bindings.cpp}   -> _shencoder
    modules/radnerfs/encoders/freqencoder/src/{freqencoder.cu,bindings.cpp} -> _freqencoder

Beside them, the UNMODIFIED reference Python of the path (PY_FILES below: renderer / radnerf / radnerf_torso /
cond_encoder / utils, the raymarching + encoder Function wrappers and utils/commons/hparams) is mirrored, byte for byte
and at build time only, into oracle/_ref/pyref/ so that the reference's own `RADNeRFTorso.render()` can run on the GPU
box where /root/reference does not exist (oracle/ref_model.py imports it from there).  oracle/_ref/ is git-ignored:
no reference source enters the repository history.

The only deviation from the reference's own JIT recipe (raymarching/backend.py:6-12)
is -std=c++17 instead of c++14 (torch 2.11 headers need C++17) and the explicit
sm_100a arch.  Outputs go to oracle/_ref/<name>/<name>.so (git-ignored, shipped
to the GPU box by gpurun).  The compiled reference is the GPU-side parity oracle
and the "kernel to beat"; nothing in the product path imports it.
"""
import os
import sys
import shutil

REF = os.environ.get("GF_REFERENCE_ROOT", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")

EXTS = {
    "_raymarching_face": "modules/radnerfs/raymarching/src",
    "_gridencoder": "modules/radnerfs/encoders/gridencoder/src",
    "_shencoder": "modules/radnerfs/encoders/shencoder/src",
    "_freqencoder": "modules/radnerfs/encoders/freqencoder/src",
}
CU = {
    "_raymarching_face": "raymarching.cu",
    "_gridencoder": "gridencoder.cu",
    "_shencoder": "shencoder.cu",
    "_freqencoder": "freqencoder.cu",
}


# reference Python mirrored (unmodified) into oracle/_ref/pyref/, relative to the reference root
PY_FILES = [
    "modules/radnerfs/renderer.py", "modules/radnerfs/radnerf.py", "modules/radnerfs/radnerf_torso.py",
    "modules/radnerfs/cond_encoder.py", "modules/radnerfs/utils.py",
    "modules/radnerfs/raymarching/__init__.py", "modules/radnerfs/raymarching/raymarching.py", "modules/radnerfs/raymarching/backend.py",
    "modules/radnerfs/encoders/encoding.py",
    "modules/radnerfs/encoders/gridencoder/__init__.py", "modules/radnerfs/encoders/gridencoder/grid.py", "modules/radnerfs/encoders/gridencoder/backend.py",
    "modules/radnerfs/encoders/shencoder/__init__.py", "modules/radnerfs/encoders/shencoder/sphere_harmonics.py", "modules/radnerfs/encoders/shencoder/backend.py",
    "modules/radnerfs/encoders/freqencoder/__init__.py", "modules/radnerfs/encoders/freqencoder/freq.py", "modules/radnerfs/encoders/freqencoder/backend.py",
    "utils/commons/hparams.py", "utils/commons/os_utils.py",
]


def mirror_python():
    """Byte-for-byte mirror of PY_FILES into oracle/_ref/pyref (namespace packages, like the reference tree)."""
    dst_root = os.path.join(OUT, "pyref")
    n = 0
    for rel in PY_FILES:
        src = os.path.join(REF, rel)
        dst = os.path.join(dst_root, rel)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        if not os.path.exists(dst) or open(src, "rb").read() != open(dst, "rb").read():
            shutil.copyfile(src, dst)
            n += 1
    print("[oracle/_ref] pyref: %d files mirrored (%d refreshed)" % (len(PY_FILES), n))


def built(name):
    return os.path.exists(os.path.join(OUT, name + ".so"))


def build_one(name, verbose=False):
    os.environ["TORCH_CUDA_ARCH_LIST"] = "10.0a"
    from torch.utils.cpp_extension import load
    src = os.path.join(REF, EXTS[name])
    bdir = os.path.join(OUT, "build_" + name)
    os.makedirs(bdir, exist_ok=True)
    load(
        name=name,
        sources=[os.path.join(src, CU[name]), os.path.join(src, "bindings.cpp")],
        extra_cflags=["-O3", "-std=c++17"],
        extra_cuda_cflags=["-O3", "-std=c++17", "-U__CUDA_NO_HALF_OPERATORS__",
                           "-U__CUDA_NO_HALF_CONVERSIONS__", "-U__CUDA_NO_HALF2_OPERATORS__"],
        build_directory=bdir,
        verbose=verbose,
        is_python_module=False,   # do not import here; tests import from oracle/_ref
    )
    shutil.copy(os.path.join(bdir, name + ".so"), os.path.join(OUT, name + ".so"))


def main(names=()):
    """Build the named extensions (all four by default); a no-op where the reference tree is absent."""
    if not os.path.isdir(REF):
        print("reference tree not present (%s): skipping oracle/_ref build" % REF)
        return 0
    os.makedirs(OUT, exist_ok=True)
    mirror_python()
    names = list(names) or list(EXTS)
    for n in names:
        if built(n):
            print("[oracle/_ref] %s already built" % n)
            continue
        print("[oracle/_ref] building %s ..." % n, flush=True)
        build_one(n, verbose=False)
        print("[oracle/_ref] %s done" % n, flush=True)
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
