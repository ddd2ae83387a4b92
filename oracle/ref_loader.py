"""Import the UNMODIFIED reference (facebookresearch/localrf) on CPU.

TEST / BENCH INFRASTRUCTURE ONLY.  Nothing under localrf_b200/ imports this file, and the repository contains
no reference source.  The reference is found in a checkout named by $LOCALRF_REFERENCE (the directory that
holds localTensoRF/), else as the bytecode that `compile_reference()` (run by __graft_entry__.build()) compiled
from such a checkout into the git-ignored oracle/_ref/.  Users: tests/golden/make_golden.py (which writes the
committed golden fixtures the GPU parity tests compare against), `bench.py --impl reference` / `reference_gpu` /
`cpu_baseline`, tests/test_bench_workloads.py and tests/test_gpu_renderer_loop.py.

The hot path's modules import a few packages that may be missing but are never *used* on the path
(kornia.create_meshgrid at utils/ray_utils.py:6, matplotlib / plyfile / skimage.measure at
utils/utils.py:10-12).  Empty stub modules are registered for those names so the reference files
import unmodified (SURVEY.md §8c).
"""
import importlib
import os
import sys
import types

COMPILED = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
DEFAULT_SOURCE = "/root/reference"        # default checkout location for compile_reference()
# the reference's modules on its render path (LocalTensorfs.forward and renderer.render)
MODULES = ["local_tensorfs", "renderer", "models/__init__", "models/tensorBase", "models/tensoRF",
           "utils/__init__", "utils/ray_utils", "utils/utils"]
REF_ROOT = os.environ.get("LOCALRF_REFERENCE") or COMPILED
REF_PKG = os.path.join(REF_ROOT, "localTensoRF")


def reference_available() -> bool:
    return any(os.path.isfile(os.path.join(REF_PKG, "local_tensorfs" + ext)) for ext in (".py", ".pyc"))


def compile_reference(src=None, verbose=True):
    """Byte-compile the reference's render-path modules from a checkout ($LOCALRF_REFERENCE, else
    DEFAULT_SOURCE) into oracle/_ref/localTensoRF/<module>.pyc: sourceless bytecode for this interpreter, which
    imports like the sources and contains none of them.  Without a checkout, oracle/_ref/ is left as it is."""
    import py_compile
    src = src or os.environ.get("LOCALRF_REFERENCE") or DEFAULT_SOURCE
    pkg = os.path.join(src, "localTensoRF")
    if not all(os.path.isfile(os.path.join(pkg, m + ".py")) for m in MODULES):
        if verbose:
            print(f"ref_loader: no reference checkout at {src}; oracle/_ref left as it is")
        return False
    for m in MODULES:
        dst = os.path.join(COMPILED, "localTensoRF", m + ".pyc")
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        py_compile.compile(os.path.join(pkg, m + ".py"), cfile=dst, dfile=os.path.join("localTensoRF", m + ".py"),
                           doraise=True)
    if verbose:
        print(f"ref_loader: {len(MODULES)} reference modules compiled into {COMPILED}")
    return True


def _stub(name, **attrs):
    try:
        importlib.import_module(name)
        return
    except Exception:
        pass
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    m.__path__ = []  # behave like a package so "import a.b" works
    sys.modules[name] = m
    if "." in name:
        parent, child = name.rsplit(".", 1)
        setattr(sys.modules[parent], child, m)


def load_reference():
    """Returns (TensorVMSplit, AlphaGridMask, LocalTensorfs, ray_utils module) of the reference."""
    if not reference_available():
        raise RuntimeError("no reference: run __graft_entry__.build() with a checkout of facebookresearch/localrf "
                           f"at $LOCALRF_REFERENCE or {DEFAULT_SOURCE}, or point LOCALRF_REFERENCE at one")
    _stub("kornia", create_meshgrid=lambda *a, **k: None)
    _stub("matplotlib", use=lambda *a, **k: None)
    _stub("matplotlib.pyplot")
    _stub("matplotlib.cm")
    _stub("plyfile")
    _stub("skimage")
    _stub("skimage.measure")
    _stub("imageio")
    _stub("lpips")
    if REF_PKG not in sys.path:
        sys.path.insert(0, REF_PKG)
    # the reference uses top-level names "models", "utils", "local_tensorfs"
    for clash in ("models", "utils", "local_tensorfs"):
        mod = sys.modules.get(clash)
        if mod is not None and not getattr(mod, "__file__", "").startswith(REF_PKG):
            del sys.modules[clash]
    from models.tensoRF import TensorVMSplit  # noqa
    from models.tensorBase import AlphaGridMask  # noqa
    from local_tensorfs import LocalTensorfs  # noqa
    import utils.ray_utils as ray_utils  # noqa
    return TensorVMSplit, AlphaGridMask, LocalTensorfs, ray_utils
