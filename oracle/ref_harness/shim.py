"""Run the *reference's own* operator code on the CPU, in this container only.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).  Nothing here is shipped and
nothing is copied from /root/reference: the reference's modules are imported
from where they lie, under

  * a minimal stand-in for the ``chainer`` names those modules touch
    (``chainer.Function`` call protocol, forward-only ``chainer.functions``
    backed by NumPy, ``chainer.Link``/``Parameter``), because chainer itself is
    not installable here, and
  * a stand-in for ``cupy`` whose ``ElementwiseKernel`` takes the CUDA-C source
    string the reference hands it, wraps it in a serial ``for (i...)`` loop with
    serial definitions of atomicAdd/Min/Max/Exch/CAS, compiles it with g++
    (``-ffp-contract=off``) into ``oracle/_ref/`` and runs it.  The arithmetic
    executed is therefore the reference's kernel text, in thread order
    i = 0..n-1 (one legal schedule of the GPU execution; for the racy
    index-selection kernels it is the schedule the oracle's tie-break mirrors).

Used by gen_golden.py to produce tests/golden/*.npz and the SHA-256 record
of them that tests/test_oracle_vs_reference.py checks.
"""

import ctypes
import hashlib
import importlib
import os
import re
import subprocess
import sys
import types

import numpy as np

REF_ROOT = os.environ.get("MOREFUSION_REFERENCE", "/root/reference")
_HERE = os.path.dirname(os.path.abspath(__file__))
REF_BUILD = os.path.join(os.path.dirname(_HERE), "_ref")


def reference_available():
    return os.path.isdir(os.path.join(REF_ROOT, "morefusion", "functions"))


# --------------------------------------------------------------------------
# forward-only Variable: an ndarray that also answers .array / .data
# --------------------------------------------------------------------------
class Var(np.ndarray):
    def __new__(cls, x):
        return np.asarray(x).view(cls)

    @property
    def array(self):
        return np.asarray(self)

    @property
    def data(self):
        return np.asarray(self)


_wrap = Var


def _unwrap(x):
    return np.asarray(x)


# --------------------------------------------------------------------------
# cupy.ElementwiseKernel emulation
# --------------------------------------------------------------------------
_CTYPES = {"float32": "float", "int32": "int", "int8": "signed char",
           "float64": "double", "int64": "long long", "bool": "bool"}
_NPTYPES = {"float32": np.float32, "int32": np.int32, "int8": np.int8,
            "float64": np.float64, "int64": np.int64}

_PRELUDE = r"""
#include <math.h>
#include <cmath>
#include <cstddef>
#include <algorithm>
using std::size_t;
#define __device__
#define __forceinline__ inline
template <typename T> static inline T atomicAdd(T* a, T v) { T o = *a; *a = o + v; return o; }
template <typename T, typename U> static inline T atomicAdd(T* a, U v) { T o = *a; *a = o + (T)v; return o; }
template <typename T> static inline T atomicMin(T* a, T v) { T o = *a; if (v < o) *a = v; return o; }
template <typename T> static inline T atomicMax(T* a, T v) { T o = *a; if (v > o) *a = v; return o; }
template <typename T> static inline T atomicExch(T* a, T v) { T o = *a; *a = v; return o; }
template <typename T, typename U> static inline T atomicExch(T* a, U v) { T o = *a; *a = (T)v; return o; }
template <typename T> static inline T atomicCAS(T* a, T c, T v) { T o = *a; if (o == c) *a = v; return o; }
"""


def _parse_params(s):
    out = []
    for tok in [t.strip() for t in s.replace("\n", " ").split(",") if t.strip()]:
        parts = tok.split()
        raw = parts[0] == "raw"
        if raw:
            parts = parts[1:]
        out.append((raw, parts[0], parts[1]))
    return out


class ElementwiseKernel:
    def __init__(self, in_params, out_params, operation, name="kernel",
                 preamble="", **kw):
        self.in_params = _parse_params(in_params)
        self.out_params = _parse_params(out_params)
        self.operation = operation
        self.name = name
        self.preamble = preamble

    def __call__(self, *args):
        params = self.in_params + self.out_params
        assert len(args) == len(params), (self.name, len(args), len(params))
        n_in = len(self.in_params)
        # resolve generic T from the first array bound to it
        tname = None
        for (raw, ty, nm), a in zip(params, args):
            if ty == "T" and isinstance(a, np.ndarray) and a.ndim > 0:
                tname = a.dtype.name
                break
        if tname is None:
            tname = "float32"

        def cty(ty):
            return _CTYPES[tname if ty == "T" else ty]

        def npty(ty):
            return _NPTYPES[tname if ty == "T" else ty]

        size = None
        kinds, keep = [], []
        for k, ((raw, ty, nm), a) in enumerate(zip(params, args)):
            is_out = k >= n_in
            arr = np.asarray(a)
            if raw:
                kinds.append("raw")
            elif arr.ndim == 0 and not is_out:
                kinds.append("scalar")
            else:
                kinds.append("elem")
                if size is None:
                    size = arr.size
                else:
                    assert size == arr.size, (self.name, nm, size, arr.size)
        assert size is not None, self.name

        sig, body_decl, call_args = [], [], []
        for k, ((raw, ty, nm), a) in enumerate(zip(params, args)):
            is_out = k >= n_in
            c = cty(ty)
            if kinds[k] == "scalar":
                sig.append(f"const {c} {nm}")
                call_args.append(("scalar", npty(ty)(np.asarray(a)), c))
                continue
            if isinstance(a, np.ndarray) and a.flags.c_contiguous and a.dtype == npty(ty):
                arr = a                      # in place (outputs must alias)
            else:
                assert not is_out, (self.name, nm, "output must be contiguous/typed")
                arr = np.ascontiguousarray(np.asarray(a), dtype=npty(ty))
            keep.append(arr)
            if kinds[k] == "raw":
                sig.append(f"{c}* {nm}")
            else:
                sig.append(f"{c}* _p_{nm}")
                body_decl.append(f"{c}& {nm} = _p_{nm}[i];")
            call_args.append(("ptr", arr, c))

        src = (
            _PRELUDE + f"typedef {_CTYPES[tname]} T;\n" + self.preamble
            + "\nstatic inline void _body(const long long _i, "
            + ", ".join(sig) + ") {\n  const int i = (int)_i;\n  "
            + "\n  ".join(body_decl) + "\n" + self.operation + "\n}\n"
            + 'extern "C" void run(long long n, void** a) {\n'
            + "  for (long long i = 0; i < n; ++i) _body(i"
        )
        for j, (kind, val, c) in enumerate(call_args):
            if kind == "scalar":
                src += f", *({c}*)a[{j}]"
            else:
                src += f", ({c}*)a[{j}]"
        src += ");\n}\n"

        fn = _compile(self.name, src)
        holders = []
        ptrs = (ctypes.c_void_p * len(call_args))()
        for j, (kind, val, c) in enumerate(call_args):
            if kind == "scalar":
                h = np.array([val])
                holders.append(h)
                ptrs[j] = h.ctypes.data
            else:
                ptrs[j] = val.ctypes.data
        fn(ctypes.c_longlong(size), ptrs)
        return None


_LIBS = {}


def _compile(name, src):
    h = hashlib.sha1(src.encode()).hexdigest()[:16]
    key = f"{name}_{h}"
    if key in _LIBS:
        return _LIBS[key]
    os.makedirs(REF_BUILD, exist_ok=True)
    so = os.path.join(REF_BUILD, key + ".so")
    if not os.path.exists(so):
        cpp = os.path.join(REF_BUILD, key + ".cpp")
        with open(cpp, "w") as f:
            f.write(src)
        subprocess.check_call(
            ["g++", "-O1", "-ffp-contract=off", "-fno-fast-math", "-shared",
             "-fPIC", "-w", "-o", so, cpp])
    lib = ctypes.CDLL(so)
    lib.run.argtypes = [ctypes.c_longlong, ctypes.c_void_p]
    lib.run.restype = None
    _LIBS[key] = lib.run
    return lib.run


def _elementwise(in_params, out_params, operation, name, **kw):
    return ElementwiseKernel(in_params, out_params, operation, name, **kw)


# --------------------------------------------------------------------------
# fake module tree
# --------------------------------------------------------------------------
def _make_cupy():
    m = types.ModuleType("cupy")
    for k in dir(np):
        if not k.startswith("_"):
            try:
                setattr(m, k, getattr(np, k))
            except Exception:
                pass
    m.ElementwiseKernel = ElementwiseKernel
    m.ndarray = np.ndarray
    return m


class _Function:
    """chainer.Function call protocol, forward only; ``mode`` picks
    forward_cpu / forward_gpu for classes that define both."""

    mode = "cpu"

    def retain_inputs(self, *a, **k):
        pass

    def retain_outputs(self, *a, **k):
        pass

    def check_type_forward(self, in_types):
        pass

    def forward(self, inputs):
        gpu = hasattr(self, "forward_gpu")
        cpu = hasattr(self, "forward_cpu")
        if gpu and (_Function.mode == "gpu" or not cpu):
            return self.forward_gpu(inputs)
        return self.forward_cpu(inputs)

    def backward(self, inputs, gy):
        gpu = hasattr(self, "backward_gpu")
        cpu = hasattr(self, "backward_cpu")
        if gpu and (_Function.mode == "gpu" or not cpu):
            return self.backward_gpu(inputs, gy)
        return self.backward_cpu(inputs, gy)

    def __call__(self, *inputs):
        ins = tuple(_unwrap(x) for x in inputs)
        self._ins = ins
        outs = self.forward(ins)
        outs = tuple(_wrap(o) for o in outs)
        return outs[0] if len(outs) == 1 else outs


def set_mode(mode):
    assert mode in ("cpu", "gpu")
    _Function.mode = mode


class _Link:
    def __init__(self):
        self.xp = sys.modules["cupy"]

    class _Scope:
        def __enter__(self):
            return self

        def __exit__(self, *a):
            return False

    def init_scope(self):
        return _Link._Scope()

    def __call__(self, *a, **k):
        return self.forward(*a, **k)


def _make_F():
    F = types.ModuleType("chainer.functions")
    F.sum = lambda x, axis=None, keepdims=False: _wrap(np.sum(_unwrap(x), axis=axis, keepdims=keepdims))
    F.sqrt = lambda x: _wrap(np.sqrt(_unwrap(x)))
    F.min = lambda x, axis=None: _wrap(np.min(_unwrap(x), axis=axis))
    F.relu = lambda x: _wrap(np.maximum(_unwrap(x), 0))
    F.minimum = lambda a, b: _wrap(np.minimum(_unwrap(a), _unwrap(b)))
    F.maximum = lambda a, b: _wrap(np.maximum(_unwrap(a), _unwrap(b)))
    F.repeat = lambda x, n, axis=None: _wrap(np.repeat(_unwrap(x), n, axis=axis))
    F.concat = lambda xs, axis=1: _wrap(np.concatenate([_unwrap(x) for x in xs], axis=axis))
    F.stack = lambda xs, axis=0: _wrap(np.stack([_unwrap(x) for x in xs], axis=axis))
    F.matmul = lambda a, b: _wrap(np.matmul(_unwrap(a), _unwrap(b)))
    F.mean = lambda x, axis=None: _wrap(np.mean(_unwrap(x), axis=axis))
    return F


_INSTALLED = False


def install():
    """Install the stand-in modules and empty ``morefusion`` package shells so
    that reference *leaf* modules import without their package __init__s."""
    global _INSTALLED
    if _INSTALLED:
        return
    assert reference_available(), REF_ROOT
    cupy = _make_cupy()
    sys.modules["cupy"] = cupy

    chainer = types.ModuleType("chainer")
    chainer.Function = _Function
    chainer.Link = _Link
    chainer.Chain = _Link
    chainer.Variable = Var
    chainer.Parameter = lambda x: _wrap(np.array(x))
    F = _make_F()
    chainer.functions = F
    backends = types.ModuleType("chainer.backends")
    cuda = types.ModuleType("chainer.backends.cuda")
    cuda.cupy = cupy
    cuda.get_array_module = lambda *a: cupy
    cuda.elementwise = _elementwise
    cuda.to_cpu = lambda x: np.asarray(x)
    cuda.to_gpu = lambda x: np.asarray(x)
    backends.cuda = cuda
    chainer.backends = backends
    chainer.cuda = cuda
    utils = types.ModuleType("chainer.utils")
    tc = types.ModuleType("chainer.utils.type_check")
    tc.expect = lambda *a, **k: None
    utils.type_check = tc
    chainer.utils = utils
    sys.modules.update({
        "chainer": chainer, "chainer.functions": F, "chainer.backends": backends,
        "chainer.backends.cuda": cuda, "chainer.cuda": cuda,
        "chainer.utils": utils, "chainer.utils.type_check": tc,
    })

    # trimesh.transformations: only quaternion_from_matrix / translation_from_matrix
    # are touched (ICC link __init__); provided by the oracle's restatement.
    from .. import transforms as _tfm
    trimesh = types.ModuleType("trimesh")
    ttf = types.ModuleType("trimesh.transformations")
    ttf.quaternion_from_matrix = _tfm.quaternion_from_matrix
    ttf.translation_from_matrix = lambda M: np.array(M, copy=True)[:3, 3]
    trimesh.transformations = ttf
    sys.modules["trimesh"] = trimesh
    sys.modules["trimesh.transformations"] = ttf
    # trimesh.voxel.ops: the two index <-> point helpers get_target_grids touches
    # (contrib/multi_instance_octree_mapping.py:64-70); trimesh>=3.5 (requirements.txt:23) defines
    # them as indices * pitch + origin and round((points - origin) / pitch).astype(int).
    tvox = types.ModuleType("trimesh.voxel")
    tops = types.ModuleType("trimesh.voxel.ops")
    tops.matrix_to_points = lambda matrix, pitch, origin: (
        np.column_stack(np.nonzero(matrix)) * pitch + np.asanyarray(origin, dtype=np.float64))
    tops.points_to_indices = lambda points, pitch, origin: np.round(
        (np.asanyarray(points, dtype=np.float64) - np.asanyarray(origin, dtype=np.float64)) / pitch).astype(int)
    tvox.ops = tops
    trimesh.voxel = tvox
    sys.modules["trimesh.voxel"] = tvox
    sys.modules["trimesh.voxel.ops"] = tops
    # octomap (octomap-python, requirements.txt:11): absent; the oracle's restatement of the
    # OcTree calls the reference makes stands in, so that the reference's OWN grid-assembly code
    # (get_target_grids) runs on top of it.
    from .. import octomap as _octomap
    sys.modules["octomap"] = _octomap

    base = os.path.join(REF_ROOT, "morefusion")
    for name, sub in [
        ("morefusion", ""), ("morefusion.functions", "functions"),
        ("morefusion.functions.geometry", "functions/geometry"),
        ("morefusion.contrib", "contrib"), ("morefusion.functions.loss", "functions/loss"),
    ]:
        pkg = types.ModuleType(name)
        pkg.__path__ = [os.path.join(base, sub)]
        pkg.__package__ = name
        sys.modules[name] = pkg
    # morefusion.geometry: only `nn` is touched (functions/loss/average_distance.py:77); its
    # __init__ imports open3d & co.  Stand-in = the body of the reference's CPU path
    # (geometry/knn/nn.py:11-14: sklearn KD-tree, first neighbour).
    import sklearn.neighbors
    geo = types.ModuleType("morefusion.geometry")
    geo.nn = lambda ref, query: sklearn.neighbors.KDTree(np.asarray(ref)).query(
        np.asarray(query), return_distance=False)[:, 0]
    sys.modules["morefusion.geometry"] = geo
    sys.modules["morefusion"].geometry = geo
    _INSTALLED = True


def ref_module(dotted):
    """Import a reference leaf module, e.g. 'functions.geometry.quaternion_matrix'."""
    install()
    return importlib.import_module("morefusion." + dotted)


def load_functions_namespace():
    """Populate morefusion.functions with the leaf callables the ICC link uses
    (what the reference's functions/__init__.py:3-15 re-exports)."""
    install()
    fm = sys.modules["morefusion.functions"]
    g = "functions.geometry."
    fm.transformation_matrix = ref_module(g + "transformation_matrix").transformation_matrix
    fm.transform_points = ref_module(g + "transform_points").transform_points
    tdf = ref_module(g + "truncated_distance_function")
    fm.pseudo_occupancy_voxelization = tdf.pseudo_occupancy_voxelization
    fm.truncated_distance_function = tdf.truncated_distance_function
    sys.modules["morefusion.functions.geometry"].transform_points = fm.transform_points
    return fm
