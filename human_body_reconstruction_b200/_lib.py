"""Build + ctypes binding of libhbr_b200.so (the C ABI declared in include/hbr.h).

There is no CPU fallback anywhere in this package: if the shared library is missing or the tensors are
not on a CUDA device, the ops raise.  The library is built in-tree (csrc/ -> libhbr_b200.so next to this
file) with nvcc for sm_100a only.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys
import threading

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(_HERE, "libhbr_b200.so")
INCLUDE = os.path.join(ROOT, "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "--fmad=true",        # contraction stays on for throughput code; parity-critical ops use __f*_rn intrinsics
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "-Xptxas", "-v",
]
# NOTE: never -use_fast_math: division, expf, sinf must stay IEEE/accurate for parity (SURVEY Q3).

HBR_MAX_LEVELS = 32
HBR_MAX_PEERS, HBR_PEER_MAX_CTAS, HBR_PEER_HANDLE_BYTES = 8, 128, 64
HBR_PEER_FLAG_BYTES = HBR_PEER_MAX_CTAS * HBR_MAX_PEERS * 4
HBR_F32, HBR_F16, HBR_U8, HBR_BF16 = 0, 1, 2, 3
HBR_ABI_VERSION = 2
HBR_DFEAT_LEVEL_MAJOR = -1


class HashGeom(C.Structure):
    _fields_ = [("mu", C.c_float * 3), ("sigma", C.c_float), ("L", C.c_int32), ("F", C.c_int32), ("E", C.c_int32),
                ("T", C.c_uint32), ("scale", C.c_float * HBR_MAX_LEVELS)]


class MlpDims(C.Structure):
    _fields_ = [("in0", C.c_int32), ("d_view", C.c_int32)]


DEBUG_SO_PATH = os.path.join(_HERE, "libhbr_b200_debug.so")


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _deps():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if os.path.isfile(os.path.join(CSRC, f))] + \
        [os.path.join(INCLUDE, "hbr.h")]


def _stale() -> bool:
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -shared -> libhbr_b200.so (cross-compiles without a GPU)."""
    if not force and not _stale():
        return SO_PATH
    bdir = os.path.join(_HERE, "build")
    os.makedirs(bdir, exist_ok=True)
    # several ranks of one node may find the library stale at the same moment (torchrun): one of them builds, the others
    # wait on the lock and then find it fresh; the finished library is moved into place atomically, so a process that
    # loads it concurrently sees either the old or the new file, never a half-written one
    import fcntl
    with open(os.path.join(bdir, ".lock"), "w") as lockf:
        fcntl.flock(lockf, fcntl.LOCK_EX)
        try:
            if not force and not _stale():
                return SO_PATH
            return _build_locked(bdir, force, verbose)
        finally:
            fcntl.flock(lockf, fcntl.LOCK_UN)


def _build_locked(bdir: str, force: bool, verbose: bool) -> str:
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs, procs = [], []
    for src in sources():
        obj = os.path.join(bdir, os.path.basename(src)[:-3] + ".o")
        objs.append(obj)
        if (not force) and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(d) for d in _deps()):
            continue
        cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("HBR_EXTRA_NVCC", "").split(), "-I", INCLUDE, "-c", src, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"== {os.path.basename(src)}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{out}")
    with open(os.path.join(bdir, "ptxas.log"), "a" if not force else "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    tmp_so = os.path.join(bdir, f"libhbr_b200.{os.getpid()}.so.tmp")
    cmd = [nvcc, "-shared", "-o", tmp_so, *objs, "-lcudart"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp_so, SO_PATH)
    return SO_PATH


def build_debug(force: bool = False) -> str:
    """csrc/debug/*.cu (+ abi.cu for the error plumbing) -> libhbr_b200_debug.so: probes and self tests only."""
    dbg = os.path.join(CSRC, "debug")
    srcs = sorted(os.path.join(dbg, f) for f in os.listdir(dbg) if f.endswith(".cu")) + [os.path.join(CSRC, "abi.cu")]
    deps = _deps() + [os.path.join(dbg, f) for f in os.listdir(dbg)]
    if not force and os.path.exists(DEBUG_SO_PATH) and os.path.getmtime(DEBUG_SO_PATH) > max(os.path.getmtime(d) for d in deps):
        return DEBUG_SO_PATH
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, *[f for f in NVCC_FLAGS if f not in ("-Xptxas", "-v")], "-I", INCLUDE, "-shared", "-o", DEBUG_SO_PATH, *srcs,
           "-lcudart"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed for the debug library:\n{r.stdout}")
    return DEBUG_SO_PATH


_lib = None
_debug_lib = None
_lock = threading.Lock()

_i64, _i32, _f32, _vp = C.c_int64, C.c_int, C.c_float, C.c_void_p
_geom_p, _dims_p = C.POINTER(HashGeom), C.POINTER(MlpDims)

# name -> argtypes; every symbol include/hbr.h declares (tests/test_abi.py cross-checks the header)
SIGNATURES = {
    "hbr_abi_version": ([], C.c_int),
    "hbr_last_error": ([], C.c_char_p),
    "hbr_mlp_param_count": ([_dims_p], _i64),
    "hbr_mlp_act_floats": ([], _i64),
    "hbr_hash_encode_fwd": ([_vp, _i32, _i64, _vp, _geom_p, _vp, _i64, _vp], C.c_int),
    "hbr_hash_encode_bwd": ([_vp, _i32, _i64, _vp, _i64, _geom_p, _vp, _i32, _i32, _vp], C.c_int),
    "hbr_hash_encode_dx": ([_vp, _i32, _i64, _vp, _geom_p, _vp, _i64, _vp, _vp], C.c_int),
    "hbr_hash_indices": ([_vp, _i32, _i64, _geom_p, _vp, _vp, _vp], C.c_int),
    "hbr_dir_encode": ([_vp, _i32, _i64, _i32, _i32, _vp, _vp], C.c_int),
    "hbr_mlp_fwd_f32": ([_vp, _i64, _vp, _i64, _i64, _vp, _dims_p, _vp, _vp, _vp], C.c_int),
    "hbr_mlp_bwd_f32": ([_vp, _i64, _vp, _i64, _i64, _vp, _dims_p, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp], C.c_int),
    "hbr_mlp_tc_scratch_bytes": ([_dims_p], _i64),
    "hbr_mlp_fwd_tc": ([_vp, _i32, _i64, _vp, _i64, _i64, _vp, _dims_p, _i32, _vp, _vp, _i32, _vp, _vp, _vp], C.c_int),
    "hbr_mlp_bwd_tc": ([_vp, _i32, _i64, _vp, _i64, _i64, _vp, _dims_p, _i32, _vp, _vp, _vp, _i64, _vp, _vp, _f32, _vp, _i32, _i32,
                        _vp, _vp, _vp], C.c_int),
    "hbr_occupancy_update": ([_vp, _i64, _vp, _i64, _vp, _i32, C.POINTER(C.c_float), _f32, _vp, _vp], C.c_int),
    "hbr_compact_samples": ([_vp, _vp, _vp, _i64, _i64, _i64, _vp, _i32, C.POINTER(C.c_float), _f32, _vp, _vp, _vp, _vp, _vp],
                            C.c_int),
    "hbr_hash_encode_fwd_pts": ([_vp, _i64, _vp, _vp, _geom_p, _vp, _i64, _i32, _vp], C.c_int),
    "hbr_hash_encode_bwd_pts": ([_vp, _i64, _vp, _vp, _i64, _geom_p, _vp, _i32, _i32, _vp], C.c_int),
    "hbr_mlp_tc_prepare": ([_vp, _dims_p, _i32, _vp, _vp], C.c_int),
    "hbr_mlp_tc_reduce_grads": ([_dims_p, _i64, _vp, _vp, _vp], C.c_int),
    "hbr_strat_depths": ([_vp, _vp, _f32, _f32, _i64, _vp, _vp], C.c_int),
    "hbr_mse_pair_fwd": ([_vp, _vp, _vp, _i64, _f32, _vp, _vp], C.c_int),
    "hbr_mse_pair_bwd": ([_vp, _vp, _vp, _i64, _f32, _vp, _vp, _vp, _vp], C.c_int),
    "hbr_hash_encode_fwd_rays": ([_vp, _vp, _vp, _i64, _i64, _i64, _vp, _geom_p, _vp, _i64, _i32, _vp], C.c_int),
    "hbr_field_bwd_rays_tc": ([_vp, _vp, _vp, _vp, _i64, _i64, _i64, _geom_p, _vp, _vp, _dims_p, _i32, _vp, _vp, _vp, _vp, _vp, _f32,
                               _vp, _i32, _i32, _vp], C.c_int),
    "hbr_field_fwd_rays_tc": ([_vp, _vp, _vp, _i64, _i64, _i64, _vp, _geom_p, _vp, _vp, _dims_p, _i32, _vp, _vp, _vp, _i32, _vp],
                              C.c_int),
    "hbr_hash_encode_bwd_rays": ([_vp, _vp, _vp, _i64, _i64, _i64, _vp, _i64, _geom_p, _vp, _i32, _i32, _vp], C.c_int),
    "hbr_field_fwd_tc": ([_vp, _i64, _vp, _geom_p, _vp, _i64, _vp, _dims_p, _i32, _vp, _vp, _vp, _vp], C.c_int),
    "hbr_field_bwd_tc": ([_vp, _i64, _geom_p, _vp, _i64, _vp, _dims_p, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp],
                         C.c_int),
    "hbr_adam_step": ([_vp, _vp, _vp, _vp, _i64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, _i32, _i64,
                       C.c_double, _vp, _vp], C.c_int),
    "hbr_adam_tick": ([_vp, _vp, _vp], C.c_int),
    "hbr_adam_step_dev": ([_vp, _vp, _vp, _vp, _i64, _vp, C.c_double, C.c_double, C.c_double, C.c_double, _i32, _vp, C.c_double,
                           _vp, _vp, _vp], C.c_int),
    "hbr_ray_gen": ([_vp, _i64, _i32, _i32, _f32, _f32, _f32, _f32, _vp, _i64, _i64, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp],
                    C.c_int),
    "hbr_ray_bbox": ([_vp, _i64, _i32, _i32, _f32, _f32, _f32, _f32, _f32, _f32, _vp, _vp], C.c_int),
    "hbr_peer_alloc": ([C.POINTER(_vp), _i64], C.c_int),
    "hbr_peer_free": ([_vp], C.c_int),
    "hbr_peer_export": ([_vp, C.POINTER(C.c_ubyte)], C.c_int),
    "hbr_peer_import": ([C.POINTER(C.c_ubyte), C.POINTER(_vp)], C.c_int),
    "hbr_peer_release": ([_vp], C.c_int),
    "hbr_allreduce_peer": ([C.POINTER(_vp), C.POINTER(_vp), _vp, _i32, _i32, _i64, _f32, _i32, _vp, _vp], C.c_int),
    "hbr_hash_bwd_stream_tiles": ([_i64], _i64),
    "hbr_hash_encode_bwd_stream": ([_vp, _i32, _i64, _vp, _i64, _geom_p, _vp, C.POINTER(C.c_int), _i32, _vp, _vp], C.c_int),
    "hbr_hash_encode_bwd_rays_stream": ([_vp, _vp, _vp, _i64, _i64, _i64, _vp, _i64, _geom_p, _vp, C.POINTER(C.c_int), _i32, _vp,
                                         _vp], C.c_int),
    "hbr_hash_bwd_lm_ctas": ([_i64], _i64),
    "hbr_hash_encode_bwd_lm": ([_vp, _i32, _i64, _vp, _geom_p, _vp, C.POINTER(C.c_int), _i32, _vp, _vp], C.c_int),
    "hbr_hash_encode_bwd_rays_lm": ([_vp, _vp, _vp, _i64, _i64, _i64, _vp, _geom_p, _vp, C.POINTER(C.c_int), _i32, _vp, _vp],
                                    C.c_int),
    "hbr_allreduce_peer_stream": ([C.POINTER(_vp), C.POINTER(_vp), _vp, _i32, _i32, _i32, C.POINTER(_i64), C.POINTER(_i64),
                                   C.POINTER(C.c_uint), C.POINTER(C.c_int), _vp, _f32, _i32, _vp, _vp], C.c_int),
    "hbr_ray_points": ([_vp, _vp, _vp, _i64, _i64, _i64, _vp, _vp], C.c_int),
    "hbr_occupancy_mask": ([_vp, _i64, _vp, _i32, C.POINTER(C.c_float), _f32, _vp, _vp], C.c_int),
    "hbr_composite_fwd": ([_vp, _i64, _vp, _i64, _vp, _i64, _vp, _f32, _vp, _vp, _i64, _i64, _vp, _vp, _f32, _vp], C.c_int),
    "hbr_composite_bwd": ([_vp, _i64, _vp, _i64, _vp, _i64, _vp, _f32, _vp, _vp, _i64, _i64, _vp, _vp, _i64, _vp, _i64, _f32, _vp],
                          C.c_int),
    "hbr_composite_maps_fwd": ([_vp, _i64, _vp, _i64, _vp, _i64, _vp, _f32, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _f32, _vp],
                               C.c_int),
    "hbr_composite_maps_bwd": ([_vp, _i64, _vp, _i64, _vp, _i64, _vp, _f32, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _i64, _vp,
                                _i64, _f32, _vp], C.c_int),
    "hbr_hier_sample": ([_vp, _vp, _vp, _vp, _i64, _i64, _i32, _vp, _vp], C.c_int),
    "hbr_composite_sdf_fwd": ([_vp, _i64, _vp, _i64, _i32, _vp, _i64, _i64, _vp, _vp, _vp], C.c_int),
    "hbr_composite_sdf_bwd": ([_vp, _i64, _vp, _i64, _i32, _vp, _i64, _i64, _vp, _vp, _vp, _i64, _vp, _i64, _vp, _vp], C.c_int),
    "hbr_sdf_stencil_points": ([_vp, _i64, _f32, C.POINTER(C.c_float), C.POINTER(C.c_float), _vp, _vp], C.c_int),
    "hbr_sdf_eikonal_fwd": ([_vp, _i64, _f32, _vp, _vp, _vp], C.c_int),
    "hbr_sdf_eikonal_bwd": ([_vp, _i64, _f32, _vp, _vp, _vp], C.c_int),
    "hbr_grid_points": ([C.POINTER(C.c_double), C.POINTER(C.c_double), _i32, _i64, _i64, _vp, _vp], C.c_int),
    "hbr_grid_density": ([C.POINTER(C.c_double), C.POINTER(C.c_double), _i32, _i64, _i64, _vp, _geom_p, _vp, _dims_p,
                          _vp, _vp, _vp, _vp, _i64, _i32, _vp], C.c_int),
    "hbr_mlp_density_tf32x3": ([_vp, _i64, _vp, _dims_p, _vp, _vp], C.c_int),
    "hbr_mc_count": ([_vp, _i32, _i32, _i32, _f32, _i32, _i32, _vp, _vp], C.c_int),
    "hbr_mc_emit": ([_vp, _i32, _i32, _i32, _f32, _i32, _i32, _vp, _vp, _i64, _vp, _i64, _vp, _vp], C.c_int),
    "hbr_grid_interp": ([_vp, _i32, _i32, _i32, _i32, _vp, _i64, _vp, _vp], C.c_int),
}

# probes / self tests: a separate library (csrc/debug/ -> libhbr_b200_debug.so), not part of the product ABI
DEBUG_SIGNATURES = {
    "hbr_debug_umma": ([_i32, _i32, _vp, _vp, _vp, _i32, _i32, _vp], C.c_int),
    "hbr_debug_umma_bench": ([_i32, _i32, _i32, _i32, _i32, _vp, _vp], C.c_int),
    "hbr_debug_umma_chain_bench": ([_i32, _i32, _i32, _vp, _vp], C.c_int),
    "hbr_debug_mlp_trace": ([_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp], C.c_int),
    "hbr_debug_mlp_trace_bwd": ([_vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp], C.c_int),
}


# kernels launched by one call of each entry point (for bench.py's gpu_launches claim)
KERNELS_PER_CALL = {
    "hbr_hash_encode_fwd": 1, "hbr_hash_encode_bwd": 1, "hbr_hash_encode_dx": 1, "hbr_hash_encode_fwd_rays": 1, "hbr_hash_encode_bwd_rays": 1, "hbr_hash_indices": 1, "hbr_dir_encode": 1,
    "hbr_mlp_fwd_f32": 1, "hbr_mlp_bwd_f32": 2, "hbr_mlp_fwd_tc": 2, "hbr_mlp_bwd_tc": 3, "hbr_field_fwd_tc": 2, "hbr_field_bwd_tc": 3, "hbr_field_bwd_rays_tc": 3, "hbr_field_fwd_rays_tc": 1, "hbr_adam_step": 1, "hbr_adam_tick": 1, "hbr_adam_step_dev": 1, "hbr_allreduce_peer": 1, "hbr_allreduce_peer_stream": 1, "hbr_hash_encode_bwd_stream": 1, "hbr_hash_encode_bwd_rays_stream": 1, "hbr_hash_encode_bwd_lm": 1, "hbr_hash_encode_bwd_rays_lm": 1, "hbr_ray_gen": 1, "hbr_ray_bbox": 1, "hbr_ray_points": 1, "hbr_occupancy_mask": 1, "hbr_occupancy_update": 2, "hbr_compact_samples": 1, "hbr_hash_encode_fwd_pts": 1, "hbr_hash_encode_bwd_pts": 1,
    "hbr_composite_fwd": 1, "hbr_composite_bwd": 1, "hbr_composite_maps_fwd": 1, "hbr_composite_maps_bwd": 1, "hbr_strat_depths": 1, "hbr_mse_pair_fwd": 1, "hbr_mse_pair_bwd": 1, "hbr_mlp_tc_prepare": 1, "hbr_mlp_tc_reduce_grads": 1, "hbr_hier_sample": 1, "hbr_grid_points": 1,
    "hbr_composite_sdf_fwd": 1, "hbr_composite_sdf_bwd": 1, "hbr_sdf_stencil_points": 1, "hbr_sdf_eikonal_fwd": 1, "hbr_sdf_eikonal_bwd": 1,
    "hbr_grid_density": 3, "hbr_mlp_density_tf32x3": 1, "hbr_mc_count": 1, "hbr_mc_emit": 2, "hbr_grid_interp": 1,
}


class _Stats:
    """Launch accounting + optional per-call CUDA-event timing (bench.py turns it on inside its timed region)."""

    def __init__(self):
        self.launches = 0
        self.calls = {}
        self.timing = False
        self.events = []            # (name, start_event, end_event)
        self.graph_events = []      # the same for calls made while a CUDA graph was being captured: EXTERNAL events, i.e. event
                                    # record nodes of that graph -- every replay re-records them (read after a synchronize)

    def reset(self):
        self.launches = 0
        self.calls = {}
        self.events = []
        self.graph_events = []

    def graph_times(self):
        """name -> [ms of each call of the last replay]; call after the replay has been synchronised."""
        out = {}
        for name, a, b in self.graph_events:
            out.setdefault(name, []).append(a.elapsed_time(b))
        return out

    def summary(self):
        """name -> (count, mean_ms); call after torch.cuda.synchronize()."""
        acc = {}
        for name, a, b in self.events:
            c, s = acc.get(name, (0, 0.0))
            acc[name] = (c + 1, s + a.elapsed_time(b))
        return {k: (c, s / c) for k, (c, s) in acc.items()}


STATS = _Stats()


class _Counted:
    __slots__ = ("fn", "name", "k")

    def __init__(self, fn, name):
        self.fn, self.name, self.k = fn, name, KERNELS_PER_CALL.get(name, 0)

    def __call__(self, *a):
        st = STATS
        st.launches += self.k
        st.calls[self.name] = st.calls.get(self.name, 0) + 1
        if st.timing and self.k:
            ext = torch.cuda.is_current_stream_capturing()
            e0 = torch.cuda.Event(enable_timing=True, external=ext)
            e1 = torch.cuda.Event(enable_timing=True, external=ext)
            s = torch.cuda.current_stream()
            e0.record(s)
            rc = self.fn(*a)
            e1.record(s)
            (st.graph_events if ext else st.events).append((self.name, e0, e1))
            return rc
        return self.fn(*a)


class _Lib:
    pass


def lib():
    """The loaded shared library.  Builds it if the sources are newer; raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if _stale():
                if os.environ.get("HBR_NO_BUILD") == "1":
                    raise RuntimeError("libhbr_b200.so is missing/stale and HBR_NO_BUILD=1")
                build()
            l = C.CDLL(SO_PATH)
            wrapped = _Lib()
            for name, (args, res) in SIGNATURES.items():
                fn = getattr(l, name)            # AttributeError if the .so does not export a declared symbol
                fn.argtypes = args
                fn.restype = res
                setattr(wrapped, name, _Counted(fn, name) if name in KERNELS_PER_CALL else fn)
            if l.hbr_abi_version() != HBR_ABI_VERSION:
                raise RuntimeError("libhbr_b200.so ABI version mismatch")
            wrapped.cdll = l
            _lib = wrapped
    return _lib


def debug_lib():
    """The probe / self-test library (tests and scripts/dbg_*.py only)."""
    global _debug_lib
    with _lock:
        if _debug_lib is None:
            l = C.CDLL(build_debug())
            wrapped = _Lib()
            for name, (args, res) in DEBUG_SIGNATURES.items():
                fn = getattr(l, name)
                fn.argtypes = args
                fn.restype = res
                setattr(wrapped, name, fn)
            l.hbr_last_error.restype = C.c_char_p
            wrapped.cdll = l
            _debug_lib = wrapped
    return _debug_lib


def check(rc: int):
    if rc != 0:
        raise RuntimeError(f"libhbr_b200: {lib().hbr_last_error().decode()} (status {rc})")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream():
    """cudaStream_t of torch's current stream on the current device (raw getter: ~1 us instead of ~15 us for
    torch.cuda.current_stream(), which every C-ABI call would otherwise pay)."""
    return C.c_void_p(torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice()))


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("human_body_reconstruction_b200 ops run on CUDA tensors only (no CPU fallback); "
                               f"got a tensor on {t.device}")
