"""ctypes binding of libdpn_b200.so (include/dpn_b200.h).  The library is built in-tree by
`__graft_entry__.build()`; there is NO fallback: if it is missing or a call fails, we raise."""
import ctypes as C
import os

import torch

from .config import PhysicsConsts

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DPN_LIB_OVERRIDE") or os.path.join(_HERE, "_lib", "libdpn_b200.so")   # override: kernel experiments only

MODE_FP32, MODE_BF16, MODE_BF16X3, MODE_F16X3, MODE_F16X3A = 0, 1, 2, 3, 4
MODES = {"fp32": MODE_FP32, "bf16": MODE_BF16, "bf16x3": MODE_BF16X3, "f16x3": MODE_F16X3, "f16x3a": MODE_F16X3A}
WEIGHT_FIELDS = ("W1", "b1", "W2", "b2", "e", "Wd", "bd", "Wa", "ba", "Wb", "bb", "wo", "bo")


class DpnShape(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("mode", C.c_int32),
                ("n_norm", C.c_int64), ("seed_scale", C.c_float), ("chunk", C.c_int32)]


class DpnConsts(C.Structure):
    _fields_ = [("dx", C.c_double), ("dy", C.c_double), ("lat_size", C.c_int32), ("lon_size", C.c_int32),
                ("t_span", C.c_double), ("with_clip", C.c_int32), ("pad_", C.c_int32),
                ("mean", C.c_double * 6), ("std", C.c_double * 6), ("lo", C.c_double * 6), ("hi", C.c_double * 6),
                ("factor", C.c_double * 6),
                ("c_p", C.c_double), ("L", C.c_double), ("R_v", C.c_double), ("R_d", C.c_double),
                ("band_coord", C.c_float * 32), ("band_data", C.c_float * 16)]


class DpnPoints(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("x", "y", "t", "f", "coord_pe", "coord_data", "ref")]


class DpnWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in WEIGHT_FIELDS]


class DpnGrads(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in WEIGHT_FIELDS]


class DpnPdeOut(C.Structure):
    _fields_ = [("loss_terms", C.c_void_p), ("vals", C.c_void_p), ("jac", C.c_void_p)]


class DpnMargin(C.Structure):
    _fields_ = [("target", C.c_void_p), ("beta", C.c_double), ("factor", C.c_double), ("loss", C.c_void_p), ("o", C.c_void_p)]


class DpnQueryGen(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("lat_size", C.c_int32), ("lon_size", C.c_int32), ("t_steps", C.c_int32),
                ("on_grid", C.c_int32), ("dx", C.c_double), ("dy", C.c_double), ("dt", C.c_double),
                ("seed", C.c_uint64), ("offset", C.c_uint64)]


class DpnSampler(C.Structure):
    _fields_ = [("B", C.c_int32), ("N", C.c_int32), ("Tt", C.c_int32), ("Hc", C.c_int32), ("Wc", C.c_int32),
                ("pad_", C.c_int32), ("dx", C.c_double), ("dy", C.c_double), ("cells_per_coarse", C.c_double),
                ("t_step", C.c_double), ("begin_lat", C.c_double), ("deg_per_cell", C.c_double), ("omega", C.c_double)]


class DpnLattice(C.Structure):
    _fields_ = [("nx", C.c_int32), ("ny", C.c_int32), ("nt", C.c_int32), ("pad_", C.c_int32),
                ("x0", C.c_double), ("y0", C.c_double), ("t0", C.c_double),
                ("sx", C.c_double), ("sy", C.c_double), ("st", C.c_double)]


_lib = None

ABI_VERSION = 2
EXPORTS = ("dpn_abi_version", "dpn_last_error", "dpn_workspace_bytes", "dpn_pde_fwd_bwd", "dpn_pde_margin_fwd_bwd",
           "dpn_decoder_fwd", "dpn_decoder_bwd", "dpn_sample_field", "dpn_generate_queries", "dpn_last_launch_count",
           "dpn_lattice_workspace_bytes", "dpn_decoder_lattice")


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("%s not built - run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU/PyTorch fallback for this path)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        L.dpn_abi_version.restype = C.c_int
        L.dpn_last_error.restype = C.c_size_t
        L.dpn_last_error.argtypes = [C.c_char_p, C.c_size_t]
        L.dpn_workspace_bytes.argtypes = [C.POINTER(DpnShape), C.POINTER(C.c_size_t)]
        L.dpn_pde_fwd_bwd.argtypes = [C.POINTER(DpnShape), C.POINTER(DpnConsts), C.POINTER(DpnPoints),
                                      C.POINTER(DpnWeights), C.POINTER(DpnPdeOut), C.POINTER(DpnGrads),
                                      C.c_void_p, C.c_size_t, C.c_void_p]
        L.dpn_pde_margin_fwd_bwd.argtypes = [C.POINTER(DpnShape), C.POINTER(DpnConsts), C.POINTER(DpnPoints),
                                             C.POINTER(DpnWeights), C.POINTER(DpnMargin), C.POINTER(DpnPdeOut), C.POINTER(DpnGrads),
                                             C.c_void_p, C.c_size_t, C.c_void_p]
        L.dpn_generate_queries.argtypes = [C.POINTER(DpnQueryGen), C.POINTER(DpnSampler)] + [C.c_void_p] * 7
        L.dpn_decoder_fwd.argtypes = [C.POINTER(DpnShape), C.POINTER(DpnConsts), C.POINTER(DpnPoints),
                                      C.POINTER(DpnWeights), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        L.dpn_decoder_bwd.argtypes = [C.POINTER(DpnShape), C.POINTER(DpnConsts), C.POINTER(DpnPoints),
                                      C.POINTER(DpnWeights), C.c_void_p, C.POINTER(DpnGrads),
                                      C.c_void_p, C.c_size_t, C.c_void_p]
        L.dpn_sample_field.argtypes = [C.POINTER(DpnSampler)] + [C.c_void_p] * 7
        L.dpn_last_launch_count.restype = C.c_int
        L.dpn_lattice_workspace_bytes.argtypes = [C.POINTER(DpnShape), C.POINTER(C.c_size_t)]
        L.dpn_decoder_lattice.argtypes = [C.POINTER(DpnShape), C.POINTER(DpnConsts), C.POINTER(DpnLattice), C.POINTER(DpnSampler),
                                          C.c_void_p, C.POINTER(DpnWeights), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
        if L.dpn_abi_version() != ABI_VERSION:
            raise RuntimeError("libdpn_b200.so ABI version mismatch")
        _lib = L
    return _lib


def check(rc, what):
    if rc != 0:
        buf = C.create_string_buffer(1024)
        lib().dpn_last_error(buf, 1024)
        raise RuntimeError("%s failed (code %d): %s" % (what, rc, buf.value.decode(errors="replace")))


def make_consts(pc: PhysicsConsts) -> DpnConsts:
    c = DpnConsts()
    c.dx, c.dy, c.lat_size, c.lon_size = pc.dx, pc.dy, pc.lat_size, pc.lon_size
    c.t_span, c.with_clip = float(pc.pred_t_span), int(bool(pc.with_clip))
    for name in ("mean", "std", "lo", "hi", "factor"):
        arr = getattr(c, name)
        for i, v in enumerate(getattr(pc, name)):
            arr[i] = float(v)
    c.c_p, c.L, c.R_v, c.R_d = pc.c_p, pc.L, pc.R_v, pc.R_d
    for i, v in enumerate(_bands(32)):
        c.band_coord[i] = v
    for i, v in enumerate(_bands(16)):
        c.band_data[i] = v
    return c


_band_cache = {}


def _bands(n):
    # the same torch expression the reference evaluates at module init (position_encoding.py:27) -> bit-identical
    if n not in _band_cache:
        from .pe import freq_bands
        _band_cache[n] = [float(v) for v in freq_bands(n).to(torch.float32)]
    return _band_cache[n]


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


_ws = {}


def workspace(shape: DpnShape, device, nbytes=None):
    """Caller-owned scratch for one library call on the CURRENT stream (torch caching-allocator memory): dpn_workspace_bytes(shape)
    bytes, or `nbytes` when given (dpn_lattice_workspace_bytes for dpn_decoder_lattice).

    * Outside CUDA-graph capture: one buffer per (device, stream), grown on demand.  A dropped buffer returns to the caching
      allocator, which only re-issues it in stream order, so kernels already enqueued on that stream stay safe; two streams
      never share a buffer.
    * During capture: a fresh allocation from the capturing graph's private pool.  The graph bakes the pointer into its
      kernel nodes, so the memory must belong to the graph - it then lives exactly as long as the graph does, whatever later
      eager calls (a larger shape, another mode) do to the cached buffers."""
    need = C.c_size_t(0)
    if nbytes is None:
        check(lib().dpn_workspace_bytes(C.byref(shape), C.byref(need)), "dpn_workspace_bytes")
    else:
        need.value = int(nbytes)
    nbytes = max(need.value, 256)
    if device.type == "cuda" and torch.cuda.is_current_stream_capturing():
        return torch.empty(nbytes, dtype=torch.uint8, device=device), need.value
    key = (device.type, device.index, torch.cuda.current_stream(device).cuda_stream if device.type == "cuda" else 0)
    buf = _ws.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(nbytes, dtype=torch.uint8, device=device)
        _ws[key] = buf
    return buf, need.value


def release_workspaces():
    """Drops every cached scratch buffer (they are re-created on demand)."""
    _ws.clear()
