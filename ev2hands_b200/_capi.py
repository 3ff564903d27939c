"""ctypes binding of libev2h.so (include/ev2h.h) for torch CUDA tensors.

PyTorch is plumbing here: it owns device memory and streams; every compute step
is a call into the C ABI with raw pointers.  There is no fallback: if the
library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import os

import torch

_PKG = os.path.dirname(os.path.abspath(__file__))
# EV2H_LIB selects another build of the same ABI (kernel experiments); default is the in-tree library
LIB_PATH = os.environ.get("EV2H_LIB") or os.path.join(_PKG, "libev2h.so")
_lib = None

c_int, c_i64, c_f, c_d, c_vp = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_double, ctypes.c_void_p

# name -> argtypes (restype is always int except where noted); mirrors include/ev2h.h
_SIGNATURES = {
    "ev2h_fps_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "ev2h_fps_variant_f32": [c_int, c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "ev2h_ball_query_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_int,
                            ctypes.POINTER(c_f), ctypes.POINTER(ctypes.c_int32), c_vp, c_vp],
    "ev2h_square_distance_f32": [c_vp, c_vp, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_index_rows_f32": [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_group_gather_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_vp, c_vp, c_int, c_int,
                              c_int, c_int, c_int, c_int, c_vp, c_int, c_vp],
    "ev2h_group_gather_bwd_f32": [c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_wgrad_splits": [c_i64, c_int, c_int],
    "ev2h_wgrad_f32": [c_vp, c_int, c_vp, c_int, c_i64, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "ev2h_point_records_f32": [c_vp, c_i64, c_i64, c_i64, c_int, c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_vp, c_vp],
    "ev2h_transpose_f32": [c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_int, c_vp, c_i64, c_i64, c_i64, c_vp],
    "ev2h_fold_conv_bn_f32": [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_d, c_int, c_int, c_vp, c_vp, c_vp],
    "ev2h_linear_relu_f32": [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_vp],
    "ev2h_tc_pack_weights": [c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_tc_pack_weights_kc": [c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_sa_msg_fused_kc": [c_int, ctypes.POINTER(ctypes.c_int32)],
    "ev2h_linear_relu_tc": [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_tc_set_debug": [c_int],
    "ev2h_linear_tc": [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_fused_set_debug_buffer": [c_vp],
    "ev2h_linear_f32": [c_vp, c_i64, c_int, c_int, c_vp, c_vp, c_int, c_vp, c_int, c_int, c_vp],
    "ev2h_sa_msg_fused_tc": [c_vp, c_int, c_int, c_vp, c_int, c_int, c_int, c_int,
                             c_vp, c_int, c_vp, c_int, c_vp,
                             c_vp, c_int, c_int, c_vp, c_int, c_int,
                             c_int, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(c_vp), ctypes.POINTER(c_vp),
                             c_vp, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_ball_query_cnt_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_int, ctypes.POINTER(c_f),
                                ctypes.POINTER(ctypes.c_int32), c_vp, c_vp, c_vp],
    "ev2h_first_occurrence_u8": [c_vp, c_int, c_int, c_vp, c_vp],
    "ev2h_ball_query_uniq_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_int, ctypes.POINTER(c_f),
                                 ctypes.POINTER(ctypes.c_int32), c_vp, c_vp, c_vp, c_vp, c_vp],
    "ev2h_ball_query_compact_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_int, ctypes.POINTER(c_f),
                                    ctypes.POINTER(ctypes.c_int32), c_vp, c_vp, c_vp, ctypes.POINTER(c_vp), ctypes.POINTER(c_vp),
                                    c_vp, c_vp],
    "ev2h_group_compact_i32": [c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, ctypes.POINTER(ctypes.c_int32),
                               ctypes.POINTER(c_vp), ctypes.POINTER(c_vp), c_vp, c_vp],
    "ev2h_sa_msg_fused_compact_tc": [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_int,
                                     c_vp, c_int, c_vp, c_int, c_vp,
                                     c_vp, c_int, c_int, c_vp, c_int, c_int,
                                     c_int, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(c_vp), ctypes.POINTER(c_vp),
                                     c_vp, c_int, c_int, c_int, c_vp, c_vp],
    "ev2h_three_nn_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_i64, c_i64, c_i64, c_int, c_int, c_int, c_vp, c_vp, c_vp],
    "ev2h_three_interp_f32": [c_vp, c_int, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_int, c_int, c_vp],
    "ev2h_window_aggregate_f64": [c_vp, c_i64, c_vp, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp],
    "ev2h_window_sample_f32": [c_vp, c_int, c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp],
    "ev2h_fps_range_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp],
    "ev2h_ball_query_compact_range_f32": [c_vp, c_i64, c_i64, c_i64, c_vp, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                          ctypes.POINTER(c_f), ctypes.POINTER(ctypes.c_int32), c_vp, c_vp, c_vp,
                                          ctypes.POINTER(c_vp), ctypes.POINTER(c_vp), c_vp, c_vp],
    "ev2h_conv1d_tc": [c_vp, c_i64, c_int, c_int, c_int, c_int, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp,
                       c_vp],
    "ev2h_class_attention_f32": [c_vp, c_int, c_vp, c_int, c_vp, c_int, c_int, c_int, c_int, c_int, c_f, c_vp, c_vp, c_vp],
    "ev2h_group_max_f32": [c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp, c_vp],
    "ev2h_group_max_bwd_f32": [c_vp, c_vp, c_int, c_int, c_int, c_int, c_vp, c_vp],
}


def declared_symbols():
    """Every function include/ev2h.h declares (parsed from the header itself)."""
    import re
    with open(os.path.join(_PKG, "..", "include", "ev2h.h")) as f:
        return sorted(set(re.findall(r"EV2H_API\s+[\w\s\*]+?\b(ev2h_\w+)\s*\(", f.read())))


def lib() -> ctypes.CDLL:
    """Load libev2h.so; raise loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libev2h.so is not built (%s). Run `python -m ev2hands_b200.build` "
                "(needs nvcc); there is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        L.ev2h_version.restype = c_int
        L.ev2h_last_error.restype = ctypes.c_char_p
        L.ev2h_tc_packed_bytes.argtypes = [c_int, c_int, c_int]
        L.ev2h_tc_packed_bytes.restype = c_i64
        L.ev2h_tc_packed_bytes_kc.argtypes = [c_int, c_int, c_int, c_int, c_int]
        L.ev2h_tc_packed_bytes_kc.restype = c_i64
        for name, args in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = c_int
        _lib = L
    return _lib


class LaunchLog:
    """Counts kernel launches (every compute entry point of the ABI enqueues exactly one
    kernel) and, when ``timing`` is on, brackets each with CUDA events on its stream so
    bench.py can report per-kernel device time from inside the timed region."""

    def __init__(self):
        self.count = 0
        self.timing = False
        self.events = []          # (name, start_event, end_event)

    def reset(self, timing: bool = False):
        self.count = 0
        self.timing = timing
        self.events = []

    def totals_ms(self):
        """{name: (launches, total_ms)}; call after a device synchronize."""
        out = {}
        for name, a, b in self.events:
            n, t = out.get(name, (0, 0.0))
            out[name] = (n + 1, t + a.elapsed_time(b))
        return out


LOG = LaunchLog()


class _timed:
    def __init__(self, name, launches=1):
        self.name = name
        self.launches = launches

    def __enter__(self):
        LOG.count += self.launches
        if LOG.timing:
            self.a = torch.cuda.Event(enable_timing=True)
            self.b = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if LOG.timing:
            self.b.record()
            LOG.events.append((self.name, self.a, self.b))
        return False


def _check(status: int, what: str):
    if status != 0:
        msg = lib().ev2h_last_error().decode("utf-8", "replace")
        raise RuntimeError("%s failed (status %d): %s" % (what, status, msg))


def _stream(t: torch.Tensor):
    return c_vp(torch.cuda.current_stream(t.device).cuda_stream)


def _p(t):
    return c_vp(0) if t is None else c_vp(t.data_ptr())


def _need_cuda_f32(t: torch.Tensor, name: str):
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: ev2hands_b200 has no CPU path" % name)
    if t.dtype != torch.float32:
        raise RuntimeError("%s must be float32, got %s" % (name, t.dtype))


def cf_strides(xyz_cf: torch.Tensor):
    """Element strides (batch, channel, point) of a channel-first [B,3,N] tensor."""
    return xyz_cf.stride(0), xyz_cf.stride(1), xyz_cf.stride(2)


def rows_strides(xyz_rows: torch.Tensor):
    """Same triple for a point-major [B,N,3] tensor."""
    return xyz_rows.stride(0), xyz_rows.stride(2), xyz_rows.stride(1)


def fps(xyz: torch.Tensor, strides, start: torch.Tensor, B: int, N: int, S: int,
        want_rows=True, want_cf=True, variant: int = 0):
    """-> (idx int32 [B,S], centres_rows [B,S,3] | None, centres_cf [B,3,S] | None); variant: kernel for N > 4096
    (ev2h_fps_variant_f32: 1 exhaustive, 2 cluster, 3 pruned; 0 = the library's choice)"""
    _need_cuda_f32(xyz, "xyz")
    dev = xyz.device
    if tuple(start.shape) != (B,):
        raise RuntimeError("FPS start indices must have shape [%d], got %s" % (B, tuple(start.shape)))
    if not start.is_cuda:
        # host-drawn start indices (the reference's torch.randint on the CPU generator).  Inside a CUDA-graph capture
        # an upload from a temporary pinned block would be baked into the graph and replayed from recycled memory
        # (and the draw itself frozen), so a captured forward must be given device-resident start tensors.
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("FPS start indices are host tensors (or were drawn on the host) during CUDA-graph capture: "
                               "pass device-resident fps_start / fps_starts tensors and refill them between replays")
        start = start.to(dtype=torch.int64).contiguous()
        if B > 0 and (int(start.min()) < 0 or int(start.max()) >= N):     # the reference would raise an IndexError (:77)
            raise IndexError("FPS start index out of range [0, %d)" % N)
        # upload from pinned memory without blocking, so the host keeps running ahead of the device instead of
        # syncing with it twice per step
        start = start.pin_memory().to(dev, non_blocking=True)
    else:
        start = start.to(device=dev, dtype=torch.int64).contiguous()
    idx = torch.empty((B, S), dtype=torch.int32, device=dev)
    rows = torch.empty((B, S, 3), dtype=torch.float32, device=dev) if want_rows else None
    cf = torch.empty((B, 3, S), dtype=torch.float32, device=dev) if want_cf else None
    with torch.cuda.device(dev):
        with _timed("ev2h_fps_f32"):
            if variant:
                _check(lib().ev2h_fps_variant_f32(int(variant), _p(xyz), strides[0], strides[1], strides[2], _p(start), B, N, S,
                                                  _p(idx), _p(rows), _p(cf), _stream(xyz)), "ev2h_fps_variant_f32")
            else:
                _check(lib().ev2h_fps_f32(_p(xyz), strides[0], strides[1], strides[2], _p(start), B, N, S,
                                          _p(idx), _p(rows), _p(cf), _stream(xyz)), "ev2h_fps_f32")
    return idx, rows, cf


def device_starts(start: torch.Tensor, B: int, N: int, dev) -> torch.Tensor:
    """FPS start indices as an int64 device tensor (range-checked when they come from the host, see fps())"""
    if tuple(start.shape) != (B,):
        raise RuntimeError("FPS start indices must have shape [%d], got %s" % (B, tuple(start.shape)))
    if start.is_cuda:
        return start.to(device=dev, dtype=torch.int64).contiguous()
    if torch.cuda.is_current_stream_capturing():
        raise RuntimeError("FPS start indices are host tensors (or were drawn on the host) during CUDA-graph capture: "
                           "pass device-resident fps_start / fps_starts tensors and refill them between replays")
    start = start.to(dtype=torch.int64).contiguous()
    if B > 0 and (int(start.min()) < 0 or int(start.max()) >= N):
        raise IndexError("FPS start index out of range [0, %d)" % N)
    return start.pin_memory().to(dev, non_blocking=True)


def fps_range(xyz, strides, start_dev, B, N, S, s_begin, s_end, state_best, state_cur, idx, rows, cf):
    """samples [s_begin, s_end) of a farthest point sampling into the preallocated outputs (ev2h_fps_range_f32)"""
    with torch.cuda.device(xyz.device):
        with _timed("ev2h_fps_f32"):
            _check(lib().ev2h_fps_range_f32(_p(xyz), strides[0], strides[1], strides[2], _p(start_dev), B, N, S, s_begin, s_end,
                                            _p(state_best), _p(state_cur), _p(idx), _p(rows), _p(cf), _stream(xyz)), "ev2h_fps_range_f32")


def ball_query_compact_range(xyz, strides, centres_rows, B, N, S, s_begin, s_count, reset_rows, radii, nsamples, out, first_flag,
                             uniq, rowmaps, blockgroups, n_rows):
    """ball query + compacted row lists of the centres [s_begin, s_begin + s_count) into preallocated outputs"""
    ns = len(radii)
    r2 = (c_f * ns)(*[radius_sq_f32(r) for r in radii])
    ks = (ctypes.c_int32 * ns)(*[int(k) for k in nsamples])
    a_rm = (c_vp * ns)(*[t.data_ptr() for t in rowmaps])
    a_bg = (c_vp * ns)(*[t.data_ptr() for t in blockgroups])
    with torch.cuda.device(xyz.device):
        with _timed("ev2h_ball_query_f32"):
            _check(lib().ev2h_ball_query_compact_range_f32(_p(xyz), strides[0], strides[1], strides[2], _p(centres_rows), B, N, S,
                                                           s_begin, s_count, 1 if reset_rows else 0, ns, r2, ks, _p(out), _p(first_flag),
                                                           _p(uniq), a_rm, a_bg, _p(n_rows), _stream(xyz)),
                   "ev2h_ball_query_compact_range_f32")


def radius_sq_f32(radius: float) -> float:
    """float(radius**2) rounded to fp32: what aten compares against (pointnet2_utils.py:102)."""
    return torch.tensor(float(radius) ** 2, dtype=torch.float32).item()


def ball_query(xyz: torch.Tensor, strides, centres_rows: torch.Tensor, N: int, radii, nsamples, with_counts: bool = False):
    """-> idx int32 [B,S,sum(K)]  (with_counts: also cnt int32 [n_scales,B,S], the real neighbours per scale)"""
    _need_cuda_f32(xyz, "xyz")
    _need_cuda_f32(centres_rows, "centres")
    B, S, _ = centres_rows.shape
    ns = len(radii)
    r2 = (c_f * ns)(*[radius_sq_f32(r) for r in radii])
    ks = (ctypes.c_int32 * ns)(*[int(k) for k in nsamples])
    out = torch.empty((B, S, int(sum(nsamples))), dtype=torch.int32, device=xyz.device)
    cnt = torch.empty((ns, B, S), dtype=torch.int32, device=xyz.device) if with_counts else None
    with torch.cuda.device(xyz.device):
        with _timed("ev2h_ball_query_f32"):
            if with_counts:
                _check(lib().ev2h_ball_query_cnt_f32(_p(xyz), strides[0], strides[1], strides[2], _p(centres_rows.contiguous()),
                                                     B, N, S, ns, r2, ks, _p(out), _p(cnt), _stream(xyz)), "ev2h_ball_query_cnt_f32")
            else:
                _check(lib().ev2h_ball_query_f32(_p(xyz), strides[0], strides[1], strides[2], _p(centres_rows.contiguous()),
                                                 B, N, S, ns, r2, ks, _p(out), _stream(xyz)), "ev2h_ball_query_f32")
    return (out, cnt) if with_counts else out


def first_occurrence(pts8: torch.Tensor) -> torch.Tensor:
    """pts8 [B,N,8] -> uint8 [B,N]: 1 where the point's record has not occurred earlier in its window."""
    B, N, _ = pts8.shape
    out = torch.empty((B, N), dtype=torch.uint8, device=pts8.device)
    with torch.cuda.device(pts8.device):
        with _timed("ev2h_first_occurrence_u8"):
            _check(lib().ev2h_first_occurrence_u8(_p(pts8), B, N, _p(out), _stream(pts8)), "ev2h_first_occurrence_u8")
    return out


def ball_query_uniq(xyz: torch.Tensor, strides, centres_rows: torch.Tensor, N: int, radii, nsamples, first_flag: torch.Tensor):
    """-> (idx, uniq_idx, uniq_cnt): the reference's padded list, and the same first-K hits without exact-duplicate points."""
    _need_cuda_f32(xyz, "xyz")
    _need_cuda_f32(centres_rows, "centres")
    B, S, _ = centres_rows.shape
    ns = len(radii)
    r2 = (c_f * ns)(*[radius_sq_f32(r) for r in radii])
    ks = (ctypes.c_int32 * ns)(*[int(k) for k in nsamples])
    out = torch.empty((B, S, int(sum(nsamples))), dtype=torch.int32, device=xyz.device)
    uniq = torch.empty_like(out)
    ucnt = torch.empty((ns, B, S), dtype=torch.int32, device=xyz.device)
    with torch.cuda.device(xyz.device):
        with _timed("ev2h_ball_query_f32"):
            _check(lib().ev2h_ball_query_uniq_f32(_p(xyz), strides[0], strides[1], strides[2], _p(centres_rows.contiguous()),
                                                  B, N, S, ns, r2, ks, _p(out), _p(first_flag), _p(uniq), _p(ucnt), _stream(xyz)),
                   "ev2h_ball_query_uniq_f32")
    return out, uniq, ucnt


def ball_query_compact(xyz: torch.Tensor, strides, centres_rows: torch.Tensor, N: int, radii, nsamples, first_flag=None):
    """Ball query + compacted row lists in one kernel -> (idx, rowmaps, blockgroups, n_rows); first_flag (uint8 [B,N])
    additionally lists exact-duplicate points once."""
    _need_cuda_f32(xyz, "xyz")
    _need_cuda_f32(centres_rows, "centres")
    B, S, _ = centres_rows.shape
    ns = len(radii)
    dev = xyz.device
    r2 = (c_f * ns)(*[radius_sq_f32(r) for r in radii])
    ks = (ctypes.c_int32 * ns)(*[int(k) for k in nsamples])
    out = torch.empty((B, S, int(sum(nsamples))), dtype=torch.int32, device=dev)
    uniq = torch.empty_like(out) if first_flag is not None else None
    rowmaps = [torch.empty((B * S * int(k),), dtype=torch.int32, device=dev) for k in nsamples]
    blockgroups = [torch.empty((B * S * int(k) // 8,), dtype=torch.int32, device=dev) for k in nsamples]
    n_rows = torch.empty((ns,), dtype=torch.int32, device=dev)
    a_rm = (c_vp * ns)(*[t.data_ptr() for t in rowmaps])
    a_bg = (c_vp * ns)(*[t.data_ptr() for t in blockgroups])
    with torch.cuda.device(dev):
        with _timed("ev2h_ball_query_f32"):
            _check(lib().ev2h_ball_query_compact_f32(_p(xyz), strides[0], strides[1], strides[2], _p(centres_rows.contiguous()),
                                                     B, N, S, ns, r2, ks, _p(out), _p(first_flag), _p(uniq), a_rm, a_bg, _p(n_rows),
                                                     _stream(xyz)), "ev2h_ball_query_compact_f32")
    return out, rowmaps, blockgroups, n_rows


def group_compact(idx: torch.Tensor, cnt: torch.Tensor, N: int, nsamples):
    """Compacted row lists of every scale of a layer (ev2h_group_compact_i32):
    -> (rowmaps, blockgroups, n_rows): two lists of int32 device tensors and the int32 [n_scales] row counts."""
    B, S, _ = idx.shape
    ns = len(nsamples)
    dev = idx.device
    rowmaps = [torch.empty((B * S * int(k),), dtype=torch.int32, device=dev) for k in nsamples]
    blockgroups = [torch.empty((B * S * int(k) // 8,), dtype=torch.int32, device=dev) for k in nsamples]
    n_rows = torch.empty((ns,), dtype=torch.int32, device=dev)
    ks = (ctypes.c_int32 * ns)(*[int(k) for k in nsamples])
    a_rm = (c_vp * ns)(*[t.data_ptr() for t in rowmaps])
    a_bg = (c_vp * ns)(*[t.data_ptr() for t in blockgroups])
    with torch.cuda.device(dev):
        with _timed("ev2h_group_compact_i32"):
            _check(lib().ev2h_group_compact_i32(_p(idx), idx.shape[-1], _p(cnt), B, N, S, ns, ks, a_rm, a_bg, _p(n_rows),
                                                _stream(idx)), "ev2h_group_compact_i32")
    return rowmaps, blockgroups, n_rows


def square_distance(src_rows: torch.Tensor, dst_rows: torch.Tensor) -> torch.Tensor:
    _need_cuda_f32(src_rows, "src")
    _need_cuda_f32(dst_rows, "dst")
    src_rows, dst_rows = src_rows.contiguous(), dst_rows.contiguous()
    B, S, _ = src_rows.shape
    N = dst_rows.shape[1]
    out = torch.empty((B, S, N), dtype=torch.float32, device=src_rows.device)
    with torch.cuda.device(src_rows.device):
        with _timed("ev2h_square_distance_f32"):
            _check(lib().ev2h_square_distance_f32(_p(src_rows), _p(dst_rows), B, S, N, _p(out), _stream(out)),
               "ev2h_square_distance_f32")
    return out


def index_rows(table_rows: torch.Tensor, idx: torch.Tensor) -> torch.Tensor:
    _need_cuda_f32(table_rows, "points")
    table_rows = table_rows.contiguous()
    B, N, C = table_rows.shape
    idx32 = idx.to(device=table_rows.device, dtype=torch.int32).contiguous()
    M = idx32[0].numel()
    out = torch.empty(tuple(idx.shape) + (C,), dtype=torch.float32, device=table_rows.device)
    with torch.cuda.device(table_rows.device):
        with _timed("ev2h_index_rows_f32"):
            _check(lib().ev2h_index_rows_f32(_p(table_rows), _p(idx32), B, N, M, C, _p(out), _stream(out)),
               "ev2h_index_rows_f32")
    return out


def group_gather(xyz, strides, feats_rows, D, centres_rows, idx, k_off, B, N, S, K, out, ld_out):
    with torch.cuda.device(xyz.device):
        with _timed("ev2h_group_gather_f32"):
            _check(lib().ev2h_group_gather_f32(_p(xyz), strides[0], strides[1], strides[2], _p(feats_rows), D,
                                           _p(centres_rows), _p(idx), idx.shape[-1], k_off, B, N, S, K,
                                           _p(out), ld_out, _stream(xyz)), "ev2h_group_gather_f32")


def group_gather_bwd(grad_rows, ld_grad, idx, k_off, B, N, S, K, D, grad_feats_rows):
    with torch.cuda.device(grad_rows.device):
        with _timed("ev2h_group_gather_bwd_f32"):
            _check(lib().ev2h_group_gather_bwd_f32(_p(grad_rows), ld_grad, _p(idx), idx.shape[-1], k_off, B, N, S, K, D,
                                               _p(grad_feats_rows), _stream(grad_rows)), "ev2h_group_gather_bwd_f32")


def wgrad(dy: torch.Tensor, x: torch.Tensor, want_bias: bool = False):
    """dW [Cout, Cin] = dy^T x for fp32 rows dy [M, Cout] (contiguous) and x [M, Cin] (unit column stride);
    want_bias: -> (dW, db) with db [Cout] = dy.sum(0) from the same pass"""
    M, cout = dy.shape
    cin = x.shape[1]
    splits = lib().ev2h_wgrad_splits(M, cout, cin)
    work = torch.empty((splits * cout * (cin + 1),), dtype=torch.float32, device=dy.device)
    dw = torch.empty((cout, cin), dtype=torch.float32, device=dy.device)
    db = torch.empty((cout,), dtype=torch.float32, device=dy.device) if want_bias else None
    with torch.cuda.device(dy.device):
        with _timed("ev2h_wgrad_f32", launches=3 if want_bias else 2):
            _check(lib().ev2h_wgrad_f32(_p(dy), dy.stride(0), _p(x), x.stride(0), M, cout, cin, _p(work), _p(dw), _p(db), _stream(dy)),
                   "ev2h_wgrad_f32")
    return (dw, db) if want_bias else dw


def point_records(points, xyz, strides) -> torch.Tensor:
    """[B, N, 8] records [features | xyz | 0] from channel-first points [B, D, N] (or None) and xyz [B, 3, N]"""
    B, _, N = xyz.shape
    D = 0 if points is None else points.shape[1]
    out = torch.empty((B, N, 8), dtype=torch.float32, device=xyz.device)
    ps = (0, 0, 0) if points is None else (points.stride(0), points.stride(1), points.stride(2))
    with torch.cuda.device(xyz.device):
        with _timed("ev2h_point_records_f32"):
            _check(lib().ev2h_point_records_f32(_p(points), ps[0], ps[1], ps[2], D, _p(xyz), strides[0], strides[1], strides[2],
                                                B, N, _p(out), _stream(xyz)), "ev2h_point_records_f32")
    return out


def transpose(src, src_strides, B, R, C, dst, dst_stride_b, dst_ld, dst_col_off=0):
    """dst[b, c, dst_col_off + r] = src[b, r, c] with explicit element strides."""
    with torch.cuda.device(src.device):
        with _timed("ev2h_transpose_f32"):
            _check(lib().ev2h_transpose_f32(_p(src), src_strides[0], src_strides[1], src_strides[2], B, R, C,
                                        _p(dst), dst_stride_b, dst_ld, dst_col_off, _stream(src)), "ev2h_transpose_f32")


def fold_conv_bn(conv_w, conv_b, gamma, beta, mean, var, eps: float):
    """-> (wt [Cin_pad, Cout_pad], bias [Cout_pad]) fp32 on the weights' device."""
    Cout, Cin = conv_w.shape[0], conv_w.shape[1]
    cin_pad, cout_pad = (Cin + 15) // 16 * 16, (Cout + 127) // 128 * 128
    dev = conv_w.device
    wt = torch.empty((cin_pad, cout_pad), dtype=torch.float32, device=dev)
    bias = torch.empty((cout_pad,), dtype=torch.float32, device=dev)
    args = [t.detach().contiguous().float() for t in (conv_w.reshape(Cout, Cin), conv_b, gamma, beta, mean, var)]
    with torch.cuda.device(dev):
        with _timed("ev2h_fold_conv_bn_f32"):
            _check(lib().ev2h_fold_conv_bn_f32(*[_p(a) for a in args], float(eps), Cin, Cout, _p(wt), _p(bias),
                                           _stream(wt)), "ev2h_fold_conv_bn_f32")
    return wt, bias


def linear_relu(x, M, ld_x, Cin, wt, bias, Cout, pool_rows, y, ld_y, y_col_off=0):
    with torch.cuda.device(x.device):
        with _timed("ev2h_linear_relu_f32"):
            _check(lib().ev2h_linear_relu_f32(_p(x), M, ld_x, Cin, _p(wt), _p(bias), Cout, pool_rows, _p(y), ld_y,
                                          y_col_off, _stream(x)), "ev2h_linear_relu_f32")


TC_BF16, TC_TF32X3, TC_TF32_BF16C, TC_F16X3 = 0, 1, 2, 3


def tc_supported(Cout: int, pool_rows: int) -> bool:
    """Shapes the tensor-core layer kernel covers (others go through the fp32 FFMA kernel)."""
    return (Cout <= 256 or Cout % 256 == 0) and (pool_rows in (0, 32, 64) or pool_rows % 128 == 0)


def tc_pack(wt: torch.Tensor, Cin: int, Cout: int, mode: int, kc: int = 32, row_align: int = 16) -> torch.Tensor:
    """folded wt [Cin_pad, Cout_pad] -> packed shared-memory images (uint8 buffer) for `mode`,
    `kc` input channels per image, image rows padded to a multiple of `row_align`.
    TC_F16X3: a weight outside the fp16 range (or NaN) raises the device's range flag - a BatchNorm with a tiny
    running variance and a large gamma folds into such weights (checked on the device, no synchronisation)."""
    n = lib().ev2h_tc_packed_bytes_kc(Cin, Cout, mode, kc, row_align)
    if n <= 0:
        raise RuntimeError("ev2h_tc_packed_bytes_kc(%d, %d, %d, %d, %d) failed" % (Cin, Cout, mode, kc, row_align))
    packed = torch.empty((n,), dtype=torch.uint8, device=wt.device)
    with torch.cuda.device(wt.device):
        with _timed("ev2h_tc_pack_weights"):
            _check(lib().ev2h_tc_pack_weights_kc(_p(wt), wt.shape[1], Cin, Cout, mode, kc, row_align, _p(packed), _stream(wt)),
                   "ev2h_tc_pack_weights_kc")
        if mode == TC_F16X3:
            range_flag(wt.device).bitwise_or_((~(wt.abs().amax() < 65520.0)).to(torch.int32))
    return packed


def fused_kc(mode: int, couts) -> int:
    """K-chunk length the fused kernel wants for tensor-core layers of widths `couts` (-1: unsupported)."""
    arr = (ctypes.c_int32 * 2)(*couts)
    return lib().ev2h_sa_msg_fused_kc(mode, arr)


def _f16_flag(t, mode):
    """the device's range flag for the fp16-split mode (the kernels track their inputs' range there), else NULL"""
    return range_flag(t.device) if mode == TC_F16X3 else None


def linear_relu_tc(x, M, ld_x, Cin, packed, bias, Cout, pool_rows, y, ld_y, y_col_off, mode):
    flag = _f16_flag(x, mode)
    with torch.cuda.device(x.device):
        with _timed("ev2h_linear_relu_tc"):
            _check(lib().ev2h_linear_relu_tc(_p(x), M, ld_x, Cin, _p(packed), _p(bias), Cout, pool_rows, _p(y), ld_y,
                                             y_col_off, mode, _p(flag), _stream(x)), "ev2h_linear_relu_tc")


def linear_tc_no_relu(x, M, ld_x, Cin, packed, bias, Cout, y, ld_y, y_col_off, mode):
    flag = _f16_flag(x, mode)
    with torch.cuda.device(x.device):
        with _timed("ev2h_linear_tc"):
            _check(lib().ev2h_linear_tc(_p(x), M, ld_x, Cin, _p(packed), _p(bias), Cout, _p(y), ld_y, y_col_off, mode,
                                        _p(flag), _stream(x)), "ev2h_linear_tc")


def linear_no_relu(x, M, ld_x, Cin, wt, bias, Cout, y, ld_y, y_col_off=0):
    with torch.cuda.device(x.device):
        with _timed("ev2h_linear_f32"):
            _check(lib().ev2h_linear_f32(_p(x), M, ld_x, Cin, _p(wt), _p(bias), Cout, _p(y), ld_y, y_col_off, _stream(x)),
                   "ev2h_linear_f32")


def conv1d_tc(x_rows, M, ld_x, Cin, taps, rows_per_seq, packed, bias, Cout, relu, post_scale, post_shift, y, ld_y, y_col_off, mode):
    """Conv1d (kernel size taps, zero padding taps // 2) over point-major rows [+ ReLU] [+ per-channel affine]."""
    flag = _f16_flag(x_rows, mode)
    with torch.cuda.device(x_rows.device):
        with _timed("ev2h_conv1d_tc"):
            _check(lib().ev2h_conv1d_tc(_p(x_rows), M, ld_x, Cin, taps, rows_per_seq, _p(packed), _p(bias), Cout, 1 if relu else 0,
                                        _p(post_scale), _p(post_shift), _p(y), ld_y, y_col_off, mode, _p(flag), _stream(x_rows)),
                   "ev2h_conv1d_tc")


def class_attention(key_rows, ld_k, query_rows, ld_q, value_rows, ld_v, B, N, C, D, scale):
    """AttentionBlock on rows -> context [B, C, N] channel-first."""
    dev = value_rows.device
    partial = torch.empty((B, 8, C, D), dtype=torch.float32, device=dev)
    out = torch.empty((B, C, N), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        with _timed("ev2h_class_attention_f32", launches=2):
            _check(lib().ev2h_class_attention_f32(_p(key_rows), ld_k, _p(query_rows), ld_q, _p(value_rows), ld_v, B, N, C, D, float(scale),
                                                  _p(partial), _p(out), _stream(value_rows)), "ev2h_class_attention_f32")
    return out


def fused_supported(K: int, widths, first_in: int, per_point: bool, mode: int = TC_TF32X3) -> bool:
    """Shapes ev2h_sa_msg_fused_tc covers (see include/ev2h.h): three layers, layer 1 either per point
    (wide inputs, width a multiple of 32) or in the loader warps (<= 8 input channels)."""
    if K not in (32, 64, 128) or len(widths) != 3 or any(w > 256 for w in widths):
        return False
    if per_point and widths[0] % 32 != 0:
        return False
    if not per_point and (first_in > 8 or widths[0] > 128):      # layer 1 in the loader warps: weights are kernel parameters
        return False
    return fused_kc(mode, widths[1:]) > 0


_range_flags = {}


def range_flag(device) -> torch.Tensor:
    """int32 [1] on `device`: bit 0 is set when an operand of the fp16 split (TC_F16X3) left the fp16 range or was NaN -
    by the fused kernel and the per-layer kernels (ev2h_linear_tc, ev2h_linear_relu_tc, ev2h_conv1d_tc) for their
    activation inputs, and by tc_pack for the weights it packs."""
    device = torch.device(device)
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    t = _range_flags.get(device)
    if t is None:
        t = _range_flags[device] = torch.zeros((1,), dtype=torch.int32, device=device)
    return t


def check_numeric_range(device="cuda", reset: bool = True) -> bool:
    """True if no fp16-split (TC_F16X3) kernel or weight pack on `device` saw an operand outside the fp16 range since the last reset
    (synchronises; call it at a checkpoint, not per step).  Raise-free so callers decide what to do."""
    t = range_flag(device)
    ok = int(t.item()) == 0
    if reset:
        t.zero_()
    return ok


def sa_msg_fused(idx, k_off, centres_rows, B, N, S, K, pts8, D, first_wt_host, first_bias_host, P, ld_p, p_col, C, ld_c, c_col,
                 c1, couts, packed, biases, out_rows, ld_out, out_col, mode, compact=None):
    """compact = (rowmap, blockgroup, n_rows_scalar_view) runs the kernel over the compacted row list.
    first_wt_host / first_bias_host: contiguous float32 HOST tensors (gather mode), the folded layer-1 map."""
    a_cout = (ctypes.c_int32 * 2)(*couts)
    a_w = (c_vp * 2)(*[t.data_ptr() for t in packed])
    a_b = (c_vp * 2)(*[t.data_ptr() for t in biases])
    if first_wt_host is not None and (first_wt_host.is_cuda or first_bias_host.is_cuda or not first_wt_host.is_contiguous()):
        raise RuntimeError("sa_msg_fused: the layer-1 weights of the gather mode are passed as contiguous HOST tensors")
    flag = range_flag(out_rows.device) if mode == TC_F16X3 else None
    with torch.cuda.device(out_rows.device):
        if compact is not None:
            rm, bg, nr = compact
            with _timed("ev2h_sa_msg_fused_tc"):
                _check(lib().ev2h_sa_msg_fused_compact_tc(_p(rm), _p(bg), _p(nr), _p(centres_rows), B, N, S, K,
                                                          _p(pts8), D, _p(first_wt_host), 0 if first_wt_host is None else first_wt_host.shape[1],
                                                          _p(first_bias_host), _p(P), ld_p, p_col, _p(C), ld_c, c_col,
                                                          c1, a_cout, a_w, a_b, _p(out_rows), ld_out, out_col, mode, _p(flag),
                                                          _stream(out_rows)), "ev2h_sa_msg_fused_compact_tc")
            return
        with _timed("ev2h_sa_msg_fused_tc"):
            _check(lib().ev2h_sa_msg_fused_tc(_p(idx), idx.shape[-1], k_off, _p(centres_rows), B, N, S, K,
                                              _p(pts8), D, _p(first_wt_host), 0 if first_wt_host is None else first_wt_host.shape[1],
                                              _p(first_bias_host), _p(P), ld_p, p_col, _p(C), ld_c, c_col,
                                              c1, a_cout, a_w, a_b, _p(out_rows), ld_out, out_col, mode, _p(flag),
                                              _stream(out_rows)), "ev2h_sa_msg_fused_tc")


def group_max(x: torch.Tensor, want_arg: bool = True):
    """x [B,C,K,S] contiguous -> (out [B,C,S], arg int32 [B,C,S] | None)"""
    _need_cuda_f32(x, "x")
    x = x.contiguous()
    B, C, K, S = x.shape
    out = torch.empty((B, C, S), dtype=torch.float32, device=x.device)
    arg = torch.empty((B, C, S), dtype=torch.int32, device=x.device) if want_arg else None
    with torch.cuda.device(x.device):
        with _timed("ev2h_group_max_f32"):
            _check(lib().ev2h_group_max_f32(_p(x), B, C, K, S, _p(out), _p(arg), _stream(x)), "ev2h_group_max_f32")
    return out, arg


def group_max_bwd(grad_out: torch.Tensor, arg: torch.Tensor, K: int) -> torch.Tensor:
    grad_out = grad_out.contiguous()
    B, C, S = grad_out.shape
    gx = torch.empty((B, C, K, S), dtype=torch.float32, device=grad_out.device)
    with torch.cuda.device(grad_out.device):
        with _timed("ev2h_group_max_bwd_f32"):
            _check(lib().ev2h_group_max_bwd_f32(_p(grad_out), _p(arg), B, C, K, S, _p(gx), _stream(gx)),
               "ev2h_group_max_bwd_f32")
    return gx


def three_nn(xyz1: torch.Tensor, xyz2: torch.Tensor):
    """xyz1 [B,3,N] queries, xyz2 [B,3,S] sources (channel-first, any strides) ->
    (idx int32 [B,N,3], weight fp32 [B,N,3]): three nearest sources and inverse-distance weights."""
    B, _, N = xyz1.shape
    S = xyz2.shape[2]
    idx = torch.empty((B, N, 3), dtype=torch.int32, device=xyz1.device)
    w = torch.empty((B, N, 3), dtype=torch.float32, device=xyz1.device)
    with torch.cuda.device(xyz1.device):
        with _timed("ev2h_three_nn_f32"):
            _check(lib().ev2h_three_nn_f32(_p(xyz1), xyz1.stride(0), xyz1.stride(1), xyz1.stride(2),
                                           _p(xyz2), xyz2.stride(0), xyz2.stride(1), xyz2.stride(2),
                                           B, N, S, _p(idx), _p(w), _stream(xyz1)), "ev2h_three_nn_f32")
    return idx, w


def three_interp(feats_rows, ld_f, idx, weight, B, N, S, D, out_rows, ld_out, col):
    with torch.cuda.device(out_rows.device):
        with _timed("ev2h_three_interp_f32"):
            _check(lib().ev2h_three_interp_f32(_p(feats_rows), ld_f, _p(idx), _p(weight), B, N, S, D, _p(out_rows), ld_out, col,
                                               _stream(out_rows)), "ev2h_three_interp_f32")


WINDOW_STREAM, WINDOW_ERPC = 0, 1


def window_aggregate(events: torch.Tensor, win_start: torch.Tensor, win_count: torch.Tensor, max_count: int,
                     width: int, height: int, mode: int):
    """events float64 [n, >=4] (CUDA), win_start int64 [B], win_count int32 [B] (CUDA)
    -> (records fp32 [B, max_count, 5], n_pixels int32 [B], n_bad int32 [B])."""
    if not events.is_cuda or events.dtype != torch.float64 or events.dim() != 2 or events.stride(1) != 1:
        raise RuntimeError("events must be a CUDA float64 [n, >=4] tensor with contiguous rows (there is no CPU path)")
    dev = events.device
    B = win_start.shape[0]
    win_start = win_start.to(device=dev, dtype=torch.int64).contiguous()
    win_count = win_count.to(device=dev, dtype=torch.int32).contiguous()
    records = torch.empty((B, max_count, 5), dtype=torch.float32, device=dev)
    n_pixels = torch.empty((B,), dtype=torch.int32, device=dev)
    n_bad = torch.empty((B,), dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        with _timed("ev2h_window_aggregate_f64"):
            _check(lib().ev2h_window_aggregate_f64(_p(events), events.stride(0), _p(win_start), _p(win_count), B, max_count,
                                                   width, height, mode, _p(records), _p(n_pixels), _p(n_bad), _stream(events)),
                   "ev2h_window_aggregate_f64")
    return records, n_pixels, n_bad


def window_sample(records: torch.Tensor, n_pixels: torch.Tensor, sample_idx: torch.Tensor, width: int, height: int,
                  n_bad: torch.Tensor):
    """records [B, max_count, 5], sample_idx int64 [B, N] -> windows fp32 [B, 5, N] (channel-first, the encoder's input)."""
    B, max_count, _ = records.shape
    N = sample_idx.shape[1]
    out = torch.empty((B, 5, N), dtype=torch.float32, device=records.device)
    sample_idx = sample_idx.to(device=records.device, dtype=torch.int64).contiguous()
    with torch.cuda.device(records.device):
        with _timed("ev2h_window_sample_f32"):
            _check(lib().ev2h_window_sample_f32(_p(records), max_count, _p(n_pixels), _p(sample_idx), B, N, width, height,
                                                _p(out), _p(n_bad), _stream(records)), "ev2h_window_sample_f32")
    return out
