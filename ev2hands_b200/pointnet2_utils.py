"""Drop-in replacement for the reference's ``src/Ev2Hands/model/pointnet2_utils.py``.

Same public names, constructor arguments, forward signatures, parameter and
buffer names (so reference checkpoints load with ``strict=True``), but every
step of the set-abstraction hot path runs in the hand-written sm_100a kernels of
``libev2h.so`` (C ABI in ``include/ev2h.h``):

    farthest_point_sample  -> ev2h_fps_f32             (reference :63-84)
    query_ball_point       -> ev2h_ball_query_f32      (reference :87-107)
    square_distance        -> ev2h_square_distance_f32 (reference :19-40)
    index_points           -> ev2h_index_rows_f32      (reference :43-60)
    grouping               -> ev2h_group_gather_f32    (reference :244-248)
    conv1x1+BN+ReLU, max   -> ev2h_linear_relu_f32 ... (reference :253-257)

There is no CPU path: tensors must live on a CUDA device and a missing library
raises.  ``PointNetFeaturePropagation`` (the decoder, outside the hot path) is
kept in plain PyTorch so that ``TEHNet.py:6`` can import all three names.

Eval mode runs the fused inference path (BatchNorm folded into the weights).
Training mode, or eval mode with autograd active, keeps convolution, BatchNorm
(batch statistics) and ReLU in PyTorch and uses the CUDA kernels for FPS, ball
query, grouping (with scatter-add backward) and max-pool (with arg-max backward).
"""
from __future__ import annotations

import os
import threading
import weakref

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _capi

_WORKSPACE_BYTES = int(os.environ.get("EV2H_WORKSPACE_MB", "4096")) << 20

# Arithmetic of the shared MLP in the inference path:
#   "fp32"   CUDA-core FFMA, exact fp32 (parity anchor)
#   "tf32x3" tensor cores, error-compensated 3xTF32: fp32-level accuracy (bar 1e-5)
#   "bf16"   tensor cores, bf16 operands / fp32 accumulate (bar 1e-2)
_MLP_PRECISIONS = ("fp32", "tf32x3", "bf16")
_mlp_precision = os.environ.get("EV2H_MLP", "tf32x3")


# The fused grouping + MLP + max-pool kernel (sa_fused_tc.cu) is used for every scale it
# covers when a tensor-core precision is selected; EV2H_FUSED=0 forces the layer-by-layer path.
_FUSED_ENABLED = os.environ.get("EV2H_FUSED", "1") != "0"
# fp32-level precision ("tf32x3") on the tensor cores, three split products per multiply:
#   EV2H_SPLIT=f16  (default) fp16 hi/lo pairs, three kind::f16 products - 3 tensor time units and 4 operand bytes per
#                   element; activations must stay below 65520 (ev2hands_b200.check_numeric_range() reports overflows)
#   EV2H_SPLIT=tf32 tf32 hi*hi + two bf16 correction products - 4 units, 8 bytes, fp32 exponent range (round 1's default)
#   EV2H_TF32X3_PURE=1  three tf32 products - 6 units
_TF32X3_PURE = os.environ.get("EV2H_TF32X3_PURE", "0") == "1"
_SPLIT = os.environ.get("EV2H_SPLIT", "f16")
# Run the fused kernel over compacted rows (padded duplicate neighbours skipped; bit-identical results).
_COMPACT = os.environ.get("EV2H_COMPACT", "1") != "0"
# ... and over exact-duplicate points only once (event windows are sampled with replacement).
_DEDUP = os.environ.get("EV2H_DEDUP", "1") != "0"
# The per-layer tensor-core kernel (sa3, the decoder, sa2's per-point first layer) uses the same split products as the
# fused kernel for "tf32x3"; EV2H_LINEAR_MIXED=0 keeps three tf32 products there.
_LINEAR_MIXED = os.environ.get("EV2H_LINEAR_MIXED", "1") != "0"
# The fused launches of a layer's radius scales are independent (same inputs, different output columns): issued on
# separate streams the tail of one persistent launch (pipeline drain, last partial wave) could overlap the start of the
# next.  Measured on B200 (B = 64, graph replay): 1.664 ms with, 1.638 ms without - no gain, so it is off by default.
_SCALE_STREAMS = os.environ.get("EV2H_SCALE_STREAMS", "0") == "1"
_scale_streams = {}


def _scale_stream(device, i):
    key = (device, threading.get_ident(), i)
    with _CACHE_LOCK:
        st = _scale_streams.get(key)
        if st is None:
            st = _scale_streams[key] = torch.cuda.Stream(device=device)
    return st


# Front-end pipelining: farthest point sampling is S strictly sequential iterations on B CTAs, and the ball query of a
# centre needs none of the later centres.  The sampling is cut into EV2H_FPS_SPLITS ranges (resumable kernel) and the
# ball query of each range runs on a second stream beside the sampling of the next; the point records and duplicate
# flags, which need no centre at all, run beside the first range.  0 / 1 = one sampling launch, then the ball query.
# Bit-identical (tests), but SLOWER on B200 at B = 64: 1.705 ms per step with 4 ranges, 1.693 with 2, 1.788 with 8,
# against 1.633 without - the ball query's CTAs share SMs with the sampling's, whose dependent iterations are the critical
# path, and slow them by more than the overlap hides.  Off by default.
_FPS_SPLITS = int(os.environ.get("EV2H_FPS_SPLITS", "0"))

# Evaluate layer 1 per point (instead of per gathered row) also for narrow inputs; experiment switch.
_PER_POINT_ALWAYS = os.environ.get("EV2H_PER_POINT", "0") == "1"


def set_fused(enabled: bool) -> None:
    global _FUSED_ENABLED
    _FUSED_ENABLED = bool(enabled)


def set_mlp_precision(name: str) -> None:
    global _mlp_precision
    if name not in _MLP_PRECISIONS:
        raise ValueError("mlp precision must be one of %s" % (_MLP_PRECISIONS,))
    _mlp_precision = name


def get_mlp_precision() -> str:
    return _mlp_precision


def _pad4(c: int) -> int:
    return (c + 3) // 4 * 4


# --------------------------------------------------------------------------------------
# free functions (same signatures as the reference; tensors are [B, N, C] point-major)
# --------------------------------------------------------------------------------------
def square_distance(src, dst):
    """[B,N,3],[B,M,3] -> [B,N,M]; bit-identical to the reference's expanded form (3 coordinates only)."""
    if src.dim() != 3 or dst.dim() != 3 or src.shape[-1] != 3 or dst.shape[-1] != 3 or src.shape[0] != dst.shape[0]:
        raise RuntimeError("square_distance expects [B,N,3] and [B,M,3], got %s and %s" % (tuple(src.shape), tuple(dst.shape)))
    return _capi.square_distance(src, dst)


def index_points(points, idx):
    """points [B,N,C], idx [B,...] -> [B,...,C]."""
    if points.dim() != 3 or idx.dim() < 2 or idx.shape[0] != points.shape[0]:
        raise RuntimeError("index_points expects points [B,N,C] and idx [B,...], got %s and %s" % (tuple(points.shape), tuple(idx.shape)))
    return _capi.index_rows(points, idx)


def farthest_point_sample(xyz, npoint, start=None):
    """xyz [B,N,3] -> int64 [B,npoint].  ``start`` overrides the random first index,
    which is otherwise drawn exactly like the reference does (CPU generator)."""
    B, N, _ = xyz.shape
    if start is None:
        start = torch.randint(0, N, (B,), dtype=torch.long)
    idx, _, _ = _capi.fps(xyz, _capi.rows_strides(xyz), start, B, N, npoint, want_rows=False, want_cf=False)
    return idx.long()


def query_ball_point(radius, nsample, xyz, new_xyz):
    """xyz [B,N,3], new_xyz [B,S,3] -> int64 [B,S,nsample]."""
    N = xyz.shape[1]
    return _capi.ball_query(xyz, _capi.rows_strides(xyz), new_xyz, N, [radius], [nsample]).long()


def sample_and_group(npoint, radius, nsample, xyz, points, returnfps=False):
    """Reference :110-138 - channels are [rel_xyz, points]."""
    B, N, C = xyz.shape
    fps_idx = farthest_point_sample(xyz, npoint)
    new_xyz = index_points(xyz, fps_idx)
    idx = query_ball_point(radius, nsample, xyz, new_xyz)
    grouped_xyz = index_points(xyz, idx)
    rel = grouped_xyz - new_xyz.view(B, npoint, 1, C)
    new_points = torch.cat([rel, index_points(points, idx)], dim=-1) if points is not None else rel
    if returnfps:
        return new_xyz, new_points, grouped_xyz, fps_idx
    return new_xyz, new_points


def sample_and_group_all(xyz, points):
    """Reference :141-158 - one group of all points, channels [xyz, points]."""
    B, N, C = xyz.shape
    new_xyz = torch.zeros(B, 1, C, device=xyz.device)
    g = xyz.view(B, 1, N, C)
    if points is not None:
        g = torch.cat([g, points.view(B, 1, N, -1)], dim=-1)
    return new_xyz, g


# --------------------------------------------------------------------------------------
# autograd pieces for the training path
# --------------------------------------------------------------------------------------
class _GroupGather(torch.autograd.Function):
    """rows(b,s,j) = [feats[b, idx] | xyz[idx] - centre]; gradient flows to feats only
    (xyz never requires grad in the model, SURVEY.md 3.3)."""

    @staticmethod
    def forward(ctx, feats_rows, xyz, strides, N, centres_rows, idx, k_off, K):
        B, S, _ = centres_rows.shape
        D = 0 if feats_rows is None else feats_rows.shape[2]
        ld = _pad4(D + 3)                    # 16-byte rows: the tensor-core layer kernels read them in place
        out = (torch.empty if ld == D + 3 else torch.zeros)((B, S, K, ld), dtype=torch.float32, device=centres_rows.device)
        _capi.group_gather(xyz, strides, feats_rows, D, centres_rows, idx, k_off, B, N, S, K, out, ld)
        ctx.save_for_backward(idx)
        ctx.meta = (k_off, B, N, S, K, D)
        return out if ld == D + 3 else out[..., :D + 3]

    @staticmethod
    def backward(ctx, grad):
        (idx,) = ctx.saved_tensors
        k_off, B, N, S, K, D = ctx.meta
        g_feats = None
        if D > 0 and ctx.needs_input_grad[0]:
            grad = grad.contiguous()
            g_feats = torch.zeros((B, N, D), dtype=torch.float32, device=grad.device)
            _capi.group_gather_bwd(grad, D + 3, idx, k_off, B, N, S, K, D, g_feats)
        return g_feats, None, None, None, None, None, None, None


class _GroupMax(torch.autograd.Function):
    """max over dim 2 of [B,C,K,S]; the whole gradient goes to the first arg-max."""

    @staticmethod
    def forward(ctx, x):
        out, arg = _capi.group_max(x, want_arg=True)
        ctx.save_for_backward(arg)
        ctx.K = x.shape[2]
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (arg,) = ctx.saved_tensors
        return _capi.group_max_bwd(grad_out, arg, ctx.K)


# --------------------------------------------------------------------------------------
# training-mode shared MLP on point rows
# --------------------------------------------------------------------------------------
# bn(conv(x)) in training mode needs statistics over every position of the batch between two layers, so the layers
# cannot be fused like in eval mode; but a 1x1 convolution over [B, C, K, S] is a GEMM over the B*S*K rows and
# BatchNorm2d's statistics are per-channel means over those rows.  Keeping the grouped tensor as rows [M, C] - the
# layout the gather kernel writes - turns conv / dgrad / wgrad into three plain GEMMs (cuBLAS) and drops the
# [B,S,K,C] -> [B,C,K,S] copy of every scale; cuDNN's fp32 1x1 convolutions (wgrad above all) were 60 % of the step
# (tools/train_profile.py).  EV2H_TRAIN_ROWS=0 restores the channel-first conv2d path.
_TRAIN_ROWS = os.environ.get("EV2H_TRAIN_ROWS", "1") != "0"


def _bn_rows(x2d, bn):
    """nn.BatchNorm{1,2}d.forward on rows [M, C] (positions x channels): same statistics, running-stat update and
    momentum rule as torch.nn.modules.batchnorm._BatchNorm.forward over [B, C, ...]"""
    eaf = 0.0 if bn.momentum is None else bn.momentum
    if bn.training and bn.track_running_stats and bn.num_batches_tracked is not None:
        bn.num_batches_tracked.add_(1)
        eaf = 1.0 / float(bn.num_batches_tracked) if bn.momentum is None else bn.momentum
    use_batch = bn.training or (bn.running_mean is None and bn.running_var is None)
    return F.batch_norm(x2d, bn.running_mean if (not bn.training or bn.track_running_stats) else None,
                        bn.running_var if (not bn.training or bn.track_running_stats) else None,
                        bn.weight, bn.bias, use_batch, eaf, bn.eps)


# Forward and input-gradient GEMMs of those layers on the tcgen05 layer kernel (ev2h_linear_tc) with fp32-level split
# arithmetic - the forward in the inference path's mode, the input gradient with the tf32 / bf16 split, whose operands
# keep fp32's exponent range (gradients span many orders of magnitude; fp16 parts would flush the small ones).  The
# weight gradient dW = dY^T X contracts over the M rows and stays a cuBLAS GEMM.  EV2H_TRAIN_TC: 0 = F.linear
# everywhere, dgrad (default) = input gradients on the tensor cores, 1 = forward too.  The forward is the sensitive one: its
# 2e-6 moves the weight gradients in front of a batch-statistics BatchNorm - differences of large sums - to within 3e-3
# of the reference's autograd instead of 3e-6 (measured; the input-gradient GEMM alone changes nothing at that level),
# far closer than the tf32 convolutions PyTorch runs by default but not the fp32 parity this repo promises.
_TRAIN_WGRAD = os.environ.get("EV2H_TRAIN_WGRAD", "1") != "0"        # weight gradients: ev2h_wgrad_f32 instead of cuBLAS
_TRAIN_FFMA = os.environ.get("EV2H_TRAIN_FFMA", "1") != "0"          # forward GEMMs with >= 96 outputs: ev2h_linear_f32 (exact fp32)
_TRAIN_TC = {"1": "all", "all": "all", "dgrad": "dgrad"}.get(os.environ.get("EV2H_TRAIN_TC", "dgrad"), "")   # "", "dgrad" (default), "all"


def _rows_ok(t):
    """[M, C] fp32 rows the layer kernel can read in place: unit column stride, 16-byte aligned rows"""
    return (t.dim() == 2 and t.is_cuda and t.dtype == torch.float32 and t.stride(1) == 1 and t.stride(0) % 4 == 0
            and t.stride(0) >= t.shape[1] and t.data_ptr() % 16 == 0)


def _pack_dense(w_t, mode):
    """dense [Cin, Cout] matrix (y = x @ w_t) -> (packed tensor-core image, Cin, Cout)"""
    cin, cout = w_t.shape
    wt = torch.zeros(((cin + 15) // 16 * 16, (cout + 127) // 128 * 128), dtype=torch.float32, device=w_t.device)
    wt[:cin, :cout] = w_t
    return _capi.tc_pack(wt, cin, cout, mode)


class _LinearRowsTC(torch.autograd.Function):
    """y = x W^T + b over rows [M, Cin] -> [M, Cout] (a 1x1 convolution over the grouped tensor)"""

    @staticmethod
    def forward(ctx, x, weight, bias, forward_on_tensor_cores):
        M, cin = x.shape
        cout = weight.shape[0]
        if forward_on_tensor_cores:
            mode = _layer_mode(_capi.TC_TF32X3)
            packed = _pack_dense(weight.detach().t(), mode)
            b = torch.zeros(((cout + 127) // 128 * 128,), dtype=torch.float32, device=x.device)
            if bias is not None:
                b[:cout] = bias.detach()
            y = torch.empty((M, cout), dtype=torch.float32, device=x.device)
            _capi.linear_tc_no_relu(x, M, x.stride(0), cin, packed, b, cout, y, cout, 0, mode)
        elif _TRAIN_FFMA and _rows_ok(x) and cout % 4 == 0 and cout >= 96:
            # exact fp32 on the CUDA cores (ev2h_linear_f32, 128 x 128 x 16 tiles): these GEMMs are tall and skinny (millions
            # of rows, 8-323 input channels), a shape the library's SIMT kernels run at ~13 TFLOP/s; narrower outputs would
            # waste the 128-column tile and stay with the library
            wt = torch.zeros(((cin + 15) // 16 * 16, (cout + 127) // 128 * 128), dtype=torch.float32, device=x.device)
            wt[:cin, :cout] = weight.detach().t()
            b = torch.zeros((wt.shape[1],), dtype=torch.float32, device=x.device)
            if bias is not None:
                b[:cout] = bias.detach()
            y = torch.empty((M, cout), dtype=torch.float32, device=x.device)
            _capi.linear_no_relu(x, M, x.stride(0), cin, wt, b, cout, y, cout)
        else:
            y = F.linear(x, weight, bias)
        ctx.save_for_backward(x, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x, weight = ctx.saved_tensors
        M, cin = x.shape
        cout = weight.shape[0]
        dy = dy.contiguous()
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            if _capi.tc_supported(cin, 0) and cin % 4 == 0 and cout <= 1024:
                mode = _capi.TC_TF32X3 if _TF32X3_PURE else _capi.TC_TF32_BF16C
                packed = _pack_dense(weight.detach(), mode)                    # dX = dY W: contraction over Cout
                zero = torch.zeros(((cin + 127) // 128 * 128,), dtype=torch.float32, device=dy.device)
                dx = torch.empty((M, cin), dtype=torch.float32, device=dy.device)
                _capi.linear_tc_no_relu(dy, M, cout, cout, packed, zero, cin, dx, cin, 0, mode)
            else:
                dx = dy @ weight
        want_db = ctx.has_bias and ctx.needs_input_grad[2]
        if ctx.needs_input_grad[1]:
            if _TRAIN_WGRAD and x.stride(1) == 1 and x.dtype == torch.float32:
                # contraction over the M rows: slabs in exact fp32, fixed-order sum; the bias gradient (column sums of dY)
                # comes out of the same pass over dY
                if want_db:
                    dw, db = _capi.wgrad(dy, x, want_bias=True)
                else:
                    dw = _capi.wgrad(dy, x)
            else:
                dw = dy.t() @ x
        if want_db and db is None:
            db = dy.sum(0)
        return dx, dw, db, None


def _linear_rows(x2d, weight, bias):
    cout, cin = weight.shape
    if _TRAIN_TC and _mlp_precision in ("tf32x3",) and x2d.is_cuda and cout % 4 == 0:
        fwd_tc = _TRAIN_TC == "all" and _rows_ok(x2d) and _capi.tc_supported(cout, 0) and cin <= 1024
        return _LinearRowsTC.apply(x2d, weight, bias, fwd_tc)
    return F.linear(x2d, weight, bias)


def _mlp_train_rows(x2d, convs, bns):
    """relu(bn(conv(.))) stack on rows [M, Cin] -> [M, Cout]; the convolutions have 1x1 / k = 1 kernels"""
    for conv, bn in zip(convs, bns):
        x2d = _linear_rows(x2d, conv.weight.view(conv.out_channels, -1), conv.bias)
        x2d = F.relu(_bn_rows(x2d, bn))
    return x2d


# --------------------------------------------------------------------------------------
# folded-weight cache for the inference path
# --------------------------------------------------------------------------------------
# nn.DataParallel (train.py:68) drives one Python thread per replica through the same module objects' caches:
# every cache below is keyed by device and only replaced under this lock (entries are immutable once published).
_CACHE_LOCK = threading.RLock()


class _FoldedMLP:
    """Per-device folded (conv bias + eval BatchNorm) weights of one conv/bn stack.

    Rebuilt whenever any source tensor was replaced or modified in place
    (``data_ptr`` / ``_version`` change), e.g. after ``load_state_dict`` or an
    optimiser step, and for every ``nn.DataParallel`` replica."""

    def __init__(self):
        self.by_device = {}     # device -> (key, layers); replicas on other GPUs keep their own entry
        self.generation = 0     # bumped at every refold: caches derived from the folded tensors key on it, not on addresses

    @staticmethod
    def _key(convs, bns):
        k = []
        for conv, bn in zip(convs, bns):
            for t in (conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var):
                k.append((t.data_ptr(), t._version, t.device))
        return tuple(k)

    def get(self, convs, bns, in_perm=None):
        key = self._key(convs, bns)
        dev = convs[0].weight.device
        with _CACHE_LOCK:
            hit = self.by_device.get(dev)
            if hit is not None and hit[0] == key:
                return hit[1]
            self.generation += 1
            layers = []
            for j, (conv, bn) in enumerate(zip(convs, bns)):
                w = conv.weight.detach().reshape(conv.out_channels, conv.in_channels)
                if j == 0 and in_perm is not None:
                    w = w[:, in_perm if torch.is_tensor(in_perm) else torch.tensor(list(in_perm), device=w.device)]
                wt, bias = _capi.fold_conv_bn(w, conv.bias, bn.weight, bn.bias, bn.running_mean, bn.running_var, bn.eps)
                layers.append({"wt": wt, "bias": bias, "cin": conv.in_channels, "cout": conv.out_channels, "packed": {},
                               "gen": (id(self), self.generation)})
            self.by_device[dev] = (key, layers)
            return layers


def _layer_mode(mode):
    """arithmetic of the per-layer tensor-core kernel for the selected precision: fp32-level = tf32 hi*hi + two bf16
    correction products (4 UMMA time units per 16 channels instead of the 6 of three tf32 products)"""
    if mode == _capi.TC_TF32X3 and _LINEAR_MIXED and not _TF32X3_PURE:
        return _capi.TC_F16X3 if _SPLIT == "f16" else _capi.TC_TF32_BF16C
    return mode


def _fused_mode(mode):
    """arithmetic of the fused kernel for the selected precision (see _SPLIT)"""
    if mode == _capi.TC_TF32X3 and not _TF32X3_PURE:
        return _capi.TC_F16X3 if _SPLIT == "f16" else _capi.TC_TF32_BF16C
    return mode


def _host_first_layer(L0):
    """host copy of a folded first layer (rows 0..7 of wt, bias): the gather mode of the fused kernel takes them as kernel
    parameters.  Made once per fold (one device-to-host copy), never per step."""
    h = L0.get("host")
    if h is None:
        with _CACHE_LOCK:
            h = L0.get("host")
            if h is None:
                h = L0["host"] = (L0["wt"][:8].contiguous().cpu(), L0["bias"].cpu())
    return h


def _mlp_rows(x, M, ld_x, layers, pool_rows, out, ld_out, out_col):
    """Run the folded MLP over M rows of x; the last layer max-pools runs of pool_rows rows
    into out[:, out_col : out_col + C_last]."""
    cur, ld = x, ld_x
    mode = {"tf32x3": _capi.TC_TF32X3, "bf16": _capi.TC_BF16}.get(_mlp_precision)
    lmode = _layer_mode(mode)
    for j, L in enumerate(layers):
        last = j == len(layers) - 1
        cin, cout = L["cin"], L["cout"]
        pool = pool_rows if last else 0
        if last:
            y, ld_y, col = out, ld_out, out_col
        else:
            ld_y, col = _pad4(cout), 0
            y = torch.empty((M, ld_y), dtype=torch.float32, device=x.device)
        # The tensor cores' fp32 accumulation error grows with the contraction length (measured: 2e-6 of max|y| at
        # 515 input channels, 1.1e-5 at 1536); past 1024 channels the fp32-level mode keeps its 1e-5 bar by running
        # the layer on the CUDA cores in exact fp32 (only fp3's first layer, 1536 channels, is that long).
        too_long = mode == _capi.TC_TF32X3 and cin > 1024
        if mode is not None and not too_long and _capi.tc_supported(cout, pool):
            packed = L["packed"].get(lmode)
            if packed is None:
                packed = L["packed"][lmode] = _capi.tc_pack(L["wt"], cin, cout, lmode)
            _capi.linear_relu_tc(cur, M, ld, cin, packed, L["bias"], cout, pool, y, ld_y, col, lmode)
        else:
            _capi.linear_relu(cur, M, ld, cin, L["wt"], L["bias"], cout, pool, y, ld_y, col)
        cur, ld = y, ld_y


def _check_inputs(xyz, points):
    if xyz.dim() != 3 or xyz.shape[1] != 3:
        raise RuntimeError("xyz must be [B, 3, N], got %s" % (tuple(xyz.shape),))
    if xyz.requires_grad and torch.is_grad_enabled():
        # the reference differentiates through grouped_xyz - new_xyz; the model never asks for it (SURVEY 3.3) and the
        # gather kernels return no coordinate gradient, so say so instead of returning zeros
        raise RuntimeError("ev2hands_b200 does not differentiate with respect to xyz (xyz.requires_grad is set); "
                           "detach the coordinates or keep the reference module for that use")
    if not xyz.is_cuda:
        raise RuntimeError("ev2hands_b200 runs on CUDA devices only (xyz is on %s); there is no CPU path" % xyz.device)
    if xyz.dtype != torch.float32 or (points is not None and points.dtype != torch.float32):
        raise RuntimeError("xyz and points must be float32")
    if points is not None and (points.dim() != 3 or points.shape[0] != xyz.shape[0] or points.shape[2] != xyz.shape[2]):
        raise RuntimeError("points must be [B, D, N] matching xyz, got %s" % (tuple(points.shape),))


def _to_rows(t_cf):
    """[B,D,N] (any strides) -> contiguous [B,N,D] through the transpose kernel."""
    B, D, N = t_cf.shape
    rows = torch.empty((B, N, D), dtype=torch.float32, device=t_cf.device)
    _capi.transpose(t_cf, (t_cf.stride(0), t_cf.stride(1), t_cf.stride(2)), B, D, N, rows, N * D, D, 0)
    return rows


def _rows_to_cf(rows):
    """contiguous [B,S,C] -> contiguous [B,C,S]."""
    B, S, C = rows.shape
    cf = torch.empty((B, C, S), dtype=torch.float32, device=rows.device)
    _capi.transpose(rows, (S * C, C, 1), B, S, C, cf, C * S, S, 0)
    return cf


class _LevelRows:
    """Point-major copy of one level of the encoder, the layout the kernels work in:
    ``rows`` [B, S, ld] float32 = [features (c channels) | centre xyz (3) | zero padding].

    A set-abstraction layer's fused path produces it; the channel-first tensor the reference's API returns is a
    transpose of it, made on demand.  The record rides on that tensor (attribute ``_ev2h_rows``) so that the next
    layer reads the rows it needs - [features | xyz] is exactly the input row of its per-point first layer -
    instead of transposing the channel-first tensor back.  ``matches`` guards the shortcut: same tensor objects'
    storage, not modified in place since."""

    def __init__(self, rows, c, new_xyz):
        self.rows, self.c = rows, c
        self.B, self.S, self.ld = rows.shape
        self.xyz_cf = new_xyz
        self._xyz_key = (new_xyz.data_ptr(), new_xyz._version)
        self._cf = None          # weak reference: the tensor owns the record, not the other way round
        self._cf_key = None

    def cf(self):
        """contiguous channel-first features [B, c, S] (transpose kernel); the same tensor while it is alive."""
        cf = self._cf() if self._cf is not None else None
        if cf is None:
            cf = torch.empty((self.B, self.c, self.S), dtype=torch.float32, device=self.rows.device)
            _capi.transpose(self.rows, (self.S * self.ld, self.ld, 1), self.B, self.S, self.c, cf, self.c * self.S, self.S, 0)
            cf._ev2h_rows = self
            self._cf, self._cf_key = weakref.ref(cf), (cf.data_ptr(), cf._version)
        return cf

    def matches(self, xyz, points):
        return (self._cf is not None and points is self._cf() and (points.data_ptr(), points._version) == self._cf_key
                and (xyz.data_ptr(), xyz._version) == self._xyz_key and tuple(xyz.shape) == (self.B, 3, self.S))


# How often a layer found the previous layer's rows riding on its channel-first input ("hit"), found a record that no
# longer matches the tensor ("stale": modified in place since; the layer transposes the tensor like for any input) or
# no record at all ("none": a fresh tensor).  bench.py reports the counts so that a lost shortcut shows up.
ROW_SHORTCUT = {"hit": 0, "stale": 0, "none": 0}


def _level_rows_of(xyz, points):
    """The _LevelRows record behind ``points`` (itself, or the one riding on a channel-first tensor), or None."""
    if isinstance(points, _LevelRows):
        return points
    rec = getattr(points, "_ev2h_rows", None)
    if rec is None:
        ROW_SHORTCUT["none"] += 1
        return None
    ok = rec.matches(xyz, points)
    ROW_SHORTCUT["hit" if ok else "stale"] += 1
    return rec if ok else None


def _wants_autograd(module, *tensors):
    if module.training:
        return True
    if not torch.is_grad_enabled():
        return False
    if any(t is not None and t.requires_grad for t in tensors):
        return True
    return any(p.requires_grad for p in module.parameters())


class PointNetSetAbstractionMsg(nn.Module):
    """Multi-scale-grouping set abstraction (reference :205-262)."""

    def __init__(self, npoint, radius_list, nsample_list, in_channel, mlp_list):
        super().__init__()
        self.npoint = npoint
        self.radius_list = radius_list
        self.nsample_list = nsample_list
        self.conv_blocks = nn.ModuleList()
        self.bn_blocks = nn.ModuleList()
        for widths in mlp_list:
            convs, bns = nn.ModuleList(), nn.ModuleList()
            last = in_channel + 3
            for w in widths:
                convs.append(nn.Conv2d(last, w, 1))
                bns.append(nn.BatchNorm2d(w))
                last = w
            self.conv_blocks.append(convs)
            self.bn_blocks.append(bns)
        self._folded = [_FoldedMLP() for _ in mlp_list]
        self._first_cat = {}      # device -> concatenated first-layer weights of the fused scales (per-point mode)

    # ---- shared front end: FPS + ball query -----------------------------------------
    def _pts8(self, xyz, points, strides):
        """[features | xyz | 0] per point, 32 bytes: one sector per gathered neighbour (gather mode of the fused kernel)."""
        return _capi.point_records(points, xyz, strides)

    def _fps(self, xyz, fps_start):
        """FPS of this layer on the current stream -> geometry record (dict)."""
        B, _, N = xyz.shape
        if fps_start is None:
            # same draw, from the same (CPU) generator, as pointnet2_utils.py:75
            fps_start = torch.randint(0, N, (B,), dtype=torch.long)
        strides = _capi.cf_strides(xyz)
        fps_idx, centres_rows, new_xyz = _capi.fps(xyz, strides, fps_start, B, N, self.npoint)
        return {"strides": strides, "fps_idx": fps_idx, "centres_rows": centres_rows, "new_xyz": new_xyz}

    def _pipelined_ok(self, xyz, D):
        """can the FPS / ball-query front end of this layer be pipelined (see _FPS_SPLITS)?"""
        B, _, N = xyz.shape
        if _FPS_SPLITS < 2 or not (_FUSED_ENABLED and _COMPACT and _mlp_precision in ("tf32x3", "bf16")) or _capi.LOG.timing:
            return False
        if N > 4096 or self.npoint % (32 * _FPS_SPLITS) != 0 or not all(k % 8 == 0 for k in self.nsample_list):
            return False
        # only while the sampling leaves SMs idle (one CTA per window): with more windows than SMs there is nothing to overlap with
        return B <= torch.cuda.get_device_properties(xyz.device).multi_processor_count

    def _fps_ball_pipelined(self, xyz, points, D, fps_start):
        """FPS in ranges on the current stream, the ball query (+ compacted row lists) of each finished range on a side
        stream -> the same geometry record _ball(_fps(...)) gives (bit-identical indices; the ORDER of the groups in the
        compacted row lists differs, as it already does from run to run: rows are reserved with atomics)."""
        B, _, N = xyz.shape
        S = self.npoint
        dev = xyz.device
        if fps_start is None:
            fps_start = torch.randint(0, N, (B,), dtype=torch.long)      # same draw, same (CPU) generator, as pointnet2_utils.py:75
        strides = _capi.cf_strides(xyz)
        start_dev = _capi.device_starts(fps_start, B, N, dev)
        ns = len(self.nsample_list)
        k_total = int(sum(self.nsample_list))
        fps_idx = torch.empty((B, S), dtype=torch.int32, device=dev)
        centres_rows = torch.empty((B, S, 3), dtype=torch.float32, device=dev)
        new_xyz = torch.empty((B, 3, S), dtype=torch.float32, device=dev)
        state_best = torch.empty((B, N), dtype=torch.float32, device=dev)
        state_cur = torch.empty((B,), dtype=torch.int32, device=dev)
        ball = torch.empty((B, S, k_total), dtype=torch.int32, device=dev)
        dedup = _DEDUP and D + 3 <= 8 and N <= 16384
        uniq = torch.empty_like(ball) if dedup else None
        rowmaps = [torch.empty((B * S * int(k),), dtype=torch.int32, device=dev) for k in self.nsample_list]
        blockgroups = [torch.empty((B * S * int(k) // 8,), dtype=torch.int32, device=dev) for k in self.nsample_list]
        n_rows = torch.empty((ns,), dtype=torch.int32, device=dev)
        main, side = torch.cuda.current_stream(dev), _scale_stream(dev, 9)
        side.wait_stream(main)
        pts8 = first = None
        with torch.cuda.stream(side):
            if dedup:
                pts8 = self._pts8(xyz, points, strides)
                first = _capi.first_occurrence(pts8)
        seg = S // _FPS_SPLITS
        for i in range(_FPS_SPLITS):
            _capi.fps_range(xyz, strides, start_dev, B, N, S, i * seg, (i + 1) * seg, state_best, state_cur, fps_idx, centres_rows, new_xyz)
            side.wait_stream(main)
            with torch.cuda.stream(side):
                _capi.ball_query_compact_range(xyz, strides, centres_rows, B, N, S, i * seg, seg, i == 0, self.radius_list,
                                               self.nsample_list, ball, first, uniq, rowmaps, blockgroups, n_rows)
        main.wait_stream(side)
        return {"strides": strides, "fps_idx": fps_idx, "centres_rows": centres_rows, "new_xyz": new_xyz, "pts8": pts8,
                "compact": (rowmaps, blockgroups, n_rows), "ball": ball}

    def _ball(self, geom, xyz, points, D, fused):
        """Ball query of every scale (plus the compacted row lists of the fused path) on the current stream;
        ``points`` is only needed for narrow inputs (the 32-byte gather records), ``D`` = feature channels."""
        B, _, N = xyz.shape
        strides, centres_rows = geom["strides"], geom["centres_rows"]
        geom["pts8"] = geom["compact"] = None
        want_fused = fused and _FUSED_ENABLED and _mlp_precision in ("tf32x3", "bf16")
        if want_fused and _COMPACT and all(k % 8 == 0 for k in self.nsample_list):
            # compacted row lists come out of the ball query itself; in gather mode (narrow inputs, N <= 4096) neighbours
            # whose 32-byte record repeats an earlier point give identical rows and are listed once
            first = None
            if _DEDUP and D + 3 <= 8 and N <= 16384:
                geom["pts8"] = self._pts8(xyz, points, strides)
                first = _capi.first_occurrence(geom["pts8"])
            ball, rowmaps, blockgroups, n_rows = _capi.ball_query_compact(xyz, strides, centres_rows, N, self.radius_list,
                                                                          self.nsample_list, first)
            geom["compact"] = (rowmaps, blockgroups, n_rows)
        else:
            ball = _capi.ball_query(xyz, strides, centres_rows, N, self.radius_list, self.nsample_list)
        geom["ball"] = ball
        return geom

    def forward(self, xyz, points, fps_start=None):
        """xyz [B,3,N], points [B,D,N] or None -> (new_xyz [B,3,S], new_points [B,sum D',S])."""
        _check_inputs(xyz, points)
        if _wants_autograd(self, points):
            with torch.no_grad():
                geom = self._ball(self._fps(xyz.detach(), fps_start), xyz.detach(), None, 0, fused=False)
            self.last_fps_idx, self.last_ball_idx = geom["fps_idx"], geom["ball"]        # exposed for parity tests
            return geom["new_xyz"], self._forward_autograd(xyz, points, geom["strides"], geom["centres_rows"], geom["ball"])
        new_xyz, rec = self.forward_rows(xyz, points, fps_start)
        return new_xyz, rec.cf()

    def forward_rows(self, xyz, points, fps_start=None, geom=None):
        """The inference path in the kernels' own layout: like ``forward`` but returns the level as a ``_LevelRows``
        record (point-major rows; ``.cf()`` gives the reference's channel-first tensor).  ``points`` may be such a
        record from the previous layer; ``geom`` = this layer's FPS + ball query if the caller already ran them
        (``_fps`` / ``_ball``, e.g. on another stream)."""
        with torch.no_grad():
            rows_in = _level_rows_of(xyz, points)
            D = rows_in.c if rows_in is not None else (0 if points is None else points.shape[1])
            if isinstance(points, _LevelRows):
                # wide inputs are consumed as rows; narrow ones (gather records) want the channel-first tensor
                points = None if (D + 3 > 8 or _PER_POINT_ALWAYS) else rows_in.cf()
            if geom is None:
                if self._pipelined_ok(xyz, D):
                    geom = self._fps_ball_pipelined(xyz, points, D, fps_start)
                else:
                    geom = self._ball(self._fps(xyz, fps_start), xyz, points, D, fused=True)
            self.last_fps_idx, self.last_ball_idx = geom["fps_idx"], geom["ball"]        # exposed for parity tests
            return geom["new_xyz"], self._forward_fused(xyz, points, rows_in, D, geom)

    def _forward_fused(self, xyz, points, rows_in, D, geom):
        """``points`` [B,D,N] channel-first, or ``rows_in`` (the previous layer's _LevelRows: [features | xyz] rows)."""
        B, _, N = xyz.shape
        S = self.npoint
        strides, centres_rows, ball = geom["strides"], geom["centres_rows"], geom["ball"]
        c_total = sum(convs[-1].out_channels for convs in self.conv_blocks)
        # pooled features, then the centres: [features | xyz | 0] is the next layer's per-point input row
        ld_out = _pad4(c_total + 3)
        out_rows = torch.zeros((B, S, ld_out), dtype=torch.float32, device=xyz.device)
        out_rows[:, :, c_total:c_total + 3] = centres_rows
        mode = {"tf32x3": _capi.TC_TF32X3, "bf16": _capi.TC_BF16}.get(_mlp_precision)
        fmode = _fused_mode(mode)
        all_layers = [self._folded[i].get(self.conv_blocks[i], self.bn_blocks[i]) for i in range(len(self.nsample_list))]
        widths = [[L["cout"] for L in layers] for layers in all_layers]

        # Which scales can run in the fused tensor-core kernel, and with which first-layer mode.
        per_point = D + 3 > 8 or _PER_POINT_ALWAYS
        fused = [mode is not None and _FUSED_ENABLED and _capi.fused_supported(K, w, D + 3, per_point, fmode)
                 for K, w in zip(self.nsample_list, widths)]

        pts8 = P = C = None
        p_cols = []
        if any(fused) and not per_point:
            pts8 = geom["pts8"] if geom["pts8"] is not None else self._pts8(xyz, points, strides)
        elif any(fused):
            # layer 1 once per point: P = W1'[f; xyz] + b1' for every fused scale side by side,
            # C = W1'_xyz centre per centre (see sa_fused_tc.cu)
            if rows_in is not None:
                x_pts, ld_pts = rows_in.rows.view(B * N, rows_in.ld), rows_in.ld      # the previous layer left them ready
            else:
                ld_pts = _pad4(D + 3)
                x_pts = torch.zeros((B * N, ld_pts), dtype=torch.float32, device=xyz.device)
                _capi.transpose(points, (points.stride(0), points.stride(1), points.stride(2)), B, D, N, x_pts, N * ld_pts, ld_pts, 0)
                _capi.transpose(xyz, strides, B, 3, N, x_pts, N * ld_pts, ld_pts, D)
            c1_total = sum(w[0] for w, f in zip(widths, fused) if f)
            P = torch.empty((B * N, c1_total), dtype=torch.float32, device=xyz.device)
            C = torch.empty((B * S, c1_total), dtype=torch.float32, device=xyz.device)
            if c_total % 4 == 0:
                # this layer's output rows already hold [features | centre xyz | 0]: the centre GEMM reads the xyz columns in place
                ctr4, ld_ctr = out_rows.view(B * S, ld_out)[:, c_total:], ld_out
            else:
                ctr4, ld_ctr = torch.zeros((B * S, 4), dtype=torch.float32, device=xyz.device), 4
                ctr4[:, :3] = centres_rows.reshape(B * S, 3)
            # every fused scale's first layer in ONE GEMM: the folded weights side by side (same input rows)
            firsts = [layers[0] for layers, f in zip(all_layers, fused) if f]
            # keyed on the refold generation of every source stack (an address can be handed out again by the caching
            # allocator after a refold) and kept per device in an object nn.DataParallel replicas share
            key = tuple(L0["gen"] for L0 in firsts)
            with _CACHE_LOCK:
                cat = self._first_cat.get(xyz.device)
            if cat is None or cat["key"] != key:
                rows = firsts[0]["wt"].shape[0]
                wt = torch.zeros((rows, (c1_total + 127) // 128 * 128), dtype=torch.float32, device=xyz.device)
                bias = torch.zeros((wt.shape[1],), dtype=torch.float32, device=xyz.device)
                c = 0
                for L0 in firsts:
                    wt[:, c:c + L0["cout"]] = L0["wt"][:, :L0["cout"]]
                    bias[c:c + L0["cout"]] = L0["bias"][:L0["cout"]]
                    c += L0["cout"]
                wx = torch.zeros((16, wt.shape[1]), dtype=torch.float32, device=xyz.device)
                wx[:3] = wt[D:D + 3]
                cat = {"key": key, "wt": wt, "bias": bias, "wt_xyz": wx, "zero_bias": torch.zeros_like(bias), "packed": {}}
                with _CACHE_LOCK:
                    self._first_cat[xyz.device] = cat
            if mode == _capi.TC_TF32X3 and _capi.tc_supported(c1_total, 0):
                # the wide per-point layer on the tensor cores (fp32-level accuracy); bf16 mode keeps it
                # in exact fp32 so that only the two tensor-core layers carry bf16 rounding
                lmode = _layer_mode(mode)
                if lmode not in cat["packed"]:
                    cat["packed"][lmode] = _capi.tc_pack(cat["wt"], D + 3, c1_total, lmode)
                _capi.linear_tc_no_relu(x_pts, B * N, ld_pts, D + 3, cat["packed"][lmode], cat["bias"], c1_total, P, c1_total, 0, lmode)
            else:
                _capi.linear_no_relu(x_pts, B * N, ld_pts, D + 3, cat["wt"], cat["bias"], c1_total, P, c1_total, 0)
            _capi.linear_no_relu(ctr4, B * S, ld_ctr, 3, cat["wt_xyz"], cat["zero_bias"], c1_total, C, c1_total, 0)
            col = 0
            for layers, f in zip(all_layers, fused):
                p_cols.append(col if f else None)
                if f:
                    col += layers[0]["cout"]

        compact = geom["compact"] if any(fused) else None
        self.last_compact_rows = None if compact is None else compact[2]     # int32 [n_scales] on the device (diagnostics)

        feats_rows = None
        ld_x = _pad4(D + 3)
        k_off = col = 0
        main_stream = torch.cuda.current_stream(xyz.device)
        forked = []
        n_fused_seen = 0
        for i, K in enumerate(self.nsample_list):
            layers = all_layers[i]
            if fused[i]:
                launch_stream = main_stream
                if _SCALE_STREAMS and sum(fused) > 1 and n_fused_seen > 0 and not _capi.LOG.timing:
                    launch_stream = _scale_stream(xyz.device, n_fused_seen)
                n_fused_seen += 1
                use = layers[1:]      # layer 1: per point (wide inputs) or in the loader warps (<= 8 channels)
                kc = _capi.fused_kc(fmode, [L["cout"] for L in use])
                packed = []
                for li, L in enumerate(use):
                    # the last layer's weights are the UMMA A operand (output channels = TMEM lanes): 128-row images
                    key = (fmode, kc, 128 if li == 1 else 16)
                    if key not in L["packed"]:
                        L["packed"][key] = _capi.tc_pack(L["wt"], L["cin"], L["cout"], fmode, kc, key[2])
                    packed.append(L["packed"][key])
                w1_host, b1_host = (None, None) if per_point else _host_first_layer(layers[0])
                if launch_stream is not main_stream:
                    launch_stream.wait_stream(main_stream)        # behind everything issued so far (inputs, packed weights)
                    forked.append(launch_stream)
                with torch.cuda.stream(launch_stream):
                    _capi.sa_msg_fused(ball, k_off, centres_rows, B, N, S, K, pts8, D, w1_host, b1_host,
                                       P, 0 if P is None else P.shape[1], p_cols[i] if per_point else 0,
                                       C, 0 if C is None else C.shape[1], p_cols[i] if per_point else 0,
                                       layers[0]["cout"], [L["cout"] for L in use], packed, [L["bias"] for L in use],
                                       out_rows, ld_out, col, fmode,
                                       compact=None if compact is None else (compact[0][i], compact[1][i], compact[2][i:i + 1]))
            else:
                if feats_rows is None and rows_in is not None:
                    feats_rows = rows_in.rows[:, :, :D].contiguous()
                elif feats_rows is None and points is not None:
                    feats_rows = _to_rows(points)
                per_window = S * K * 4 * (ld_x + sum(_pad4(l["cout"]) for l in layers[:-1]))
                chunk = max(1, min(B, _WORKSPACE_BYTES // per_window))
                for b0 in range(0, B, chunk):
                    nb = min(chunk, B - b0)
                    M = nb * S * K
                    x = torch.empty((M, ld_x), dtype=torch.float32, device=xyz.device)
                    _capi.group_gather(xyz[b0:b0 + nb], strides, None if feats_rows is None else feats_rows[b0:b0 + nb], D,
                                       centres_rows[b0:b0 + nb], ball[b0:b0 + nb], k_off, nb, N, S, K, x, ld_x)
                    _mlp_rows(x, M, ld_x, layers, K, out_rows[b0:b0 + nb], ld_out, col)
            k_off += K
            col += layers[-1]["cout"]
        for st in forked:
            main_stream.wait_stream(st)
        return _LevelRows(out_rows, c_total, geom["new_xyz"])

    def _forward_autograd(self, xyz, points, strides, centres_rows, ball):
        B, _, N = xyz.shape
        feats_rows = points.permute(0, 2, 1).contiguous() if points is not None else None
        pooled = []
        k_off = 0
        for i, K in enumerate(self.nsample_list):
            g = _GroupGather.apply(feats_rows, xyz.detach(), strides, N, centres_rows, ball, k_off, K)  # [B,S,K,D+3]
            if _TRAIN_ROWS:
                Bg, Sg = g.shape[:2]
                h = _mlp_train_rows(g.flatten(0, 2), self.conv_blocks[i], self.bn_blocks[i])      # a view, also of padded rows
                pooled.append(h.view(Bg, Sg, K, h.shape[-1]).max(dim=2)[0].permute(0, 2, 1))    # torch.max(x, 2)[0], :257
            else:
                g = g.permute(0, 3, 2, 1).contiguous()                                              # [B,D+3,K,S]
                for conv, bn in zip(self.conv_blocks[i], self.bn_blocks[i]):
                    g = F.relu(bn(conv(g)))
                pooled.append(_GroupMax.apply(g))
            k_off += K
        return torch.cat(pooled, dim=1)


class PointNetSetAbstraction(nn.Module):
    """Single-scale set abstraction (reference :161-202); the model only uses
    ``group_all=True`` (TEHNet.py:44, :129)."""

    def __init__(self, npoint, radius, nsample, in_channel, mlp, group_all):
        super().__init__()
        self.npoint = npoint
        self.radius = radius
        self.nsample = nsample
        self.mlp_convs = nn.ModuleList()
        self.mlp_bns = nn.ModuleList()
        last = in_channel
        for w in mlp:
            self.mlp_convs.append(nn.Conv2d(last, w, 1))
            self.mlp_bns.append(nn.BatchNorm2d(w))
            last = w
        self.group_all = group_all
        self._folded = _FoldedMLP()
        self._folded_rows = _FoldedMLP()       # first layer's input channels in [points | xyz] order (see _group_all_rows)

    def forward(self, xyz, points, fps_start=None):
        """xyz [B,3,N], points [B,D,N] or None -> (new_xyz [B,3,S], new_points [B,D',S])."""
        _check_inputs(xyz, points)
        autograd = _wants_autograd(self, points)
        if self.group_all:
            B = xyz.shape[0]
            new_xyz = torch.zeros((B, 3, 1), dtype=torch.float32, device=xyz.device)
            if autograd:
                return new_xyz, self._group_all_autograd(xyz, points)
            with torch.no_grad():
                rows_in = _level_rows_of(xyz, points)
                if rows_in is not None:
                    return new_xyz, self._group_all_rows(rows_in)
                return new_xyz, self._group_all_fused(xyz, points)
        return self._forward_sampled(xyz, points, fps_start, autograd)

    def forward_rows(self, xyz, points):
        """group_all inference on the previous layer's ``_LevelRows`` record -> pooled features [B, D', 1]."""
        if not self.group_all or not isinstance(points, _LevelRows):
            raise RuntimeError("forward_rows: group_all layers fed with a _LevelRows record only")
        with torch.no_grad():
            return self._group_all_rows(points)

    # ---- group_all ---------------------------------------------------------------------
    def _group_all_rows(self, rec):
        """group_all over the previous layer's rows [points | xyz | 0] as they are: the reference's channel order
        is [xyz, points] (:141-158), so the first layer's input channels are permuted instead of the data."""
        B, N, D = rec.B, rec.S, rec.c
        layers = self._folded_rows.get(self.mlp_convs, self.mlp_bns, in_perm=list(range(3, 3 + D)) + [0, 1, 2])
        c_out = layers[-1]["cout"]
        out = torch.zeros((B, c_out), dtype=torch.float32, device=rec.rows.device)
        _mlp_rows(rec.rows.view(B * N, rec.ld), B * N, rec.ld, layers, N, out, c_out, 0)
        return out.view(B, c_out, 1)

    def _group_all_fused(self, xyz, points):
        B, _, N = xyz.shape
        D = 0 if points is None else points.shape[1]
        cin = 3 + D
        ld_x = _pad4(cin)
        # rows = [xyz | points], the channel order of sample_and_group_all (:141-158)
        x = torch.zeros((B * N, ld_x), dtype=torch.float32, device=xyz.device) if ld_x != cin else \
            torch.empty((B * N, ld_x), dtype=torch.float32, device=xyz.device)
        _capi.transpose(xyz, _capi.cf_strides(xyz), B, 3, N, x, N * ld_x, ld_x, 0)
        if points is not None:
            _capi.transpose(points, (points.stride(0), points.stride(1), points.stride(2)), B, D, N, x, N * ld_x, ld_x, 3)
        layers = self._folded.get(self.mlp_convs, self.mlp_bns)
        c_out = layers[-1]["cout"]
        out = torch.zeros((B, c_out), dtype=torch.float32, device=xyz.device)
        _mlp_rows(x, B * N, ld_x, layers, N, out, c_out, 0)
        return out.view(B, c_out, 1)

    def _group_all_autograd(self, xyz, points):
        g = xyz if points is None else torch.cat([xyz, points], dim=1)                               # [B,C,N]
        if _TRAIN_ROWS:
            B, C, N = g.shape
            h = _mlp_train_rows(g.permute(0, 2, 1).reshape(B * N, C), self.mlp_convs, self.mlp_bns)
            return h.view(B, N, h.shape[-1]).max(dim=1)[0].unsqueeze(-1)                              # [B,C',1]
        g = g.unsqueeze(-1)                                                                          # [B,C,N,1]
        for conv, bn in zip(self.mlp_convs, self.mlp_bns):
            g = F.relu(bn(conv(g)))
        return _GroupMax.apply(g)

    # ---- sampled single-scale (not reached by the model; API completeness) --------------
    def _forward_sampled(self, xyz, points, fps_start, autograd):
        B, _, N = xyz.shape
        S, K = self.npoint, self.nsample
        D = 0 if points is None else points.shape[1]
        with torch.no_grad():
            if fps_start is None:
                fps_start = torch.randint(0, N, (B,), dtype=torch.long)
            strides = _capi.cf_strides(xyz)
            _, centres_rows, new_xyz = _capi.fps(xyz.detach(), strides, fps_start, B, N, S)
            ball = _capi.ball_query(xyz.detach(), strides, centres_rows, N, [self.radius], [K])
        # reference channel order here is [rel_xyz, points] (:128); the gather kernel emits
        # [points, rel_xyz], so the first layer's input channels are permuted instead
        perm = torch.tensor(list(range(3, 3 + D)) + [0, 1, 2], device=xyz.device)
        if autograd:
            feats_rows = points.permute(0, 2, 1).contiguous() if points is not None else None
            g = _GroupGather.apply(feats_rows, xyz.detach(), strides, N, centres_rows, ball, 0, K)
            g = g[..., torch.argsort(perm)].permute(0, 3, 2, 1).contiguous()
            for conv, bn in zip(self.mlp_convs, self.mlp_bns):
                g = F.relu(bn(conv(g)))
            return new_xyz, _GroupMax.apply(g)
        with torch.no_grad():
            feats_rows = _to_rows(points) if points is not None else None
            layers = self._folded.get(self.mlp_convs, self.mlp_bns, in_perm=perm)
            ld_x = _pad4(D + 3)
            c_out = layers[-1]["cout"]
            out_rows = torch.zeros((B, S, c_out), dtype=torch.float32, device=xyz.device)
            x = torch.empty((B * S * K, ld_x), dtype=torch.float32, device=xyz.device)
            _capi.group_gather(xyz, strides, feats_rows, D, centres_rows, ball, 0, B, N, S, K, x, ld_x)
            _mlp_rows(x, B * S * K, ld_x, layers, K, out_rows, c_out, 0)
            return new_xyz, _rows_to_cf(out_rows)


class PointNetFeaturePropagation(nn.Module):
    """Decoder block (reference :265-315; SURVEY.md section 8f row N1): inverse-distance interpolation of
    the coarse level's features onto the fine level's points, concat with the skip features, Conv1d +
    BatchNorm1d + ReLU stack.  ``eval()`` + ``no_grad`` runs the CUDA path (3-NN scan, interpolation written
    straight into the concat buffer, tensor-core MLP over rows); training keeps the PyTorch formulation."""

    def __init__(self, in_channel, mlp):
        super().__init__()
        self.mlp_convs = nn.ModuleList()
        self.mlp_bns = nn.ModuleList()
        last = in_channel
        for w in mlp:
            self.mlp_convs.append(nn.Conv1d(last, w, 1))
            self.mlp_bns.append(nn.BatchNorm1d(w))
            last = w
        self._folded = _FoldedMLP()

    def forward(self, xyz1, xyz2, points1, points2):
        """xyz1 [B,3,N], xyz2 [B,3,S], points1 [B,D1,N] or None, points2 [B,D2,S] -> [B,D',N]."""
        S = xyz2.shape[2]
        if not xyz1.is_cuda:
            raise RuntimeError("ev2hands_b200 runs on CUDA devices only (xyz1 is on %s); there is no CPU path" % xyz1.device)
        if _wants_autograd(self, points1, points2) or (S != 1 and S < 3):
            return self._forward_autograd(xyz1, xyz2, points1, points2)
        with torch.no_grad():
            return self._forward_cuda(xyz1, xyz2, points1, points2)

    def _forward_cuda(self, xyz1, xyz2, points1, points2):
        _check_inputs(xyz1, points1)
        _check_inputs(xyz2, points2)
        B, _, N = xyz1.shape
        S = xyz2.shape[2]
        D1 = 0 if points1 is None else points1.shape[1]
        D2 = points2.shape[1]
        dev = xyz1.device
        if S == 1:        # points2.repeat(1, N, 1) (:291): the single source with weight 1
            idx = torch.zeros((B, N, 3), dtype=torch.int32, device=dev)
            weight = torch.zeros((B, N, 3), dtype=torch.float32, device=dev)
            weight[:, :, 0] = 1.0
        else:
            idx, weight = _capi.three_nn(xyz1, xyz2)
        self.last_idx, self.last_weight = idx, weight             # exposed for parity tests
        f2 = _to_rows(points2)                                    # [B,S,ld2]
        ld_x = _pad4(D1 + D2)
        # rows = [points1 | interpolated], the order of the reference's cat (:305)
        x = (torch.zeros if ld_x != D1 + D2 else torch.empty)((B * N, ld_x), dtype=torch.float32, device=dev)
        if points1 is not None:
            _capi.transpose(points1, (points1.stride(0), points1.stride(1), points1.stride(2)), B, D1, N, x, N * ld_x, ld_x, 0)
        _capi.three_interp(f2, f2.shape[2], idx, weight, B, N, S, D2, x, ld_x, D1)
        layers = self._folded.get(self.mlp_convs, self.mlp_bns)
        c_out = layers[-1]["cout"]
        ld_o = _pad4(c_out)
        out = torch.empty((B, N, ld_o), dtype=torch.float32, device=dev)
        _mlp_rows(x, B * N, ld_x, layers, 0, out, ld_o, 0)
        cf = torch.empty((B, c_out, N), dtype=torch.float32, device=dev)
        _capi.transpose(out, (N * ld_o, ld_o, 1), B, N, c_out, cf, c_out * N, N, 0)
        # the point-major rows ride on the channel-first result (like _LevelRows): the heads that follow the decoder
        # (ev2hands_b200.tehnet) work on rows and read them instead of transposing back
        cf._ev2h_fp_rows = (out, ld_o, c_out, cf._version)
        return cf

    def _forward_autograd(self, xyz1, xyz2, points1, points2):
        p1 = xyz1.transpose(1, 2)
        p2 = xyz2.transpose(1, 2)
        f2 = points2.transpose(1, 2)
        B, N, _ = p1.shape
        S = p2.shape[1]
        if S == 1:
            up = f2.expand(B, N, f2.shape[-1])
        else:
            d = -2 * torch.matmul(p1, p2.transpose(1, 2))
            d = d + (p1 * p1).sum(-1, keepdim=True) + (p2 * p2).sum(-1).unsqueeze(1)
            d3, i3 = d.sort(dim=-1)
            d3, i3 = d3[..., :3], i3[..., :3]
            w = 1.0 / (d3 + 1e-8)
            w = w / w.sum(dim=2, keepdim=True)
            # min(3, S) neighbours: with S = 2 both sources are interpolated
            nb = torch.gather(f2.unsqueeze(1).expand(B, N, S, f2.shape[-1]), 2,
                              i3.unsqueeze(-1).expand(B, N, i3.shape[-1], f2.shape[-1]))
            up = (nb * w.unsqueeze(-1)).sum(dim=2)
        h = up if points1 is None else torch.cat([points1.transpose(1, 2), up], dim=-1)
        if _TRAIN_ROWS:
            h = _mlp_train_rows(h.reshape(B * N, h.shape[-1]), self.mlp_convs, self.mlp_bns)
            return h.view(B, N, h.shape[-1]).transpose(1, 2)
        h = h.transpose(1, 2)
        for conv, bn in zip(self.mlp_convs, self.mlp_bns):
            h = F.relu(bn(conv(h)))
        return h
