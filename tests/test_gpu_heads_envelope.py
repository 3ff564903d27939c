"""Envelope of the decoder and head kernels against float64 restatements of the same operations.

What follows the encoder in TEHNet's eval path runs on four kernels: the 3-NN scan and the inverse-distance
interpolation of the decoder (three_nn.cu), then the decoder's MLP on the per-layer tensor-core kernel; the Conv1d of
the classifier and the query convolutions, whose shifted rows are gathered by that kernel's loaders and whose optional
per-channel affine follows the ReLU (linear_tc.cu), and the class-wise attention (attention.cu).  Each is checked here
at the shapes and edges where such kernels go wrong: sequences shorter than the tap reach, several accumulator blocks
under a per-channel affine, NaN next to a sequence boundary and in padding columns, empty attention splits, softmax
logits near fp32's exp range, ties at the 3-NN source tile edge, both interpolation paths and the grid-stride wrap,
unaligned output views, and the decoder and heads modules at B = 64 and at the long window N = 16384.

Bars: module and per-layer results within 1e-5 of max|reference| per tensor in the fp32-level modes (fp16 split,
tf32 + bf16 corrections, three tf32 products, exact fp32) and 1e-2 in bf16 (in proportion for contractions longer
than 1024 channels, and with sqrt(N / 2048) for the heads beyond the model's 2048 points; see the tests); per-kernel
results elementwise against
the same operation over absolute values (the first-order rounding bound of exact fp32 kernels, or 1e-5 / 1e-2 of it
for the tensor-core modes); the 3-NN indices, weights and interpolation bit for bit against fp32 restatements in the
kernels' operation order."""
import json
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import ev2hands_b200 as e2h
from ev2hands_b200 import _capi, synth, tehnet
from ev2hands_b200 import pointnet2_utils as pu
from ev2hands_b200.encoder import load_numpy_state
from oracle import sa_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24                      # unit roundoff of fp32
MODES = ("f16", "tf32", "pure", "bf16")
TOL = {"f16": 1e-5, "tf32": 1e-5, "pure": 1e-5, "bf16": 1e-2, "fp32": 1e-5}
TC_MODE = {"f16": _capi.TC_F16X3, "tf32": _capi.TC_TF32_BF16C, "pure": _capi.TC_TF32X3, "bf16": _capi.TC_BF16}
MEASURED = {}


def _record(key, payload):
    """collect the measured errors; with EV2H_TEST_RECORD_DIR set, also write them there as heads_envelope.json"""
    MEASURED[key] = payload
    d = os.environ.get("EV2H_TEST_RECORD_DIR")
    if not d:
        return
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "heads_envelope.json"), "w") as f:
            json.dump(MEASURED, f, indent=1, sort_keys=True)
    except OSError:
        pass


@pytest.fixture(autouse=True)
def strict_fp32():
    """the float64 references use cuBLAS / cuDNN: keep any fp32 op they touch out of tf32"""
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _set_mode(monkeypatch, mode):
    """module globals, not environment variables (several knobs are read once at import)"""
    monkeypatch.setattr(pu, "_mlp_precision", {"bf16": "bf16", "fp32": "fp32"}.get(mode, "tf32x3"))
    monkeypatch.setattr(pu, "_SPLIT", "tf32" if mode == "tf32" else "f16")
    monkeypatch.setattr(pu, "_TF32X3_PURE", mode == "pure")
    monkeypatch.setattr(pu, "_LINEAR_MIXED", True)


def rel_err(got, want):
    got, want = got.detach().double(), want.detach().double().to(got.device)
    return float((got - want).abs().max() / max(float(want.abs().max()), 1e-30))


def _elementwise(err, bound):
    """max of |err| / bound (bound: the same operation over absolute values); 0 / 0 counts as 0, and a NaN error as
    infinite (a NaN result must not pass as a small one)"""
    r = torch.where(bound > 0, err.abs() / bound, torch.where(err == 0, 0.0, float("inf")))
    return float(torch.nan_to_num(r, nan=float("inf")).max())


def _lib_fixed_unaligned():
    """unaligned output views are only legal from ABI 102 on (before, they meet float4 stores): never run them on an
    older library loaded through EV2H_LIB"""
    return _capi.lib().ev2h_version() >= 102


def _unaligned_view(shape, fill=0.0):
    """a float32 [rows, cols] view whose base is 4 bytes past a 16-byte boundary (a storage offset of one element)"""
    n = int(np.prod(shape))
    buf = torch.full((n + 4,), fill, dtype=torch.float32, device=DEV)
    v = buf[1:n + 1].view(shape)
    assert v.data_ptr() % 16 == 4
    return v


# ================================================================== A. ev2h_conv1d_tc ==============================
def _conv_w(cin, cout, taps, seed):
    """fp32-representable Conv1d weights [Cout, Cin, T] and bias, as float64 on the device"""
    g = torch.Generator().manual_seed(seed)
    w = (torch.randn(cout, cin, taps, generator=g) / (cin * taps) ** 0.5).double()
    b = (0.1 * torch.randn(cout, generator=g)).double()
    return w.to(DEV), b.to(DEV)


POST_VARIANTS = [(kind, relu) for kind in ("both", "scale", "shift", "none") for relu in (True, False)]


def _post(cout, kind, seed):
    """per-channel affine after the activation: random scale in [-1, 2) (negative scales included) and shift"""
    g = torch.Generator().manual_seed(seed)
    scale = (3 * torch.rand(cout, generator=g) - 1).to(DEV) if kind in ("both", "scale") else None
    shift = torch.randn(cout, generator=g).to(DEV) if kind in ("both", "shift") else None
    return scale, shift


def conv_ref(x64, w, b, seq, relu, scale, shift):
    """float64 Conv1d over sequences of `seq` rows of x64 [M, Cin] (zero padding taps // 2), then ReLU, then
    * scale + shift -> (y [M, Cout], bound: the same over absolute values)"""
    M, cin = x64.shape
    s = x64.view(M // seq, seq, cin).permute(0, 2, 1)
    pad = w.shape[2] // 2
    y = F.conv1d(s, w, b, padding=pad).permute(0, 2, 1).reshape(M, -1)
    bound = F.conv1d(s.abs(), w.abs(), b.abs(), padding=pad).permute(0, 2, 1).reshape(M, -1)
    if relu:
        y = torch.relu(y)
    if scale is not None:
        y, bound = y * scale.double(), bound * scale.double().abs()
    if shift is not None:
        y, bound = y + shift.double(), bound + shift.double().abs()
    return y, bound


def _padded_width(cout):
    """columns the kernel writes without pooling: Cout rounded up to its accumulator block width"""
    return (cout + 15) // 16 * 16 if cout < 256 else (cout + 255) // 256 * 256


_PACKS = {}


def _pack(w, b, tc, key):
    k = (key, tc)
    if k not in _PACKS:
        _PACKS[k] = tehnet._pack_conv1d(w, b, tc)
    return _PACKS[k]


def run_conv(x, cin, taps, seq, L, relu, scale, shift, tc, y=None, col=0):
    """ev2h_conv1d_tc on rows x [M, ld_x]; y defaults to [M, pad4(Cout)] rows"""
    M, ld_x = x.shape
    cout = L["cout"]
    if y is None:
        y = torch.full((M, pu._pad4(cout)), 777.0, dtype=torch.float32, device=DEV)
    _capi.conv1d_tc(x, M, ld_x, cin, taps, seq, L["packed"], L["bias"], cout, relu, scale, shift, y, y.shape[1], col, tc)
    torch.cuda.synchronize()
    return y


# name -> (B, N, Cin, Cout, taps); the post-affine variant cycles through POST_VARIANTS by case
CONV_CASES = {
    # the model's layers: classifier (k = 1, 256 -> 256 and 256 -> 4 classes), query convolution (k = 3)
    "cls1": (4, 2048, 256, 256, 1), "cls2": (4, 2048, 256, 4, 1), "query": (4, 2048, 256, 256, 3),
    # 5 taps: sequences shorter than the tap reach, many sequences per 128-row tile
    "t5-n1": (37, 1, 32, 16, 5), "t5-n2": (29, 2, 32, 100, 5), "t5-n3": (50, 3, 288, 16, 5),
    "t5-n5": (40, 5, 32, 256, 5), "t5-n130": (3, 130, 288, 512, 5),
    # 3 taps: sequence lengths around the tile size, 1 to 3 accumulator blocks
    "t3-n1": (64, 1, 32, 4, 3), "t3-n2": (70, 2, 512, 16, 3), "t3-n3": (45, 3, 32, 768, 3),
    "t3-n64": (9, 64, 288, 100, 3), "t3-n127": (5, 127, 32, 256, 3), "t3-n129": (5, 129, 512, 100, 3),
    "t3-n200": (3, 200, 288, 768, 3), "t3-n4097": (2, 4097, 32, 512, 3),
    # k = 1 at the other widths
    "k1-288x768": (3, 300, 288, 768, 1), "k1-512x100": (2, 777, 512, 100, 1),
    # dozens of tiles per CTA (4096 tiles on 148 SMs); the reference runs on sampled sequences
    "long": (256, 2048, 256, 256, 3),
}
LONG_SAMPLE = [0, 1, 77, 128, 200, 255]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(CONV_CASES))
def test_conv1d_tc_vs_f64(name, mode):
    B, N, cin, cout, taps = CONV_CASES[name]
    i = list(CONV_CASES).index(name)
    kind, relu = POST_VARIANTS[i % len(POST_VARIANTS)]
    tc = TC_MODE[mode]
    w, b = _conv_w(cin, cout, taps, seed=100 + i)
    L = _pack(w, b, tc, name)
    scale, shift = _post(cout, kind, seed=200 + i)
    M = B * N
    x = torch.randn(M, cin, device=DEV, generator=torch.Generator(device=DEV).manual_seed(300 + i))
    e2h.check_numeric_range(DEV)
    y = run_conv(x, cin, taps, N, L, relu, scale, shift, tc)
    assert e2h.check_numeric_range(DEV), "range flag raised by in-range inputs"
    assert (y[:, cout:] == 0).all(), "padding columns up to pad4(Cout) must be zero"
    if name == "long":
        rows = torch.cat([torch.arange(s * N, (s + 1) * N, device=DEV) for s in LONG_SAMPLE])
        x, y, seq_m = x[rows], y[rows], len(LONG_SAMPLE) * N
    else:
        seq_m = M
    want, bound = conv_ref(x.double(), w, b, N, relu, scale, shift)
    got = y[:seq_m, :cout]
    res = {"rel": rel_err(got, want), "elem": _elementwise(got.double() - want, bound)}
    _record("conv-%s-%s" % (name, mode), res)
    assert torch.isfinite(got).all()
    # the per-tensor bar holds for contractions of up to 1024 channels (the library sends longer fp32-level layers of
    # the MLP to the exact fp32 kernel for that reason, pointnet2_utils._mlp_rows); the tensor cores' fp32
    # accumulation error grows with the length, so longer ones (taps * Cin up to 2560 here) get it in proportion -
    # the elementwise bar below stays the same for every length
    assert res["rel"] <= TOL[mode] * max(1.0, taps * cin / 1024), res
    assert res["elem"] <= TOL[mode], res


@pytest.mark.parametrize("mode", MODES)
def test_conv1d_post_affine_variants(mode):
    """every combination of scale / shift (each may be NULL on its own) with ReLU on and off, at Cout = 768: three
    accumulator blocks, so a per-channel affine indexed without the block's column offset would show"""
    B, N, cin, cout, taps = 3, 200, 288, 768, 3
    tc = TC_MODE[mode]
    w, b = _conv_w(cin, cout, taps, seed=41)
    L = _pack(w, b, tc, "affine")
    x = torch.randn(B * N, cin, device=DEV, generator=torch.Generator(device=DEV).manual_seed(42))
    res = {}
    for j, (kind, relu) in enumerate(POST_VARIANTS):
        scale, shift = _post(cout, kind, seed=43 + j)
        y = run_conv(x, cin, taps, N, L, relu, scale, shift, tc)[:, :cout]
        want, bound = conv_ref(x.double(), w, b, N, relu, scale, shift)
        res["%s-relu%d" % (kind, relu)] = (rel_err(y, want), _elementwise(y.double() - want, bound))
    _record("conv-affine-%s" % mode, res)
    for k, (r, e) in res.items():
        assert r <= TOL[mode] and e <= TOL[mode], (k, r, e)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("taps", [3, 5])
def test_conv1d_padding_columns_and_sequence_boundaries(taps, mode):
    """NaN in the padding columns ld_x > Cin changes no bit and raises no flag; NaN or 1e30 in the last row of one
    sequence and the first row of another changes no bit of the neighbouring sequences (ReLU off: fmaxf would map a
    NaN to 0 by design), so neither a leak across the boundary nor zero padding by multiplication (NaN * 0) passes"""
    B, N, cin, cout = 6, 200, 64, 100
    tc = TC_MODE[mode]
    w, b = _conv_w(cin, cout, taps, seed=51 + taps)
    L = _pack(w, b, tc, "pad%d" % taps)
    M, ld = B * N, cin + 8
    clean = torch.zeros(M, ld, device=DEV)
    clean[:, :cin] = torch.randn(M, cin, device=DEV, generator=torch.Generator(device=DEV).manual_seed(52))
    e2h.check_numeric_range(DEV)
    y0 = run_conv(clean, cin, taps, N, L, False, None, None, tc)
    dirty = clean.clone()
    dirty[:, cin:] = float("nan")
    assert torch.equal(run_conv(dirty, cin, taps, N, L, False, None, None, tc), y0)
    assert e2h.check_numeric_range(DEV)
    want, bound = conv_ref(clean[:, :cin].double(), w, b, N, False, None, None)
    assert _elementwise(y0[:, :cout].double() - want, bound) <= TOL[mode]
    reach = taps // 2
    for fill in (float("nan"), 1e30):
        x = clean.clone()
        x[3 * N - 1, :cin] = fill                       # last row of sequence 2
        x[4 * N, :cin] = fill                           # first row of sequence 4
        y = run_conv(x, cin, taps, N, L, False, None, None, tc)
        e2h.check_numeric_range(DEV)                    # 1e30 leaves the fp16 range: the flag may be raised, reset it
        touched = torch.zeros(M, dtype=torch.bool, device=DEV)
        touched[3 * N - 1 - reach:3 * N] = True
        touched[4 * N:4 * N + 1 + reach] = True
        assert torch.equal(y[~touched], y0[~touched]), fill
        assert torch.equal(y[3 * N:4 * N], y0[3 * N:4 * N]), fill        # sequence 3, between the two poisoned rows


@pytest.mark.parametrize("mode", MODES)
def test_conv1d_sequence_alone_equals_in_batch(mode):
    """a row's product does not depend on its tile position: each sequence alone equals, bit for bit, the same
    sequence inside the batch (its first row at tile offsets 0, 72, 16, 88, 32)"""
    B, N, cin, cout, taps = 5, 200, 256, 100, 3
    tc = TC_MODE[mode]
    w, b = _conv_w(cin, cout, taps, seed=61)
    L = _pack(w, b, tc, "alone")
    scale, shift = _post(cout, "both", seed=62)
    x = torch.randn(B * N, cin, device=DEV, generator=torch.Generator(device=DEV).manual_seed(63))
    y = run_conv(x, cin, taps, N, L, True, scale, shift, tc)
    for s in range(B):
        alone = run_conv(x[s * N:(s + 1) * N], cin, taps, N, L, True, scale, shift, tc)
        assert torch.equal(alone, y[s * N:(s + 1) * N]), s


@pytest.mark.parametrize("col", [0, 3, 4])
def test_conv1d_output_columns(col):
    """the header's output-column contract: the Cout results at y_col_off, exact +0.0 in the padding columns up to
    the accumulator block width (as far as ld_y allows), every other column untouched"""
    B, N, cin, taps = 3, 200, 64, 3
    for cout in (4, 100, 256):
        w, b = _conv_w(cin, cout, taps, seed=70 + cout)
        x = torch.randn(B * N, cin, device=DEV, generator=torch.Generator(device=DEV).manual_seed(71))
        want, _ = conv_ref(x.double(), w, b, N, True, None, None)
        ld_y = col + cout + 40
        end = col + min(ld_y - col, _padded_width(cout))
        for mode in MODES:
            tc = TC_MODE[mode]
            L = _pack(w, b, tc, "cols%d" % cout)
            y = torch.full((B * N, ld_y), 777.0, device=DEV)
            run_conv(x, cin, taps, N, L, True, None, None, tc, y=y, col=col)
            assert rel_err(y[:, col:col + cout], want) <= TOL[mode], (cout, mode)
            pad = y[:, col + cout:end]
            assert (pad == 0).all() and not torch.signbit(pad).any(), (cout, mode)
            assert (y[:, :col] == 777.0).all() and (y[:, end:] == 777.0).all(), (cout, mode)


def test_per_layer_outputs_to_unaligned_views():
    """y may be any float-aligned view (a storage offset, a column slice): the vector stores of ev2h_conv1d_tc,
    ev2h_linear_tc, ev2h_linear_relu_tc and the exact fp32 ev2h_linear_f32 / ev2h_linear_relu_f32 fall back to
    scalar stores there, and write the same bits as into an aligned buffer"""
    if not _lib_fixed_unaligned():
        pytest.skip("library older than ABI 102: unaligned outputs would meet float4 stores")
    B, N, cin, cout = 2, 300, 64, 100
    M, ld_y = B * N, pu._pad4(cout)
    w, b = _conv_w(cin, cout, 3, seed=81)
    x = torch.randn(M, cin, device=DEV, generator=torch.Generator(device=DEV).manual_seed(82))
    w1, b1 = _conv_w(cin, cout, 1, seed=83)
    wt = torch.zeros(((cin + 15) // 16 * 16, 128), device=DEV)
    wt[:cin, :cout] = w1[:, :, 0].t().float()
    bias = torch.zeros(128, device=DEV)
    bias[:cout] = b1.float()
    for mode in MODES:
        tc = TC_MODE[mode]
        L3, L1 = _pack(w, b, tc, "unal3"), _pack(w1, b1, tc, "unal1")
        for fn in ("conv1d", "linear_tc", "linear_relu_tc"):
            outs = []
            for y in (torch.zeros(M, ld_y, device=DEV), _unaligned_view((M, ld_y))):
                if fn == "conv1d":
                    run_conv(x, cin, 3, N, L3, True, None, None, tc, y=y)
                elif fn == "linear_tc":
                    _capi.linear_tc_no_relu(x, M, cin, cin, L1["packed"], L1["bias"], cout, y, ld_y, 0, tc)
                else:
                    _capi.linear_relu_tc(x, M, cin, cin, L1["packed"], L1["bias"], cout, 0, y, ld_y, 0, tc)
                torch.cuda.synchronize()
                outs.append(y.clone())
            assert torch.equal(outs[0], outs[1]), (fn, mode)
    for relu in (True, False):
        outs = []
        for y in (torch.zeros(M, ld_y, device=DEV), _unaligned_view((M, ld_y))):
            if relu:
                _capi.linear_relu(x, M, cin, cin, wt, bias, cout, 0, y, ld_y)
            else:
                _capi.linear_no_relu(x, M, cin, cin, wt, bias, cout, y, ld_y)
            torch.cuda.synchronize()
            outs.append(y.clone())
        assert torch.equal(outs[0], outs[1]), relu
        want = x.double() @ w1[:, :, 0].t() + b1
        assert rel_err(outs[0][:, :cout], torch.relu(want) if relu else want) <= 1e-5


# ================================================================== B. ev2h_class_attention_f32 ====================
ATTN_SHAPES = [(1, 1, 4, 256), (2, 5, 4, 64), (3, 7, 1, 32), (2, 8, 8, 1024), (2, 9, 3, 96), (1, 63, 4, 256),
               (1, 65, 4, 256), (64, 2048, 4, 256), (4, 16384, 4, 256)]


def attn_inputs(B, N, C, D, seed, ld_k=None, ld_q=None, key_scale=1.0, equal_keys=False):
    """key [B*N, ld_k], query and value [B*N, ld_q]; columns past C / D hold NaN"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    ld_k, ld_q = ld_k or C, ld_q or D
    key = torch.full((B * N, ld_k), float("nan"), device=DEV)
    k = torch.randn(B * N, 1 if equal_keys else C, device=DEV, generator=g) * key_scale
    key[:, :C] = k.expand(B * N, C)
    q = torch.full((B * N, ld_q), float("nan"), device=DEV)
    v = torch.full((B * N, ld_q), float("nan"), device=DEV)
    q[:, :D] = torch.randn(B * N, D, device=DEV, generator=g)
    v[:, :D] = torch.randn(B * N, D, device=DEV, generator=g)
    return key, q, v


def attn_ref(key, q, v, B, N, C, D, scale):
    """float64 attention -> (context [B, C, N], first-order bound of the exact fp32 kernel's error, sim [B, C, D]).

    sim: a chain of ceil(N/8) fmaf per split, 8 partials summed, one product by scale: gamma(ceil(N/8) + 9) of
    scale * sum |k||q|.  Softmax: a perturbation ds_c of the logits moves w_c by at most (ds_c + sum_j w_j ds_j) w_c;
    fp32 adds u |s_c - max| (the subtraction), 2 ulp of expf (4u), the C-term denominator and the division.
    Context: a chain of D/32 fmaf per lane and 5 shuffle additions: gamma(D/32 + 5) of sum_d w |v|."""
    k = key[:, :C].double().view(B, N, C)
    qq = q[:, :D].double().view(B, N, D)
    vv = v[:, :D].double().view(B, N, D)
    s = scale * torch.einsum("bnc,bnd->bcd", k, qq)
    ds = (math.ceil(N / 8) + 9) * U * scale * torch.einsum("bnc,bnd->bcd", k.abs(), qq.abs())
    w = torch.softmax(s, dim=1)
    gap = (s - s.amax(1, keepdim=True)).abs()
    e = U * gap + 4 * U                                             # per-term error of exp(s - max)
    eps_w = ds + (w * ds).sum(1, keepdim=True) + e + (w * e).sum(1, keepdim=True) + C * U
    ctx = torch.einsum("bcd,bnd->bcn", w, vv)
    bound = torch.einsum("bcd,bnd->bcn", (eps_w + (D // 32 + 5) * U) * w, vv.abs())
    return ctx, bound, s


def run_attn(key, q, v, B, N, C, D, scale):
    out = _capi.class_attention(key, key.shape[1], q, q.shape[1], v, v.shape[1], B, N, C, D, scale)
    torch.cuda.synchronize()
    return out


def _scale32(D):
    return float(np.float32(D ** -0.5))        # the kernel takes the scale as fp32: the reference uses that value


@pytest.mark.parametrize("shape", ATTN_SHAPES, ids=lambda s: "B%d-N%d-C%d-D%d" % s)
def test_class_attention_vs_f64(shape):
    B, N, C, D = shape
    res = {}
    for variant in ("dense", "padded", "ld_k8", "large"):
        ld_k = 8 if variant == "ld_k8" else (C if variant != "padded" else C + 1)
        ld_q = D + 4 if variant in ("padded", "ld_k8") else D
        key, q, v = attn_inputs(B, N, C, D, seed=sum(shape), ld_k=ld_k, ld_q=ld_q)
        if variant == "large":                          # logits of ~1e3: exp without the max subtraction overflows
            _, _, s = attn_ref(key, q, v, B, N, C, D, _scale32(D))
            key = key * (1e3 / float(s.abs().max()))
        out = run_attn(key, q, v, B, N, C, D, _scale32(D))
        ctx, bound, s = attn_ref(key, q, v, B, N, C, D, _scale32(D))
        assert torch.isfinite(out).all(), variant
        if variant == "large":
            assert float(s.abs().max()) >= 999.0
        res[variant] = _elementwise(out.double() - ctx, bound)
    _record("attn-B%d-N%d-C%d-D%d" % shape, res)
    for k, r in res.items():
        assert r <= 1.0, (k, r)


@pytest.mark.parametrize("C", [3, 4, 8])
def test_class_attention_equal_keys(C):
    """identical logits for every class: each softmax weight is exactly fl(1/C), so every class row of the context
    is the same bits"""
    B, N, D = 2, 300, 256
    key, q, v = attn_inputs(B, N, C, D, seed=C, equal_keys=True)
    out = run_attn(key, q, v, B, N, C, D, _scale32(D))
    for c in range(1, C):
        assert torch.equal(out[:, c], out[:, 0]), c
    ctx, bound, _ = attn_ref(key, q, v, B, N, C, D, _scale32(D))
    assert _elementwise(out.double() - ctx, bound) <= 1.0
    want = v[:, :D].double().view(B, N, D).sum(-1) / C   # weights 1/C: the context is the sum over d of v, over C
    assert rel_err(out[:, 0], want) <= 1e-5


def test_class_attention_batch_repeat_and_limits():
    """a batch of 3 windows equals each window run alone bit for bit, a repeat run is bitwise equal, and shapes the
    kernel does not cover (C = 9, D not a multiple of 32, D > 1024) raise instead of launching"""
    B, N, C, D = 3, 200, 4, 256
    key, q, v = attn_inputs(B, N, C, D, seed=91)
    out = run_attn(key, q, v, B, N, C, D, _scale32(D))
    assert torch.equal(run_attn(key, q, v, B, N, C, D, _scale32(D)), out)
    for b in range(B):
        sl = slice(b * N, (b + 1) * N)
        assert torch.equal(run_attn(key[sl], q[sl], v[sl], 1, N, C, D, _scale32(D))[0], out[b]), b
    for (c, d) in ((9, 64), (4, 48), (4, 1056)):
        k2, q2, v2 = attn_inputs(1, 16, c, d, seed=92)
        with pytest.raises(RuntimeError):
            run_attn(k2, q2, v2, 1, 16, c, d, _scale32(d))


# ================================================================== C. three_nn / three_interp =====================
NN_SHAPES = {"s3-n1": (1, 1, 3), "s3-n5": (2, 5, 3), "s1024": (2, 777, 1024), "s1025-tie": (2, 777, 1025),
             "n4097-s2049": (1, 4097, 2049), "n16384": (4, 16384, 512), "b64": (64, 2048, 512)}
NN_INPUTS = ("random", "identical", "on-sources", "offset", "strided")


def _nn_points(name, inputs):
    B, N, S = NN_SHAPES[name]
    rs = np.random.RandomState(sum(map(ord, name + inputs)))
    q = rs.rand(B, N, 3).astype(np.float32)
    s = rs.rand(B, S, 3).astype(np.float32)
    if name == "s1025-tie":
        s[:, 1024] = s[:, 1023]                          # equal sources on both sides of the 1024-source tile edge
        q[:, :4] = s[:, 1021:1025]                       # and queries for which they are among the three nearest
    if inputs == "identical":
        s[:] = s[:, :1]
    elif inputs == "on-sources":
        m = min(N, S)
        q[:, :m] = s[:, rs.permutation(S)[:m]]
    elif inputs == "offset":
        q += np.float32(1e3)
        s += np.float32(1e3)
    return q, s


def _nn_device(q, s, strided):
    """channel-first [B,3,*] device views: contiguous, or a channel slice of a wider tensor and a transposed view"""
    if not strided:
        return (torch.from_numpy(np.ascontiguousarray(q.transpose(0, 2, 1))).to(DEV),
                torch.from_numpy(np.ascontiguousarray(s.transpose(0, 2, 1))).to(DEV))
    B, N, _ = q.shape
    wide = torch.zeros(B, 6, N, device=DEV)
    wide[:, 1:4] = torch.from_numpy(q).to(DEV).permute(0, 2, 1)
    return wide[:, 1:4], torch.from_numpy(s).to(DEV).permute(0, 2, 1)


def _fma32(a, b, c):
    """fmaf(a, b, c) on float32 arrays, correctly rounded: the product is exact in float64, TwoSum gives the exact
    remainder of the float64 sum, and a sum that lands on a float32 midpoint is rounded by the remainder's sign"""
    f32, f64 = np.float32, np.float64
    p, cc = a.astype(f64) * b.astype(f64), c.astype(f64)
    s = p + cc
    bb = s - p
    e = (p - (s - bb)) + (cc - bb)
    r = s.astype(f32)
    nb = np.nextafter(r, np.where(s > r.astype(f64), f32(np.inf), f32(-np.inf)).astype(f32))
    tie = (s == (r.astype(f64) + nb.astype(f64)) / 2) & (e != 0)
    return np.where(tie, np.where(e > 0, np.maximum(r, nb), np.minimum(r, nb)), r)


def sqdist_f32(q, s):
    """[B,N,3], [B,S,3] float32 -> [B,N,S]: the expanded distance -2 q.p + |q|^2 + |p|^2 in the kernel's float32
    operation order (geom.cuh: x*x', two fmaf, then the two additions one after the other)"""
    out = np.empty((q.shape[0], q.shape[1], s.shape[1]), np.float32)
    for b in range(q.shape[0]):
        qb, sb = q[b][:, None, :], s[b][None, :, :]
        dot = (qb[..., 0].astype(np.float64) * sb[..., 0]).astype(np.float32)
        dot = _fma32(qb[..., 1], sb[..., 1], dot)
        dot = _fma32(qb[..., 2], sb[..., 2], dot)
        qq = (q[b, :, 0] * q[b, :, 0] + q[b, :, 1] * q[b, :, 1]) + q[b, :, 2] * q[b, :, 2]
        ss = (s[b, :, 0] * s[b, :, 0] + s[b, :, 1] * s[b, :, 1]) + s[b, :, 2] * s[b, :, 2]
        out[b] = (np.float32(-2.0) * dot + qq[:, None]) + ss[None, :]
    return out


def _weights_f32(d3):
    """the kernel's weight arithmetic in NumPy float32: r = 1 / (d + 1e-8), norm = (r0 + r1) + r2, w = r / norm"""
    one, eps = np.float32(1.0), np.float32(1e-8)
    r = one / (d3 + eps)
    norm = (r[..., 0] + r[..., 1]) + r[..., 2]
    return r / norm[..., None]


@pytest.mark.parametrize("inputs", NN_INPUTS)
@pytest.mark.parametrize("name", list(NN_SHAPES))
def test_three_nn_vs_oracle(name, inputs):
    """indices bit-exact against a full stable sort of the expanded fp32 distances, ties resolved to the lower index
    (the kernel's rule: its strict comparison keeps an equal distance found later behind); weights bitwise equal to
    the kernel's float32 arithmetic on those distances (slightly negative for coincident points).  The distances are
    restated in the kernel's operation order: the oracle's torch.matmul rounds them the same way for large matrices
    but not for all shapes (at S = 3, N = 5 it differs by an ulp).  The oracle's own 3-NN must agree wherever its
    distance row is the same bits (exact ties aside: its sort is not stable)."""
    q, s = _nn_points(name, inputs)
    xyz1, xyz2 = _nn_device(q, s, inputs == "strided")
    idx, w = _capi.three_nn(xyz1, xyz2)
    torch.cuda.synchronize()
    gi, gw = idx.cpu().numpy().astype(np.int64), w.cpu().numpy()
    qt, st = torch.from_numpy(q), torch.from_numpy(s)
    dn = sqdist_f32(q, s)
    stable = torch.sort(torch.from_numpy(dn), dim=-1, stable=True).indices[..., :3].numpy()
    assert np.array_equal(gi, stable)
    want_i, _ = sa_oracle.three_nn_weights(qt, st)
    wi = want_i.numpy()
    same_rows = (sa_oracle.pairwise_sqdist(qt, st).numpy() == dn).all(-1)
    differ = (gi != wi) & same_rows[..., None]           # the oracle's unstable sort may order exact ties otherwise
    assert (np.take_along_axis(dn, gi, -1)[differ] == np.take_along_axis(dn, wi, -1)[differ]).all()
    if inputs == "identical":
        assert (gi == np.array([0, 1, 2])).all()
    d3 = np.take_along_axis(dn, gi, -1)
    want_w = _weights_f32(d3)
    assert np.array_equal(gw.view(np.int32), want_w.view(np.int32)), int((gw != want_w).sum())
    _record("nn-%s-%s" % (name, inputs), {"ties": int(differ.sum()), "negative_d": int((d3 < 0).sum()),
                                          "oracle_rows_other_rounding": int((~same_rows).sum())})


# (B, N, S, D, ld_f, col): scalar path for D, ld_f or col not a multiple of 4; the last case is 8.4 M quads on the
# vector path, about 14 passes of the grid-stride loop (the grid is capped at SMs * 16 CTAs)
INTERP_CASES = {"d1": (2, 777, 100, 1, 1, 0), "d3": (2, 777, 100, 3, 3, 0), "d5": (2, 777, 100, 5, 8, 5),
                "d130": (2, 777, 100, 130, 132, 3), "d256-b64": (64, 2048, 512, 256, 256, 0)}


def _interp_setup(B, N, S, D, ld_f, seed):
    rs = np.random.RandomState(seed)
    xyz1 = torch.from_numpy(rs.rand(B, 3, N).astype(np.float32)).to(DEV)
    xyz2 = torch.from_numpy(rs.rand(B, 3, S).astype(np.float32)).to(DEV)
    idx, w = _capi.three_nn(xyz1, xyz2)
    feats = torch.full((B * S, ld_f), float("nan"), device=DEV)
    feats[:, :D] = torch.randn(B * S, D, device=DEV, generator=torch.Generator(device=DEV).manual_seed(seed))
    return idx, w, feats


def _interp_refs(feats, idx, w, B, N, S, D):
    rows = (torch.arange(B, device=DEV).view(B, 1, 1) * S + idx.long()).view(B * N, 3)
    f = [feats[rows[:, k], :D] for k in range(3)]
    wk = [w.view(B * N, 3)[:, k:k + 1] for k in range(3)]
    f32 = (f[0] * wk[0] + f[1] * wk[1]) + f[2] * wk[2]                # three products, two sums, each rounded
    f64 = sum(f[k].double() * wk[k].double() for k in range(3))
    bound = 3 * U * sum(f[k].double().abs() * wk[k].double().abs() for k in range(3))
    return f32, f64, bound


@pytest.mark.parametrize("name", list(INTERP_CASES))
def test_three_interp_vs_f32_and_f64(name):
    """bitwise against float32 (f0 w0 + f1 w1) + f2 w2, within 3u sum |f||w| of float64; NaN in the padding
    columns of feats is never read, and columns of out outside [col, col + D) keep their sentinel"""
    B, N, S, D, ld_f, col = INTERP_CASES[name]
    idx, w, feats = _interp_setup(B, N, S, D, ld_f, seed=D)
    ld_out = pu._pad4(col + D) + 4
    out = torch.full((B * N, ld_out), -5.5, device=DEV)
    _capi.three_interp(feats, ld_f, idx, w, B, N, S, D, out, ld_out, col)
    torch.cuda.synchronize()
    f32, f64, bound = _interp_refs(feats, idx, w, B, N, S, D)
    got = out[:, col:col + D]
    assert torch.equal(got, f32)
    ratio = _elementwise(got.double() - f64, bound)
    _record("interp-" + name, {"elem": ratio})
    assert ratio <= 1.0
    assert (out[:, :col] == -5.5).all() and (out[:, col + D:] == -5.5).all()


def test_three_interp_unaligned_views():
    """feats and out as views one element past a 16-byte boundary: the vector path must step aside (it used to check
    only ld_f, ld_out and col) and the scalar path give the same bits"""
    if not _lib_fixed_unaligned():
        pytest.skip("library older than ABI 102: unaligned views would meet float4 loads and stores")
    B, N, S, D = 2, 777, 100, 256
    idx, w, feats = _interp_setup(B, N, S, D, D, seed=7)
    ref = torch.zeros(B * N, D, device=DEV)
    _capi.three_interp(feats, D, idx, w, B, N, S, D, ref, D, 0)
    f_un = _unaligned_view((B * S, D))
    f_un.copy_(feats)
    for src in (feats, f_un):
        out = _unaligned_view((B * N, D), fill=-5.5)
        _capi.three_interp(src, D, idx, w, B, N, S, D, out, D, 0)
        torch.cuda.synchronize()
        assert torch.equal(out, ref)
    out = torch.zeros(B * N, D, device=DEV)
    _capi.three_interp(f_un, D, idx, w, B, N, S, D, out, D, 0)
    torch.cuda.synchronize()
    assert torch.equal(out, ref)


# ================================================================== D. modules ======================================
def _fp64(mod, points1, points2, idx, weight):
    """float64 PointNetFeaturePropagation on the module's own indices and weights: points1 [B,D1,N] | None and
    points2 [B,D2,S] (any float dtype), idx / weight [B,N,k] -> [B,C',N]"""
    f2 = points2.double().permute(0, 2, 1)
    B, N = idx.shape[:2]
    g = f2[torch.arange(B, device=DEV).view(B, 1, 1), idx.long()]               # [B,N,k,D2]
    h = (g * weight.double().unsqueeze(-1)).sum(2)
    if points1 is not None:
        h = torch.cat([points1.double().permute(0, 2, 1), h], -1)
    for conv, bn in zip(mod.mlp_convs, mod.mlp_bns):
        h = h @ conv.weight.double()[:, :, 0].t() + conv.bias.double()
        h = torch.relu((h - bn.running_mean.double()) / torch.sqrt(bn.running_var.double() + bn.eps) * bn.weight.double()
                       + bn.bias.double())
    return h.permute(0, 2, 1)


def _decoder(seed):
    dec = e2h.FeaturePropagationDecoder()
    for j, n in enumerate(("fp3", "fp2", "fp1")):
        load_numpy_state(getattr(dec, n), synth.random_state_for(synth.DECODER_SPECS[n], seed=seed + j))
    return dec.to(DEV).eval()


_DEC = {}


def _decoder_case(B, N):
    if (B, N) not in _DEC:
        rs = np.random.RandomState(B + N)
        xyz = [torch.from_numpy(rs.rand(B, 3, n).astype(np.float32)).to(DEV) for n in (N, 512, 128, 1)]
        feats = [torch.from_numpy(a).to(DEV) for a in synth.decoder_test_features(B, seed=B + N)]
        _DEC[(B, N)] = (_decoder(B + N), xyz, feats)
    return _DEC[(B, N)]


@pytest.mark.parametrize("mode", MODES + ("fp32",))
@pytest.mark.parametrize("BN", [(64, 2048), (4, 16384)], ids=["B64-N2048", "B4-N16384"])
def test_decoder_vs_f64(BN, mode, monkeypatch):
    """fp3 -> fp2 -> fp1 against a float64 chain of the three modules on their own 3-NN indices and weights"""
    _set_mode(monkeypatch, mode)
    dec, (x0, x1, x2, x3), (f1, f2, f3) = _decoder_case(*BN)
    e2h.check_numeric_range(DEV)
    with torch.no_grad():
        d0, d1, d2 = dec(x0, x1, x2, x3, f1, f2, f3, return_levels=True)
    torch.cuda.synchronize()
    assert mode == "bf16" or e2h.check_numeric_range(DEV)
    r2 = _fp64(dec.fp3, f2, f3, dec.fp3.last_idx, dec.fp3.last_weight)
    r1 = _fp64(dec.fp2, f1, r2, dec.fp2.last_idx, dec.fp2.last_weight)
    r0 = _fp64(dec.fp1, None, r1, dec.fp1.last_idx, dec.fp1.last_weight)
    res = {"fp3": rel_err(d2, r2), "fp2": rel_err(d1, r1), "fp1": rel_err(d0, r0)}
    _record("decoder-B%d-N%d-%s" % (BN + (mode,)), res)
    for k, r in res.items():
        assert r <= TOL[mode], (k, r)


@pytest.mark.parametrize("S", [1, 2, 3, 7, 512])
@pytest.mark.parametrize("D2", [3, 130])
@pytest.mark.parametrize("D1", [0, 5, 64])
def test_feature_propagation_vs_f64(D1, D2, S, monkeypatch):
    """one PointNetFeaturePropagation in every mode; S = 1 repeats the single source, S = 2 takes the autograd
    formulation (two neighbours), compared with a float64 restatement of it on the expanded fp32 distances"""
    B, N = 2, 300
    spec = dict(kind="fp", in_channel=D1 + D2, mlp=[48, 24])
    mod = load_numpy_state(e2h.PointNetFeaturePropagation(D1 + D2, [48, 24]),
                           synth.random_state_for(spec, seed=D1 + D2 + S)).to(DEV).eval()
    rs = np.random.RandomState(D1 * 7 + D2 + S)
    xyz1 = torch.from_numpy(rs.rand(B, 3, N).astype(np.float32)).to(DEV)
    xyz2 = torch.from_numpy(rs.rand(B, 3, S).astype(np.float32)).to(DEV)
    p1 = torch.from_numpy(rs.randn(B, D1, N).astype(np.float32)).to(DEV) if D1 else None
    p2 = torch.from_numpy(rs.randn(B, D2, S).astype(np.float32)).to(DEV)
    if S == 2:
        d = sa_oracle.pairwise_sqdist(xyz1.permute(0, 2, 1).cpu(), xyz2.permute(0, 2, 1).cpu()).to(DEV)
        ds, idx = d.sort(dim=-1)
        r = 1.0 / (ds.double() + 1e-8)
        weight = r / r.sum(-1, keepdim=True)
    res = {}
    for mode in MODES + ("fp32",):
        _set_mode(monkeypatch, mode)
        if hasattr(mod, "last_idx"):
            del mod.last_idx, mod.last_weight
        with torch.no_grad():
            got = mod(xyz1, xyz2, p1, p2)
        if S != 2:
            idx, weight = mod.last_idx, mod.last_weight
        res[mode] = rel_err(got, _fp64(mod, p1, p2, idx, weight))
    _record("fp-D1%d-D2%d-S%d" % (D1, D2, S), res)
    for mode, r in res.items():
        assert r <= TOL[mode], (mode, r)


def _heads_net(C, seed, monkeypatch):
    """TEHNet with random head weights; some BatchNorm gammas negative, one running variance 1e-3"""
    monkeypatch.setenv("ERPC", "1")
    st = synth.random_head_state(seed=seed, num_classes=C)
    for name in ("classifier.2", "left_query_conv.2", "right_query_conv.5"):
        st[name + ".weight"][::3] *= -1
    st["left_query_conv.2.running_var"][7] = 1e-3
    net = tehnet.TEHNet(n_pose_params=6, num_classes=C)
    res = net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in st.items()}, strict=False)
    assert not res.unexpected_keys
    return net.to(DEV).eval()


def heads64(net, l0):
    """float64 classifier, query convolutions and AttentionBlock (eval BatchNorm, Dropout the identity)"""
    def bn(h, m):
        sh = (1, -1, 1)
        return ((h - m.running_mean.double().view(sh)) / torch.sqrt(m.running_var.double().view(sh) + m.eps)
                * m.weight.double().view(sh) + m.bias.double().view(sh))

    def conv(h, m):
        return F.conv1d(h, m.weight.double(), m.bias.double(), padding=m.padding)

    x = l0.double()
    c = net.classifier
    logits = conv(bn(torch.relu(conv(x, c[0])), c[2]), c[4])
    D = x.shape[1]
    out = [logits]
    for seq in (net.left_query_conv, net.right_query_conv):
        q = bn(conv(bn(torch.relu(conv(x, seq[0])), seq[2]), seq[4]), seq[5])
        sim = torch.bmm(logits, q.permute(0, 2, 1)) * D ** -0.5
        out.append(torch.bmm(torch.softmax(sim, 1), x))
    return out


HEAD_CASES = [(4, 64, 2048), (4, 2, 16384), (5, 3, 200), (5, 4, 3), (8, 7, 1), (8, 3, 2048)]


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("case", HEAD_CASES, ids=lambda c: "C%d-B%d-N%d" % c)
def test_heads_vs_f64(case, mode, monkeypatch):
    """TEHNet._heads_cuda (classifier, both query convolutions, both attentions) against float64 on sampled windows"""
    C, B, N = case
    _set_mode(monkeypatch, mode)
    net = _heads_net(C, seed=C * 10 + B, monkeypatch=monkeypatch)
    l0 = torch.randn(B, 256, N, device=DEV, generator=torch.Generator(device=DEV).manual_seed(B * N + C))
    e2h.check_numeric_range(DEV)
    with torch.no_grad():
        got = net._heads_cuda(l0)
    torch.cuda.synchronize()
    assert mode == "bf16" or e2h.check_numeric_range(DEV)
    win = sorted({0, B // 2, B - 1})
    want = heads64(net, l0[win])
    res = {k: rel_err(g[win], w) for k, g, w in zip(("seg", "left", "right"), got, want)}
    _record("heads-C%d-B%d-N%d-%s" % (case + (mode,)), res)
    # the attention's logits are sums over the window's N points: their error, made of N independent roundings of
    # the convolutions' outputs, grows like sqrt(N), and so does the context's.  The bar is the per-tensor one up to
    # the model's 2048 points and grows with sqrt(N / 2048) beyond (measured on a B200 at N = 16384: 1.7e-5 in the
    # fp32-level modes, 1.1e-2 in bf16, where N = 2048 gives up to 8.0e-6 and 3.3e-3)
    bar = TOL[mode] * max(1.0, (N / 2048) ** 0.5)
    for k, r in res.items():
        assert r <= bar, (k, r)


def test_heads_cache_follows_in_place_changes(monkeypatch):
    """the folded head weights are rebuilt when a BatchNorm buffer changes in place (_HeadWeights' key), and a
    decoder output changed in place after the decoder wrote it is read as changed (the rows it carries are only
    reused while the tensor's version is the one the decoder left)"""
    _set_mode(monkeypatch, "f16")
    net = _heads_net(4, seed=5, monkeypatch=monkeypatch)
    B, N = 2, 300
    l0 = torch.randn(B, 256, N, device=DEV, generator=torch.Generator(device=DEV).manual_seed(6))
    with torch.no_grad():
        seg0, left0, right0 = net._heads_cuda(l0)
        net.left_query_conv[2].running_mean.add_(0.5)
        net.classifier[2].running_var.mul_(2.0)
        seg1, left1, right1 = net._heads_cuda(l0)
    want = heads64(net, l0)
    assert not torch.equal(seg1, seg0) and not torch.equal(left1, left0)
    for g, w in zip((seg1, left1, right1), want):
        assert rel_err(g, w) <= 1e-5

    dec, (x0, x1, x2, x3), (f1, f2, f3) = _decoder_case(2, 2048)
    with torch.no_grad():
        d0 = dec(x0, x1, x2, x3, f1, f2, f3)
        assert getattr(d0, "_ev2h_fp_rows", None) is not None
        before = net._heads_cuda(d0)
        d0.mul_(-1.5)
        after = net._heads_cuda(d0)
        fresh = net._heads_cuda(d0.clone())
    for a, f, b in zip(after, fresh, before):
        assert torch.equal(a, f) and not torch.equal(a, b)
    for g, w in zip(after, heads64(net, d0)):
        assert rel_err(g, w) <= 1e-5
