"""Envelope of the tensor-core MLP kernels against a float64 restatement of the same operations.

The fused grouping + MLP + max-pool kernel (sa_fused_tc.cu) serves every scale ``_capi.fused_supported`` accepts, not
just the model's layer shapes: the cases below reach its layer-width paddings, partially used 128-lane blocks, the
512-TMEM-column extreme, partial last tiles, gather and per-point layer 1, D = 0 and modules that mix fused and
unfused scales, in every fp32-level split (fp16 pairs, tf32 + bf16 corrections, three tf32 products) and in bf16.
The per-layer kernel (linear_tc.cu) is checked for its contract: the fp16-split range flag on every entry, padding
columns that never enter the product, and weights outside the fp16 range.

Bars are those of the parity suite: 1e-5 of max|reference| per tensor for the fp32-level modes, 1e-2 for bf16."""
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
BN_EPS = 1e-5
# arithmetic of the shared MLP: fp16 split (default), tf32 + two bf16 corrections, three tf32 products, bf16
MODES = ("f16", "tf32", "pure", "bf16")
TOL = {"f16": 1e-5, "tf32": 1e-5, "pure": 1e-5, "bf16": 1e-2}


def rel_err(got, want):
    got = got.detach().cpu().double() if torch.is_tensor(got) else torch.as_tensor(got, dtype=torch.float64)
    want = want.detach().cpu().double() if torch.is_tensor(want) else torch.as_tensor(want, dtype=torch.float64)
    return float((got - want).abs().max() / max(float(want.abs().max()), 1e-30))


def _set_mode(monkeypatch, mode):
    """module globals, not environment variables: several knobs are read once into C statics"""
    monkeypatch.setattr(pu, "_mlp_precision", "bf16" if mode == "bf16" else "tf32x3")
    monkeypatch.setattr(pu, "_SPLIT", "tf32" if mode == "tf32" else "f16")
    monkeypatch.setattr(pu, "_TF32X3_PURE", mode == "pure")
    for name, value in (("_FUSED_ENABLED", True), ("_COMPACT", True), ("_DEDUP", True), ("_LINEAR_MIXED", True),
                        ("_PER_POINT_ALWAYS", False), ("_FPS_SPLITS", 0), ("_SCALE_STREAMS", False)):
        monkeypatch.setattr(pu, name, value)


# ------------------------------------------------------------------ float64 reference ------------------------------
def _layers64(state, i, n):
    out = []
    for j in range(n):
        c, b = "conv_blocks.%d.%d" % (i, j), "bn_blocks.%d.%d" % (i, j)
        w = state[c + ".weight"]
        out.append(tuple(torch.from_numpy(np.asarray(t, dtype=np.float64)) for t in (
            w.reshape(w.shape[0], -1), state[c + ".bias"], state[b + ".weight"], state[b + ".bias"],
            state[b + ".running_mean"], state[b + ".running_var"])))
    return out


def sa_msg_f64(state, mlp_list, nsample_list, xyz_cf, feats_cf, fps_idx, ball_idx):
    """PointNetSetAbstractionMsg's MLP + max over K in float64 on given indices (index parity is pinned elsewhere, so
    reusing the module's own isolates the MLP).  xyz_cf [B,3,N], feats_cf [B,D,N] | None: CPU float32;
    fps_idx [B,S], ball_idx [B,S,sum K] -> float64 [B, sum C', S]."""
    xyz = xyz_cf.permute(0, 2, 1)
    feats = None if feats_cf is None else feats_cf.permute(0, 2, 1)
    B, S = fps_idx.shape
    fps_idx, ball_idx = fps_idx.long(), ball_idx.long()
    pooled, k_off = [], 0
    for i, K in enumerate(nsample_list):
        layers = _layers64(state, i, len(mlp_list[i]))
        per_window = []
        for b in range(B):
            idx = ball_idx[b, :, k_off:k_off + K]                                   # [S, K]
            rel = (xyz[b][idx] - xyz[b][fps_idx[b]].view(S, 1, 3)).double()         # the subtraction in fp32, as the reference
            h = rel if feats is None else torch.cat([feats[b][idx].double(), rel], -1)
            for (w, bias, gamma, beta, mean, var) in layers:
                h = torch.relu((h @ w.t() + bias - mean) / torch.sqrt(var + BN_EPS) * gamma + beta)
            per_window.append(h.max(dim=1).values.t())                               # [C', S]
        pooled.append(torch.stack(per_window))
        k_off += K
    return torch.cat(pooled, 1)


def test_f64_helper_agrees_with_the_pinned_oracle():
    """the float64 helper restates oracle.sa_oracle.sa_msg_forward (fp32, pinned to the reference's goldens)"""
    spec = dict(kind="msg", npoint=37, radius_list=[0.2, 0.4], nsample_list=[32, 64], in_channel=5,
                mlp_list=[[24, 40, 72], [32, 128, 129]])
    state = synth.random_state_for(spec, seed=5)
    ev = torch.from_numpy(synth.make_windows(2, 777, seed=3))
    start = torch.from_numpy(synth.make_start_indices(2, 777, 1))
    with torch.no_grad():
        _, want, aux = sa_oracle.sa_msg_forward(state, spec, ev[:, :3], ev, start, return_aux=True)
    got = sa_msg_f64(state, spec["mlp_list"], spec["nsample_list"], ev[:, :3], ev, aux["fps_idx"], torch.cat(aux["ball_idx"], -1))
    assert rel_err(want, got) <= 1e-5


# ------------------------------------------------------------------ A. the fused kernel's envelope -----------------
# D input features (0: points = None), neighbours K and widths per scale, geometry.  Gather mode (D + 3 <= 8, layer 1
# in the loader warps) for g*, per-point mode (layer 1 once per point) for p*; the comment names what the case reaches
# in fused_plan (sa_fused_tc.cu).  B * S * K is not a multiple of 128 wherever K < 128 (partial last tile).
CASES = {
    # single tile (96 rows); D = 0; layer 3 uses 16 of one 128-lane block
    "g1": dict(D=0, K=[32], mlp=[[16, 16, 16]], B=1, N=777, S=3, r=[0.3]),
    # layer 1 ends mid-chunk; layer 2 padded 40 -> 48 (column mask); two CTAs per SM; window 1 is one point repeated
    "g2": dict(D=5, K=[32], mlp=[[24, 40, 72]], B=3, N=2048, S=37, r=[0.3], same=1),
    # gather layer 1 at its 128 maximum, layer 2 = 256, one CTA per SM; the radius holds the whole window
    "g3": dict(D=2, K=[64], mlp=[[128, 256, 128]], B=3, N=2048, S=37, r=[5.0]),
    # layer 2 padded 200 -> 208 / 224; layer 3 in two 128-lane blocks
    "g4": dict(D=4, K=[128], mlp=[[64, 200, 256]], B=2, N=2048, S=64, r=[0.4]),
    # the second layer-3 block holds one channel; the radius holds the centre (and its exact copies) only: distinct
    # points lie >= 2/346 apart, and the expanded distance of a point to itself rounds to up to ~1e-6 (so r = 1e-4
    # would leave balls empty, which the reference's own indexing cannot take)
    "g5": dict(D=5, K=[64], mlp=[[32, 128, 129]], B=3, N=777, S=37, r=[3e-3]),
    # 512 TMEM columns; long windows
    "g6": dict(D=1, K=[128], mlp=[[48, 256, 256]], B=2, N=16384, S=40, r=[0.2]),
    # tiny layers 1-2, wide layer 3; many tiles per CTA
    "g7": dict(D=3, K=[32], mlp=[[8, 16, 256]], B=8, N=2048, S=512, r=[0.3]),
    "p1": dict(D=6, K=[32], mlp=[[32, 32, 32]], B=3, N=2048, S=37, r=[0.3]),           # per point, two CTAs per SM
    "p2": dict(D=61, K=[64], mlp=[[256, 64, 200]], B=3, N=777, S=37, r=[0.4]),         # per-point layer 1 at 256
    "p3": dict(D=320, K=[128], mlp=[[96, 176, 256]], B=2, N=1024, S=64, r=[0.8]),      # sa2-like input, other widths
    "p4": dict(D=29, K=[32], mlp=[[160, 256, 256]], B=3, N=2048, S=37, r=[0.2]),       # per point at 512 columns
    # three scales, the K = 16 one not fused: k_off, output columns and P-table columns across fused and unfused scales
    "mix-g": dict(D=5, K=[32, 16, 128], mlp=[[24, 40, 72], [32, 32, 64], [64, 200, 256]], B=3, N=2048, S=37, r=[0.2, 0.1, 0.4]),
    "mix-p": dict(D=61, K=[32, 16, 128], mlp=[[32, 40, 72], [32, 32, 64], [64, 200, 256]], B=3, N=777, S=37, r=[0.2, 0.1, 0.4]),
    # outside the envelope (K = 16; gather layer 1 > 128; per-point layer 1 not a multiple of 32; a width > 256):
    # never fused, the layer-by-layer path meets the same bars
    "out-g": dict(D=5, K=[16, 32, 32], mlp=[[32, 32, 64], [144, 64, 64], [64, 64, 257]], B=3, N=777, S=37, r=[0.2, 0.3, 0.4]),
    "out-p": dict(D=20, K=[32], mlp=[[48, 64, 64]], B=3, N=777, S=37, r=[0.3]),
}


def _expected_fused(name):
    return [not name.startswith("out") and k != 16 for k in CASES[name]["K"]]


_CACHE = {}


def _case(name):
    """module (random weights and BatchNorm statistics), inputs, and the fp64 reference on the module's indices,
    built once per case and shared by every mode (the indices do not depend on the MLP's arithmetic)"""
    if name in _CACHE:
        return _CACHE[name]
    c = CASES[name]
    seed = sum(map(ord, name))
    B, N, S, D = c["B"], c["N"], c["S"], c["D"]
    ev = synth.make_windows(B, N, seed=seed)
    if "same" in c:
        ev[c["same"]] = ev[c["same"]][:, :1]                     # every point (and its features) identical
    xyz = torch.from_numpy(np.ascontiguousarray(ev[:, :3]))
    if D == 0:
        feats = None
    elif D <= 5:
        feats = torch.from_numpy(np.ascontiguousarray(ev[:, :D]))
    else:
        feats = torch.from_numpy(np.random.RandomState(seed).randn(B, D, N).astype(np.float32))
    n = len(c["K"])
    state = synth.random_sa_state("conv_blocks.{i}.{j}", "bn_blocks.{i}.{j}", c["mlp"], [D + 3] * n, seed)
    mod = e2h.PointNetSetAbstractionMsg(S, c["r"], c["K"], D, c["mlp"])
    mod = load_numpy_state(mod, state).to(DEV).eval()
    start = torch.from_numpy(synth.make_start_indices(B, N, seed))
    xyz_d = xyz.to(DEV)
    feats_d = None if feats is None else feats.to(DEV)
    with torch.no_grad():
        mod.forward_rows(xyz_d, feats_d, fps_start=start)
    fps_idx, ball_idx = mod.last_fps_idx.cpu(), mod.last_ball_idx.cpu()
    ref = sa_msg_f64(state, c["mlp"], c["K"], xyz, feats, fps_idx, ball_idx)
    _CACHE[name] = dict(mod=mod, xyz=xyz_d, feats=feats_d, start=start, fps_idx=fps_idx, ball_idx=ball_idx, ref=ref)
    return _CACHE[name]


def _forward_rows(case):
    with torch.no_grad():
        _, rec = case["mod"].forward_rows(case["xyz"], case["feats"], fps_start=case["start"])
    torch.cuda.synchronize()
    return rec


def _spy_fused(monkeypatch):
    """(k_off, K, out_col) of every sa_msg_fused launch (cf. tools/fused_trace.py)"""
    calls = []
    real = _capi.sa_msg_fused

    def spy(*args, **kw):
        calls.append((args[1], args[6], args[23]))
        return real(*args, **kw)
    monkeypatch.setattr(_capi, "sa_msg_fused", spy)
    return calls


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("name", list(CASES))
def test_fused_envelope_vs_f64(name, mode, monkeypatch):
    _set_mode(monkeypatch, mode)
    c = CASES[name]
    case = _case(name)
    mod, D = case["mod"], c["D"]
    calls = _spy_fused(monkeypatch)
    e2h.check_numeric_range(DEV)                                              # clear
    rec = _forward_rows(case)
    assert torch.equal(mod.last_fps_idx.cpu(), case["fps_idx"]) and torch.equal(mod.last_ball_idx.cpu(), case["ball_idx"])

    # 1. the fused kernel runs exactly the scales fused_supported accepts - and those are the ones the table expects
    fmode = pu._fused_mode(_capi.TC_BF16 if mode == "bf16" else _capi.TC_TF32X3)
    predicted = [_capi.fused_supported(k, w, D + 3, D + 3 > 8, fmode) for k, w in zip(c["K"], c["mlp"])]
    assert predicted == _expected_fused(name)
    k_offs = np.cumsum([0] + c["K"])[:-1].tolist()
    cols = np.cumsum([0] + [w[-1] for w in c["mlp"]])[:-1].tolist()
    want_calls = [(k_offs[i], c["K"][i], cols[i]) for i, f in enumerate(predicted) if f]
    assert sorted(calls) == want_calls

    # 2. features within the bar of the fp64 reference
    c_out = rec.c
    got = rec.rows[:, :, :c_out].permute(0, 2, 1)
    assert c_out == sum(w[-1] for w in c["mlp"])
    assert rel_err(got, case["ref"]) <= TOL[mode], mode

    # 4. the centre-xyz columns hold the centres bit for bit, the padding columns stay 0
    xyz_rows = case["xyz"].permute(0, 2, 1)
    centres = torch.gather(xyz_rows, 1, mod.last_fps_idx.long().unsqueeze(-1).expand(-1, -1, 3))
    assert torch.equal(rec.rows[:, :, c_out:c_out + 3], centres)
    assert (rec.rows[:, :, c_out + 3:] == 0).all()

    # 5. in range: no padded TMEM column, zero row or padding lane may trip the flag
    assert e2h.check_numeric_range(DEV)

    # 3. compacted rows, dense rows, compaction without de-duplication and a second identical run: bit for bit
    if mode == "f16":
        base = rec.rows.clone()
        assert torch.equal(_forward_rows(case).rows, base)
        monkeypatch.setattr(pu, "_COMPACT", False)
        assert torch.equal(_forward_rows(case).rows, base), "dense rows"
        monkeypatch.setattr(pu, "_COMPACT", True)
        monkeypatch.setattr(pu, "_DEDUP", False)
        assert torch.equal(_forward_rows(case).rows, base), "compaction without de-duplication"
        assert e2h.check_numeric_range(DEV)


# ------------------------------------------------------------------ B. the per-layer kernel's contract -------------
TC_MODES = {"bf16": _capi.TC_BF16, "tf32x3": _capi.TC_TF32X3, "tf32_bf16c": _capi.TC_TF32_BF16C, "f16x3": _capi.TC_F16X3}
# entry -> (taps, relu, pool_rows)
ENTRIES = {"linear_tc": (1, False, 0), "linear_relu_tc": (1, True, 0), "linear_relu_tc_pool128": (1, True, 128),
           "conv1d_tc_k1": (1, True, 0), "conv1d_tc_k3": (3, True, 0), "conv1d_tc_k5": (5, True, 0)}


def _tol(tc_mode):
    return 1e-2 if tc_mode == _capi.TC_BF16 else 1e-5


def _conv_weights(cin, cout, taps, seed):
    """fp32-representable Conv1d weights [Cout, Cin, T] and bias, as float64"""
    g = torch.Generator().manual_seed(seed)
    w = (torch.randn(cout, cin, taps, generator=g) / (cin * taps) ** 0.5).double()
    b = (0.1 * torch.randn(cout, generator=g)).double()
    return w, b


def _run_entry(entry, x, cin, L, tc_mode, rows_per_seq):
    """one per-layer tensor-core entry on rows x [M, ld_x] (device) -> y"""
    taps, relu, pool = ENTRIES[entry]
    M, ld = x.shape
    cout = L["cout"]
    y = torch.zeros((M // pool if pool else M, cout), dtype=torch.float32, device=DEV)
    if entry == "linear_tc":
        _capi.linear_tc_no_relu(x, M, ld, cin, L["packed"], L["bias"], cout, y, cout, 0, tc_mode)
    elif entry.startswith("linear_relu_tc"):
        _capi.linear_relu_tc(x, M, ld, cin, L["packed"], L["bias"], cout, pool, y, cout, 0, tc_mode)
    else:
        _capi.conv1d_tc(x, M, ld, cin, taps, rows_per_seq, L["packed"], L["bias"], cout, relu, None, None, y, cout, 0, tc_mode)
    torch.cuda.synchronize()
    return y


def _ref_entry(entry, x64, w, b, rows_per_seq):
    """float64: Conv1d over sequences of rows_per_seq rows (zero padding taps // 2) [+ ReLU] [+ max over pool rows]"""
    taps, relu, pool = ENTRIES[entry]
    M, cin = x64.shape
    seq = x64.view(M // rows_per_seq, rows_per_seq, cin).permute(0, 2, 1)
    y = F.conv1d(seq, w, b, padding=taps // 2).permute(0, 2, 1).reshape(M, -1)
    if relu:
        y = torch.relu(y)
    return y.view(M // pool, pool, -1).max(dim=1).values if pool else y


@pytest.mark.parametrize("entry", list(ENTRIES))
def test_per_layer_fp16_split_range_flag(entry):
    """every per-layer entry raises the range flag when an fp16-split input leaves the fp16 range - of either sign,
    the inputs here are not post-ReLU - and stays exact and silent just inside it; the other modes never raise it"""
    M, cin, cout, seq = 512, 64, 96, 128
    taps = ENTRIES[entry][0]
    w, b = _conv_weights(cin, cout, taps, seed=11 + taps)
    x0 = torch.randn(M, cin, generator=torch.Generator().manual_seed(3))
    for tc_mode in TC_MODES.values():
        L = tehnet._pack_conv1d(w.to(DEV), b.to(DEV), tc_mode)
        for value in (7e4, -7e4, 6.5e4, -6.5e4):
            x = x0.clone()
            x[200, 37] = value
            e2h.check_numeric_range(DEV)
            y = _run_entry(entry, x.to(DEV), cin, L, tc_mode, seq)
            flagged = not e2h.check_numeric_range(DEV)
            if tc_mode == _capi.TC_F16X3 and abs(value) >= 65520:
                assert flagged, (tc_mode, value)
            else:
                assert not flagged, (tc_mode, value)
                assert rel_err(y, _ref_entry(entry, x.double(), w, b, seq)) <= _tol(tc_mode), (tc_mode, value)


def _encoder(states):
    enc = e2h.SetAbstractionEncoder()
    for n, st in states.items():
        load_numpy_state(getattr(enc, n), st)
    return enc.to(DEV).eval()


def test_per_point_module_overflow_is_flagged_or_exact(monkeypatch):
    """per-point layer 1 runs in the per-layer kernel: features of 1e5 overflow its fp16 split, and the fused kernel's
    relu(P - C) would turn the NaN into a finite wrong value - the flag must say so (or the result be exact)"""
    c = CASES["p2"]
    B, N, S, D = c["B"], c["N"], c["S"], c["D"]
    state = synth.random_sa_state("conv_blocks.{i}.{j}", "bn_blocks.{i}.{j}", c["mlp"], [D + 3], 21)
    mod = load_numpy_state(e2h.PointNetSetAbstractionMsg(S, c["r"], c["K"], D, c["mlp"]), state).to(DEV).eval()
    xyz = torch.from_numpy(np.ascontiguousarray(synth.make_windows(B, N, seed=21)[:, :3]))
    feats = torch.from_numpy((1e5 * np.random.RandomState(21).randn(B, D, N)).astype(np.float32))
    start = torch.from_numpy(synth.make_start_indices(B, N, 21))
    for mode in ("f16", "tf32"):
        _set_mode(monkeypatch, mode)
        e2h.check_numeric_range(DEV)
        with torch.no_grad():
            _, rec = mod.forward_rows(xyz.to(DEV), feats.to(DEV), fps_start=start)
        flagged = not e2h.check_numeric_range(DEV)
        ref = sa_msg_f64(state, c["mlp"], c["K"], xyz, feats, mod.last_fps_idx.cpu(), mod.last_ball_idx.cpu())
        err = rel_err(rec.rows[:, :, :rec.c].permute(0, 2, 1), ref)
        if mode == "f16":
            assert flagged or err <= 1e-5, err
        else:                                   # the tf32 split keeps fp32's exponent range
            assert not flagged and err <= 1e-5, err


def test_encoder_overflow_after_an_in_range_layer(monkeypatch):
    """sa1's layer-3 BatchNorm shifts its outputs to ~1e5: sa1's fused launches stay in range (the pooled layer-3
    outputs are never split there), the overflow happens in sa2's per-point GEMM.  The fp16 split must raise the flag
    (or be exact); EV2H_SPLIT=tf32, the documented remedy, must neither raise it nor lose accuracy."""
    seeds = {"sa1": 81, "sa2": 82, "sa3": 83}
    states = {n: synth.random_state_for(synth.ENCODER_SPECS[n], seed=s) for n, s in seeds.items()}
    states["sa1"]["bn_blocks.0.2.bias"] = np.full_like(states["sa1"]["bn_blocks.0.2.bias"], 1e5)
    enc = _encoder(states)
    ev = synth.make_windows(2, 2048, seed=81)
    s1 = torch.from_numpy(synth.make_start_indices(2, 2048, 1))
    s2 = torch.from_numpy(synth.make_start_indices(2, 512, 2))
    with torch.no_grad():
        want = sa_oracle.encoder_forward(states, synth.ENCODER_SPECS, torch.from_numpy(ev), {"sa1": s1, "sa2": s2})[:, :, 0]
    for mode in ("f16", "tf32"):
        _set_mode(monkeypatch, mode)
        e2h.check_numeric_range(DEV)
        with torch.no_grad():
            got = enc(torch.from_numpy(ev).to(DEV), fps_starts=(s1, s2))
        flagged = not e2h.check_numeric_range(DEV)
        err = rel_err(got, want)
        if mode == "f16":
            assert flagged or err <= 1e-5, err
        else:
            assert not flagged and err <= 1e-5, err


@pytest.mark.parametrize("cin", [7, 33, 323])
def test_padding_columns_never_enter_the_product(cin):
    """columns Cin .. ld_x - 1 of the input rows are padding: NaN or 1e30 there changes no bit of any entry's output,
    in any mode, and raises no flag; the exact fp32 kernels on the same buffer agree"""
    M, cout = 1024, 48
    ld = (cin + 3) // 4 * 4 + 4
    w, b = _conv_weights(cin, cout, 1, seed=cin)
    clean = torch.zeros(M, ld, device=DEV)
    clean[:, :cin] = torch.randn(M, cin, generator=torch.Generator().manual_seed(cin)).to(DEV)
    wt = torch.zeros(((cin + 15) // 16 * 16, 128), device=DEV)
    wt[:cin, :cout] = w[:, :, 0].t().float().to(DEV)
    bias = torch.zeros(128, device=DEV)
    bias[:cout] = b.float().to(DEV)
    for tc_mode in TC_MODES.values():
        L = tehnet._pack_conv1d(w.to(DEV), b.to(DEV), tc_mode)
        for entry in ("linear_tc", "linear_relu_tc", "linear_relu_tc_pool128", "conv1d_tc_k1"):
            _, relu, pool = ENTRIES[entry]
            e2h.check_numeric_range(DEV)
            y0 = _run_entry(entry, clean, cin, L, tc_mode, M)
            for fill in (float("nan"), 1e30):
                dirty = clean.clone()
                dirty[:, cin:] = fill
                y = _run_entry(entry, dirty, cin, L, tc_mode, M)
                assert torch.equal(y, y0), (entry, tc_mode, fill)
                exact = torch.zeros_like(y)
                if relu:
                    _capi.linear_relu(dirty, M, ld, cin, wt, bias, cout, pool, exact, cout)
                else:
                    _capi.linear_no_relu(dirty, M, ld, cin, wt, bias, cout, exact, cout)
                assert torch.isfinite(exact).all() and rel_err(y, exact) <= _tol(tc_mode), (entry, tc_mode, fill)
            assert e2h.check_numeric_range(DEV), (entry, tc_mode)
    exact0 = torch.zeros(M, cout, device=DEV)
    _capi.linear_no_relu(clean, M, ld, cin, wt, bias, cout, exact0, cout)
    assert rel_err(exact0, clean[:, :cin].double().cpu() @ w[:, :, 0].t() + b) <= 1e-5


def test_weights_outside_the_fp16_range_raise_the_flag(monkeypatch):
    """a BatchNorm with running_var = 0 and gamma = 1e4 folds into weights beyond the fp16 range: the fp16 split
    cannot represent them and must say so; the tf32 split carries them"""
    spec = dict(kind="all", in_channel=16, mlp=[32])
    st = synth.random_state_for(spec, seed=4)
    st["mlp_bns.0.running_var"] = np.zeros_like(st["mlp_bns.0.running_var"])
    st["mlp_bns.0.weight"] = np.full_like(st["mlp_bns.0.weight"], 1e4)
    args = [torch.from_numpy(np.asarray(st[k], dtype=np.float32)).to(DEV) for k in
            ("mlp_convs.0.weight", "mlp_convs.0.bias", "mlp_bns.0.weight", "mlp_bns.0.bias", "mlp_bns.0.running_mean",
             "mlp_bns.0.running_var")]
    M = 1000
    x = torch.randn(M, 16, generator=torch.Generator().manual_seed(4))
    w64 = torch.from_numpy(st["mlp_convs.0.weight"].reshape(32, 16).astype(np.float64))
    scale = torch.from_numpy(st["mlp_bns.0.weight"].astype(np.float64)) / np.sqrt(BN_EPS)
    want = torch.relu((x.double() @ w64.t() + torch.from_numpy(st["mlp_convs.0.bias"].astype(np.float64))
                       - torch.from_numpy(st["mlp_bns.0.running_mean"].astype(np.float64))) * scale
                      + torch.from_numpy(st["mlp_bns.0.bias"].astype(np.float64)))
    for mode in ("f16", "tf32"):
        _set_mode(monkeypatch, mode)
        e2h.check_numeric_range(DEV)
        wt, bias = _capi.fold_conv_bn(args[0].view(32, 16), *args[1:], BN_EPS)
        assert float(wt.abs().max()) >= 65520
        layers = [{"wt": wt, "bias": bias, "cin": 16, "cout": 32, "packed": {}}]
        out = torch.zeros(M, 32, device=DEV)
        pu._mlp_rows(x.to(DEV), M, 16, layers, 0, out, 32, 0)
        flagged = not e2h.check_numeric_range(DEV)
        if mode == "f16":
            assert flagged
        else:
            assert not flagged and rel_err(out, want) <= 1e-5
