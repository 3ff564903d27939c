"""Training path of the set-abstraction modules against a float64 restatement of the same operations.

A train-mode forward of PointNetSetAbstractionMsg / PointNetSetAbstraction (group_all) runs the library's kernels in
both directions: the gather and its scatter-add backward (group.cu), the row GEMMs of _LinearRowsTC - exact fp32
forward (linear_ffma.cu) or the per-layer tensor-core kernel (linear_tc.cu), the input gradient in the tf32 + bf16
split, the weight and bias gradients in wgrad_ffma.cu - BatchNorm over rows (_bn_rows), and on the channel-first path
the max-pool kernels.  A wrong gradient there does not crash anything; it only trains worse.  So every module of the
model is checked here, at its own layer shapes, against plain float64 autograd on the module's own indices: output,
input gradient, every parameter gradient and the running statistics.  The kernels of the backward pass are also
checked one by one at their edges.

The reference takes the kernels' side of ReLU's kink wherever an input to ReLU lies within the forward bar of 0
(see mlp64), and the loss weights skip pooled outputs whose arg-max is a near tie (see route_mask): both are choices
between values equal to within rounding that fp32 and fp64 may make differently, and either moves gradients by far
more than rounding.  With them the bars are: forward 1e-5 of max|reference|; gradients 5e-5 with the exact fp32
forward (EV2H_TRAIN_TC "" and "dgrad") and 1e-4 with the tensor-core forward ("all"); running statistics 1e-5.
Measured on a B200: gradients within 7.1e-6 in every mode, forward within 1.3e-6, running statistics within 1.1e-6."""
import json
import os

import numpy as np
import pytest
import torch

import ev2hands_b200 as e2h
from ev2hands_b200 import _capi, synth
from ev2hands_b200 import pointnet2_utils as pu
from ev2hands_b200.encoder import load_numpy_state

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FWD_TOL = 1e-5
GRAD_TOL = {"": 5e-5, "dgrad": 5e-5, "all": 1e-4}
BIAS_NOISE = 2e-5             # gradient of a conv bias in front of a batch-statistics BatchNorm, over the weights' scale
STAT_TOL = 1e-5
MEASURED = {}


def rel_err(got, want):
    got, want = got.detach().double(), want.detach().double().to(got.device)
    return float((got - want).abs().max() / max(float(want.abs().max()), 1e-30))


def _record(key, payload):
    """collect the measured errors; with EV2H_TEST_RECORD_DIR set, also write them there as train_envelope.json
    (the bars and the measured margins under them are documented from such a file)"""
    MEASURED[key] = payload
    d = os.environ.get("EV2H_TEST_RECORD_DIR")
    if not d:
        return
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "train_envelope.json"), "w") as f:
            json.dump(MEASURED, f, indent=1, sort_keys=True)
    except OSError:
        pass


@pytest.fixture(autouse=True)
def strict_fp32(monkeypatch):
    """stock torch ops in exact fp32 (cuBLAS / cuDNN would otherwise run plain tf32), and the library's default
    arithmetic for everything the test does not set itself"""
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    for name, value in (("_mlp_precision", "tf32x3"), ("_SPLIT", "f16"), ("_TF32X3_PURE", False), ("_LINEAR_MIXED", True),
                        ("_TRAIN_FFMA", True), ("_TRAIN_WGRAD", True), ("_TRAIN_ROWS", True), ("_TRAIN_TC", "dgrad")):
        monkeypatch.setattr(pu, name, value)
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


# ------------------------------------------------------------------ float64 restatement ----------------------------
def _params64(convs, bns):
    """float64 leaf copies of a conv / BatchNorm stack: [(w [Cout, Cin], b, gamma, beta)]"""
    def leaf(t):
        return t.detach().double().clone().requires_grad_(True)
    return [(leaf(conv.weight.view(conv.out_channels, -1)), leaf(conv.bias), leaf(bn.weight), leaf(bn.bias))
            for conv, bn in zip(convs, bns)]


def _running0(bns):
    """the running statistics before a forward, float64"""
    return [(bn.running_mean.detach().double().clone(), bn.running_var.detach().double().clone()) for bn in bns]


def mlp64(h, layers, sides=None, flips=None, eps=1e-5):
    """relu(batchnorm(h W^T + b)) with batch statistics (biased variance to normalise) over rows h [M, Cin] ->
    (h [M, Cout], [(batch mean, unbiased batch variance)] per layer, the last layer's input to ReLU, detached).

    sides: per layer, where the kernels' own input to ReLU was positive (bool [M, Cout]).  Within the forward bar of 0
    ReLU takes the kernels' side: such an input can land on either side of the kink in fp32, and the backward of a
    batch-statistics BatchNorm hands every row a share of every winner's gradient, so one element taken the other way
    anywhere moves the layer's weight and BatchNorm gradients by up to 1e-3 of their maximum (measured in sa2); taking
    the kernels' side there changes a value by less than the bar.  flips counts the elements where the sides differ:
    "near" (followed) and "far" (outside the bar: a wrong activation, which the caller asserts never happens)."""
    stats = []
    for i, (w, b, gamma, beta) in enumerate(layers):
        h = h @ w.t() + b
        mean, var = h.mean(0), h.var(0, unbiased=False)
        stats.append((mean.detach(), h.detach().var(0, unbiased=True)))
        z = (h - mean) / torch.sqrt(var + eps) * gamma + beta
        if sides is None:
            h = torch.relu(z)
            continue
        own = z.detach() > 0
        near = z.detach().abs() < FWD_TOL * float(z.detach().abs().max())
        differ = sides[i] != own
        flips["near"] += int((differ & near).sum())
        flips["far"] += int((differ & ~near).sum())
        h = z * torch.where(near, sides[i], own)
    return h, stats, z.detach()


def msg64(layers_per_scale, nsample_list, xyz_cf, feats64_cf, new_xyz_cf, ball, sides=None, flips=None):
    """PointNetSetAbstractionMsg's train-mode forward: rows [feats | xyz - centre] (the cat order of
    pointnet2_utils.py:244-248, the subtraction in fp32 like the reference), the layer stack, max over K.
    sides: the kernels' ReLU sides (see mlp64), scale after scale.
    -> (out [B, sum C', S], the last layer's input to ReLU per scale [B, S, K, C'], batch statistics per scale)"""
    B, _, N = xyz_cf.shape
    xyz = xyz_cf.permute(0, 2, 1)
    centres = new_xyz_cf.permute(0, 2, 1)
    S = centres.shape[1]
    ball = ball.long()
    assert int(ball.min()) >= 0 and int(ball.max()) < N
    bi = torch.arange(B, device=ball.device).view(B, 1, 1)
    pooled, pre, stats, k_off = [], [], [], 0
    for i, (layers, K) in enumerate(zip(layers_per_scale, nsample_list)):
        idx = ball[:, :, k_off:k_off + K]
        rel = (xyz[bi, idx] - centres.view(B, S, 1, 3)).double()
        h = rel if feats64_cf is None else torch.cat([feats64_cf.permute(0, 2, 1)[bi, idx], rel], -1)
        h, st, z = mlp64(h.reshape(B * S * K, -1), layers, None if sides is None else sides[i], flips)
        pre.append(z.view(B, S, K, -1))
        pooled.append(h.view(B, S, K, -1).max(dim=2).values.permute(0, 2, 1))
        stats.append(st)
        k_off += K
    return torch.cat(pooled, 1), pre, stats


def all64(layers, xyz_cf, feats64_cf, sides=None, flips=None):
    """group_all: channels [xyz, points] (pointnet2_utils.py:141-158), the layer stack, max over the N points"""
    B, _, N = xyz_cf.shape
    g = xyz_cf.double() if feats64_cf is None else torch.cat([xyz_cf.double(), feats64_cf], 1)
    h, st, z = mlp64(g.permute(0, 2, 1).reshape(B * N, -1), layers, None if sides is None else sides[0], flips)
    return h.view(B, 1, N, -1).max(dim=2).values.permute(0, 2, 1), [z.view(B, 1, N, -1)], [st]


def running64(rm, rv, batch_stats, momentum):
    """the running-statistics rule of torch's _BatchNorm over successive batches from (rm, rv), num_batches_tracked
    starting at 0 (momentum None: cumulative average)"""
    for n, (mean, var) in enumerate(batch_stats, 1):
        f = 1.0 / n if momentum is None else momentum
        rm, rv = (1 - f) * rm + f * mean, (1 - f) * rv + f * var
    return rm, rv


def route_mask(pre, out64, tol):
    """loss weights that keep fp32 and fp64 on the same arg-max: 0 where the pooled winner's input to ReLU is within
    10 x the forward bar of the best strictly smaller value, or of 0 (ReLU's kink).  A winner below -bar routes nothing
    (ReLU's gradient is 0 for every candidate).  Exact copies of a row (K-padding copies of the first neighbour) are
    bitwise equal in both precisions and route identically, so they are no tie.
    pre: [B, S, K, C] per scale -> keep [B, sum C, S] (bool)"""
    thr = 10 * tol * float(out64.detach().abs().max())
    keep = []
    for z in pre:
        top = z.max(dim=2, keepdim=True).values
        below = torch.where(z < top, z, torch.full_like(z, -float("inf"))).max(dim=2).values
        top = top.squeeze(2)
        keep.append(((top.abs() >= thr) & ((top < 0) | (top - below >= thr))).permute(0, 2, 1))
    return torch.cat(keep, 1)


def _spy_relu_sides(monkeypatch, bns):
    """records, layer after layer, where the module's input to ReLU is positive, as rows [M, C] in the restatement's
    order: _bn_rows' output on the rows path, the BatchNorm modules' output [B, C, K, S] on the channel-first path"""
    sides = []
    real = pu._bn_rows

    def spy(x2d, bn):
        y = real(x2d, bn)
        sides.append(y.detach() > 0)
        return y
    monkeypatch.setattr(pu, "_bn_rows", spy)
    hooks = [bn.register_forward_hook(lambda mod, args, y: sides.append(
        (y.detach() > 0).permute(0, 3, 2, 1).reshape(-1, y.shape[1]))) for bn in bns]
    return sides, hooks


# ------------------------------------------------------------------ 1. the restatement against the reference -------
def test_f64_restatement_agrees_with_the_reference_autograd(golden):
    """the float64 restatement reproduces the reference module's own CPU autograd (tests/golden/train_sa2.npz) within
    that golden's bars, so that it can stand in for the reference at the other modules' shapes"""
    g = golden("train_sa2")
    spec = synth.ENCODER_SPECS["sa2"]
    m = e2h.PointNetSetAbstractionMsg(spec["npoint"], spec["radius_list"], spec["nsample_list"], spec["in_channel"], spec["mlp_list"])
    load_numpy_state(m, synth.random_state_for(spec, seed=int(g["weight_seed"])))
    m = m.to(DEV).train()
    ev = torch.from_numpy(g["events"]).to(DEV)
    feats = torch.from_numpy(np.random.RandomState(int(g["feats_seed"])).randn(2, 320, 512).astype(np.float32)).to(DEV)
    layers = [_params64(m.conv_blocks[i], m.bn_blocks[i]) for i in range(2)]
    run0 = [_running0(b) for b in m.bn_blocks]
    with torch.no_grad():
        new_xyz, _ = m(ev[:, :3], feats, fps_start=torch.from_numpy(g["start"]))
    assert np.array_equal(new_xyz.cpu().numpy(), g["new_xyz"])
    f64 = feats.double().requires_grad_(True)
    out, _, stats = msg64(layers, spec["nsample_list"], ev[:, :3], f64, new_xyz, m.last_ball_idx)
    lw = torch.from_numpy(np.linspace(0.5, 1.5, out.numel())).view_as(out).to(DEV)
    (out * lw).sum().backward()
    assert rel_err(out[:, ::4, ::4], torch.from_numpy(g["out_every4"])) <= 2e-5
    assert rel_err(f64.grad[:, :, ::8], torch.from_numpy(g["grad_feats_every8"])) <= 2e-4
    names = {"conv_blocks.0.0.weight": layers[0][0][0], "conv_blocks.1.1.weight": layers[1][1][0],
             "bn_blocks.0.1.weight": layers[0][1][2], "bn_blocks.1.0.bias": layers[1][0][3]}
    for n, p in names.items():
        assert rel_err(p.grad.view(g["grad." + n].shape), torch.from_numpy(g["grad." + n])) <= 2e-4, n
    # the golden holds the running statistics after one train-mode forward from the state's
    for (i, j, key, which) in ((0, 0, "running_mean_0_0", 0), (1, 2, "running_var_1_2", 1)):
        want = running64(*run0[i][j], [stats[i][j]], m.bn_blocks[i][j].momentum)[which]
        assert rel_err(want, torch.from_numpy(g[key])) <= 1e-5, key


# ------------------------------------------------------------------ 2. the five modules in train mode --------------
# the model's five set-abstraction instances (synth specs), at B = 2 and the point counts they see in the model
MODULES = {
    "enc_sa1": dict(spec=synth.ENCODER_SPECS["sa1"], B=2, N=2048, D=5),
    "enc_sa2": dict(spec=synth.ENCODER_SPECS["sa2"], B=2, N=512, D=320),
    "enc_sa3": dict(spec=synth.ENCODER_SPECS["sa3"], B=2, N=128, D=512),
    "reg_sa1": dict(spec=synth.REGRESSOR_SPECS["sa1"], B=2, N=2048, D=4),
    "reg_sa2": dict(spec=synth.REGRESSOR_SPECS["sa2"], B=2, N=128, D=512),
}
# (module, EV2H_TRAIN_TC, rows path, BatchNorm momentum, batch)
RUNS = [(name, tc, True, 0.1, None) for name in MODULES for tc in ("", "dgrad", "all")] + [
    # B = 8: B*S*K*D = 2.6M gradient elements at K = 128, past one pass of the gather backward's capped grid
    ("enc_sa1", "dgrad", True, 0.1, 8),
    # the channel-first path: cuDNN convolutions, max-pool and its backward in the library's kernels
    ("enc_sa1", "dgrad", False, 0.1, None),
    ("enc_sa3", "dgrad", False, 0.1, None),
    # momentum None: _bn_rows' cumulative-average rule
    ("reg_sa1", "dgrad", True, None, None),
]


def _run_id(r):
    name, tc, rows, momentum, B = r
    return "%s-%s%s%s%s" % (name, tc or "fp32", "" if rows else "-cf", "" if momentum is not None else "-cma",
                           "" if B is None else "-B%d" % B)


def _build(name, B):
    c = MODULES[name]
    spec, N, D = c["spec"], c["N"], c["D"]
    B = B or c["B"]
    seed = sum(map(ord, name))
    if spec["kind"] == "msg":
        m = e2h.PointNetSetAbstractionMsg(spec["npoint"], spec["radius_list"], spec["nsample_list"], spec["in_channel"], spec["mlp_list"])
    else:
        m = e2h.PointNetSetAbstraction(None, None, None, spec["in_channel"], spec["mlp"], group_all=True)
    load_numpy_state(m, synth.random_state_for(spec, seed=seed))
    xyz = torch.from_numpy(np.ascontiguousarray(synth.make_windows(B, N, seed=seed)[:, :3])).to(DEV)
    rs = np.random.RandomState(seed)
    feats = [torch.from_numpy(rs.randn(B, D, N).astype(np.float32)).to(DEV) for _ in range(2)]
    start = torch.from_numpy(synth.make_start_indices(B, N, seed))
    return m.to(DEV).train(), xyz, feats, start


@pytest.mark.parametrize("run", RUNS, ids=_run_id)
def test_train_mode_module_vs_f64(run, monkeypatch):
    name, tc, rows, momentum, B = run
    monkeypatch.setattr(pu, "_TRAIN_TC", tc)
    monkeypatch.setattr(pu, "_TRAIN_ROWS", rows)
    m, xyz, feats, start = _build(name, B)
    msg = isinstance(m, e2h.PointNetSetAbstractionMsg)
    convs_bns = [(m.conv_blocks[i], m.bn_blocks[i]) for i in range(len(m.conv_blocks))] if msg else [(m.mlp_convs, m.mlp_bns)]
    bn_list = [bn for _, bns in convs_bns for bn in bns]
    for bn in bn_list:
        bn.momentum = momentum
    layers = [_params64(convs, bns) for convs, bns in convs_bns]
    run0 = _running0(bn_list)
    e2h.check_numeric_range(DEV)

    # fp32 forward (the kernels), then the float64 forward on the same indices and ReLU sides
    recorded, hooks = _spy_relu_sides(monkeypatch, bn_list)
    f32 = feats[0].clone().requires_grad_(True)
    new_xyz, out = m(xyz, f32, fps_start=start)
    for h in hooks:
        h.remove()
    sides = list(recorded)
    widths = [len(bns) for _, bns in convs_bns]
    assert len(sides) == sum(widths)
    sides = [sides[sum(widths[:i]):sum(widths[:i + 1])] for i in range(len(widths))]
    f64 = feats[0].double().requires_grad_(True)
    flips = {"near": 0, "far": 0}
    if msg:
        out64, pre, stats = msg64(layers, m.nsample_list, xyz, f64, new_xyz, m.last_ball_idx, sides, flips)
    else:
        out64, pre, stats = all64(layers[0], xyz, f64, sides, flips)
    fwd = rel_err(out, out64)

    # loss weights: a seeded linear ramp, zero where fp32 and fp64 could pick different winners of a max
    keep = route_mask(pre, out64, FWD_TOL)
    masked = 1.0 - float(keep.double().mean())
    lw = torch.from_numpy(np.linspace(0.5, 1.5, out.numel(), dtype=np.float32)).view_as(out).to(DEV) * keep
    (out * lw).sum().backward()
    (out64 * lw.double()).sum().backward()

    errs = {"out": fwd, "feats.grad": rel_err(f32.grad, f64.grad), "masked_fraction": masked}
    n_relu = sum(int(t.numel()) for scale in sides for t in scale)
    bias_noise = {}
    prefix = ("conv_blocks.%d.%d", "bn_blocks.%d.%d") if msg else ("mlp_convs.%d", "mlp_bns.%d")
    params = dict(m.named_parameters())
    for i, scale in enumerate(layers):
        for j, (w, b, gamma, beta) in enumerate(scale):
            ij = (i, j) if msg else (j,)
            cname, bname = prefix[0] % ij, prefix[1] % ij
            errs[cname + ".weight"] = rel_err(params[cname + ".weight"].grad.view_as(w), w.grad)
            errs[bname + ".weight"] = rel_err(params[bname + ".weight"].grad, gamma.grad)
            errs[bname + ".bias"] = rel_err(params[bname + ".bias"].grad, beta.grad)
            # a convolution bias in front of a batch-statistics BatchNorm has an exactly zero gradient (the mean is
            # subtracted): what either side holds is rounding noise, compared with the layer's weight-gradient scale
            wscale = float(w.grad.abs().max())
            bias_noise[cname + ".bias"] = max(float(params[cname + ".bias"].grad.abs().max()), float(b.grad.abs().max())) / wscale

    # a second train-mode forward on other features: running statistics over two batches
    with torch.no_grad():
        m(xyz, feats[1], fps_start=start)
        if msg:
            _, _, stats2 = msg64(layers, m.nsample_list, xyz, feats[1].double(), new_xyz, m.last_ball_idx)
        else:
            _, _, stats2 = all64(layers[0], xyz, feats[1].double())
    batches = [pair for s1, s2 in zip(stats, stats2) for pair in zip(s1, s2)]          # per BatchNorm, in bn_list order
    stat_err = 0.0
    for bn, (rm, rv), pair in zip(bn_list, run0, batches):
        rm, rv = running64(rm, rv, pair, momentum)
        stat_err = max(stat_err, rel_err(bn.running_mean, rm), rel_err(bn.running_var, rv))
        assert int(bn.num_batches_tracked) == 2
    errs["running_stats"] = stat_err
    flag_clear = e2h.check_numeric_range(DEV)
    gtol = GRAD_TOL[tc]
    grads = {k: v for k, v in errs.items() if k not in ("out", "running_stats") and not k.startswith("masked")}
    _record(_run_id(run), dict(errs, max_grad=max(grads.values()), max_bias_noise=max(bias_noise.values()), flag_clear=flag_clear,
                               relu_followed=flips["near"], relu_wrong=flips["far"], relu_elements=n_relu))

    assert flips["far"] == 0, flips           # every hidden activation on the right side of ReLU, up to the bar
    assert masked < 0.01, masked
    assert fwd <= FWD_TOL, fwd
    for key, e in grads.items():
        assert e <= gtol, (key, e)
    for key, e in bias_noise.items():
        assert e <= BIAS_NOISE, (key, e)
    assert stat_err <= STAT_TOL, stat_err
    if tc == "all":
        assert flag_clear                      # in-range inputs: a raised flag would be a false positive


# ------------------------------------------------------------------ 3. the backward kernels at their edges ---------
# (M, Cin, Cout, row stride of x) of every layer the five modules run at B = 2, plus the edges of the kernels behind them
LINEAR_SHAPES = sorted({
    # encoder sa1: S = 512, K = 32 / 64 / 128, [feats(5) | rel(3)] rows; the input gradient of layer 1 has 8 columns
    (32768, 8, 32, 8), (32768, 32, 32, 32), (32768, 32, 64, 32),
    (65536, 8, 64, 8), (65536, 64, 64, 64), (65536, 64, 128, 64),
    (131072, 8, 64, 8), (131072, 64, 96, 64), (131072, 96, 128, 96),
    # encoder sa2 (S = 128, K = 64 / 128, 323 channels in 324-wide rows) and regressor sa1 (7 channels in 8-wide rows)
    (16384, 323, 128, 324), (16384, 128, 128, 128), (16384, 128, 256, 128),
    (32768, 323, 128, 324), (32768, 128, 196, 128), (32768, 196, 256, 196),
    (16384, 7, 128, 8), (32768, 7, 128, 8),
    # encoder sa3 / regressor sa2 over B * N = 256 rows; sa3's input gradient contracts over 1024 channels into 512
    (256, 515, 256, 515), (256, 256, 512, 256), (256, 512, 1024, 512),
    # M not a multiple of 128, and M >= 2^20
    (1000, 8, 64, 8), (4001, 196, 256, 196), ((1 << 20) + 37, 8, 64, 8),
})


def _grad_like(M, cout, seed):
    """an output gradient with a gradient's dynamic range: rows scaled by 10^-U(0, 8)"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    dy = torch.randn(M, cout, device=DEV, generator=g)
    return dy * torch.pow(10.0, -8 * torch.rand(M, 1, device=DEV, generator=g))


def _elementwise(err, bound):
    """max of |err| / bound (bound: the same product over absolute values), 0 / 0 counted as 0"""
    return float(torch.where(bound > 0, err.abs() / bound, err.abs() * float("inf")).nan_to_num(0.0).max())


@pytest.mark.parametrize("pure", [False, True], ids=["tf32_bf16c", "tf32x3"])
@pytest.mark.parametrize("shape", LINEAR_SHAPES, ids=lambda s: "M%d-%dx%d-ld%d" % s)
def test_linear_rows_forward_backward_vs_f64(shape, pure, monkeypatch):
    """_LinearRowsTC at every layer shape of the training path, elementwise against float64: forward (exact fp32, or
    the tensor-core kernel in the mode _layer_mode gives it), input gradient (the per-layer kernel in the tf32 + bf16
    split or three tf32 products: fp32's exponent range, so rows of 1e-8 keep their accuracy), weight and bias
    gradient (wgrad_ffma.cu).  Each error is measured against the same product over absolute values."""
    M, cin, cout, ld = shape
    monkeypatch.setattr(pu, "_TF32X3_PURE", pure)
    g = torch.Generator(device=DEV).manual_seed(M + cin + cout)
    base = torch.randn(M, ld, device=DEV, generator=g)
    w = torch.randn(cout, cin, device=DEV, generator=g) / cin ** 0.5
    b = 0.1 * torch.randn(cout, device=DEV, generator=g)
    dy = _grad_like(M, cout, seed=cin * cout)
    x64, w64, b64, dy64 = base[:, :cin].double(), w.double(), b.double(), dy.double()
    y64 = x64 @ w64.t() + b64
    ybound = x64.abs() @ w64.abs().t() + b64.abs()
    res = {}
    fwd_tc_ok = pu._rows_ok(base[:, :cin]) and _capi.tc_supported(cout, 0) and cin <= 1024 and cout % 4 == 0
    for fwd_tc in ([False, True] if fwd_tc_ok else [False]):
        xb = base.clone().requires_grad_(True)
        wl, bl = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
        y = pu._LinearRowsTC.apply(xb[:, :cin], wl, bl, fwd_tc)
        y.backward(dy)
        key = "tc" if fwd_tc else "fp32"
        res["fwd_" + key] = rel_err(y, y64)
        res["fwd_elem_" + key] = _elementwise(y.double() - y64, ybound)
        if fwd_tc:
            continue
        res["dx"] = _elementwise(xb.grad[:, :cin].double() - dy64 @ w64, dy64.abs() @ w64.abs())
        res["dx_padding_zero"] = bool((xb.grad[:, cin:] == 0).all())
        res["dw"] = _elementwise(wl.grad.double() - dy64.t() @ x64, dy64.abs().t() @ x64.abs())
        res["db"] = _elementwise(bl.grad.double() - dy64.sum(0), dy64.abs().sum(0))
    _record("linear-%s-M%d-%dx%d-ld%d" % ((("tf32x3" if pure else "tf32_bf16c"),) + shape), res)
    for key in ("fwd_fp32", "fwd_tc"):
        if key in res:
            assert res[key] <= FWD_TOL, (key, res[key])
    assert res["dx_padding_zero"]
    assert res["dx"] <= 1e-5, res["dx"]
    assert res["dw"] <= 5e-6 and res["db"] <= 5e-6, res


# (B, N, S, K, D, idx_ld, k_off, ld_grad): scale offsets into multi-scale index blocks, gradient rows wider than
# D + 3, D from 1 to 320, and work past one pass of the capped grid (148 * 32 CTAs of 256 threads)
GATHER_CASES = {
    "d1": (2, 300, 37, 32, 1, 32, 0, 4),
    "d4-koff": (3, 777, 40, 64, 4, 224, 32, 8),
    "d5-ld12": (2, 2048, 64, 128, 5, 224, 96, 12),
    "d5-wrap": (8, 2048, 512, 128, 5, 224, 96, 8),
    "d320-wrap": (2, 512, 128, 128, 320, 192, 64, 324),
}


@pytest.mark.parametrize("case", list(GATHER_CASES))
def test_group_gather_backward_vs_f64_index_add(case):
    """ev2h_group_gather_bwd_f32 against a float64 index_add_: sentinel entries (N, negative) are skipped, a group
    whose K entries are one point adds K rows into it, other points get nothing; each element within the fp32
    summation bound n eps sum|g| of its own n contributions (atomics choose the order)"""
    B, N, S, K, D, idx_ld, k_off, ld = GATHER_CASES[case]
    g = torch.Generator(device=DEV).manual_seed(sum(map(ord, case)))
    idx = torch.randint(0, N, (B, S, idx_ld), device=DEV, generator=g, dtype=torch.int64)
    blk = idx[:, :, k_off:k_off + K]
    blk[0, 1] = 3                                                      # every neighbour the same point
    blk[B - 1, S - 1, K // 2:] = N                                     # ball-query sentinel
    blk[0, 2, 1] = -1
    blk[B - 1, 0, ::3] = -7
    idx = idx.to(torch.int32)
    grad = torch.randn(B, S, K, ld, device=DEV, generator=g)
    grad[..., D:] = float("nan")                                       # columns >= D are not the features' gradient
    out = torch.zeros(B, N, D, device=DEV)
    _capi.group_gather_bwd(grad, ld, idx, k_off, B, N, S, K, D, out)
    p = idx[:, :, k_off:k_off + K].long()
    valid = ((p >= 0) & (p < N)).reshape(-1)
    dst = (torch.arange(B, device=DEV).view(B, 1, 1) * N + p).reshape(-1)[valid]
    rows = grad[..., :D].reshape(-1, D)[valid].double()
    want = torch.zeros(B * N, D, dtype=torch.float64, device=DEV).index_add_(0, dst, rows)
    count = torch.zeros(B * N, 1, dtype=torch.float64, device=DEV).index_add_(0, dst, torch.ones_like(rows[:, :1]))
    asum = torch.zeros(B * N, D, dtype=torch.float64, device=DEV).index_add_(0, dst, rows.abs())
    err = (out.view(B * N, D).double() - want).abs()
    ratio = _elementwise(err, count * 2.0 ** -24 * asum)
    _record("gather_bwd-" + case, {"work_over_grid": B * S * K * D / (148 * 32 * 256), "err_over_bound": ratio})
    assert torch.isfinite(out).all()
    assert ratio <= 1.0, ratio              # also: points nobody gathered (bound 0) hold exactly 0


def _max_cases():
    """[B, C, K, S] inputs for the max-pool kernels: S and C off multiples of 32, K = 1, -inf, ties and NaN"""
    g = torch.Generator(device=DEV).manual_seed(7)
    cases = {"k1": torch.randn(2, 37, 1, 45, device=DEV, generator=g)}
    x = torch.randn(3, 37, 16, 45, device=DEV, generator=g)
    x[0, 0, :, 0] = -float("inf")                      # a column of -inf: index 0, value -inf
    x[0, 1, :, 1] = 0.25                               # all equal: the first index wins
    x[0, 2, 5:, 2] = -float("inf")
    x[1, 3, 4, 3] = x[1, 3, 9, 3] = 9.0                # a duplicated maximum
    x[1, 4, 0, 4] = float("nan")                       # NaN first
    x[1, 5, 7, 5] = float("nan")                       # NaN mid-column
    x[2, 6, [2, 8, 15], 6] = float("nan")              # several NaN
    x[2, 7, 15, 7] = float("nan")                      # NaN last, behind a large maximum
    x[2, 7, 3, 7] = 1e30
    x[2, 8, :, 8] = float("nan")                       # all NaN
    cases["edges"] = x
    cases["k128"] = torch.randn(2, 70, 128, 33, device=DEV, generator=g)
    return cases


@pytest.mark.parametrize("case", ["k1", "edges", "k128"])
def test_group_max_and_backward_vs_torch_max(case):
    """ev2h_group_max_f32 returns torch.max(dim=2)'s values and indices - the first maximum, NaN propagating from
    its first occurrence, as torch does on CUDA - and the backward routes the whole gradient to exactly that index"""
    x = _max_cases()[case]
    want = x.double().max(dim=2)
    out, arg = _capi.group_max(x, want_arg=True)
    assert torch.equal(out.isnan(), want.values.isnan())
    assert torch.equal(out.double().nan_to_num(), want.values.nan_to_num())
    assert torch.equal(arg.long(), want.indices)
    assert torch.equal(x.float().max(dim=2).indices, want.indices)     # fp32 torch agrees with its fp64
    go = torch.randn_like(out)
    gx = _capi.group_max_bwd(go, arg, x.shape[2])
    routed = torch.zeros_like(x).scatter_(2, want.indices.unsqueeze(2), go.unsqueeze(2))
    assert torch.equal(gx, routed)
    xa = x.clone().requires_grad_(True)
    xb = x.clone().requires_grad_(True)
    pu._GroupMax.apply(xa).backward(go)
    xb.max(dim=2).values.backward(go)
    assert torch.equal(xa.grad, xb.grad)
