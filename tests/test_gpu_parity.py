"""Parity of the CUDA path (through the C ABI, libev2h.so) with the oracles and with
the golden vectors the real reference produced.

Bars (BASELINE.json north_star): FPS and ball-query indices bit-exact; features within
1e-5 of the tensor's max magnitude in fp32.  All tests here need a GPU."""
import numpy as np
import pytest
import torch

import ev2hands_b200 as e2h
from ev2hands_b200 import _capi, synth
from ev2hands_b200.encoder import load_numpy_state
from oracle import c_oracle, sa_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FEAT_TOL = 1e-5     # max|got - want| <= FEAT_TOL * max|want|, per tensor (fp32 path)


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def rel_err(got, want):
    got = got.detach().cpu().double().numpy() if torch.is_tensor(got) else np.asarray(got, dtype=np.float64)
    want = want.detach().cpu().double().numpy() if torch.is_tensor(want) else np.asarray(want, dtype=np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


# ------------------------------------------------------------------ FPS -------------------------
def test_fps_golden(golden):
    g = golden("fps_ball")
    got = e2h.farthest_point_sample(dev(g["xyz"]), 512, start=torch.from_numpy(g["start"]))
    assert got.dtype == torch.int64
    assert np.array_equal(got.cpu().numpy(), g["fps_idx"].astype(np.int64))


def test_fps_edge_cases(golden):
    g = golden("edge")
    for key, s in (("same", 16), ("grid", 96), ("odd", 40)):
        got = e2h.farthest_point_sample(dev(g[key + "_xyz"]), s, start=torch.from_numpy(g[key + "_start"]))
        assert np.array_equal(got.cpu().numpy(), g[key + "_fps"]), key


@pytest.mark.parametrize("n,s", [(1, 1), (33, 40), (128, 128), (512, 128), (777, 64), (2048, 512),
                                 (3000, 100), (4096, 64), (8192, 48), (16384, 512)])
def test_fps_vs_c_oracle(n, s):
    b = 3
    ev = synth.make_windows(b, n, seed=40 + n) if n >= 64 else synth.make_windows(b, n, seed=1, mode="uniform")
    xyz = np.ascontiguousarray(ev[:, :3].transpose(0, 2, 1))
    start = synth.make_start_indices(b, n, seed=n)
    want = c_oracle.fps(xyz, s, start)
    got = e2h.farthest_point_sample(dev(xyz), s, start=torch.from_numpy(start)).cpu().numpy()
    assert np.array_equal(got, want)


def test_fps_reads_strided_channel_first_view():
    # TEHNet.py:174 hands the module xyz[:, :3, :], a non-contiguous view of [B,5,N]
    ev = dev(synth.make_windows(2, 2048, seed=3))
    start = torch.from_numpy(synth.make_start_indices(2, 2048, seed=9))
    view = ev[:, :3, :]
    idx, rows, cf = _capi.fps(view, _capi.cf_strides(view), start, 2, 2048, 512)
    xyz_rows = view.permute(0, 2, 1).contiguous()
    want = c_oracle.fps(xyz_rows.cpu().numpy(), 512, start.numpy())
    assert np.array_equal(idx.cpu().numpy(), want)
    picked = torch.gather(xyz_rows, 1, idx.long().unsqueeze(-1).expand(-1, -1, 3))
    assert torch.equal(rows, picked) and torch.equal(cf, picked.permute(0, 2, 1))


# ------------------------------------------------------------------ ball query / sqdist ---------
@pytest.mark.parametrize("r,k", [(0.1, 32), (0.2, 64), (0.4, 128)])
def test_ball_query_golden(golden, r, k):
    g = golden("fps_ball")
    xyz = dev(g["xyz"])
    idx = torch.from_numpy(g["fps_idx"].astype(np.int64)).to(DEV)
    centres = torch.gather(xyz, 1, idx.unsqueeze(-1).expand(-1, -1, 3))
    got = e2h.query_ball_point(r, k, xyz, centres)
    assert np.array_equal(got.cpu().numpy(), g["ball_r%g" % r].astype(np.int64))


def test_ball_query_multi_radius_one_pass(golden):
    g = golden("fps_ball")
    xyz = dev(g["xyz"])
    idx = torch.from_numpy(g["fps_idx"].astype(np.int64)).to(DEV)
    centres = torch.gather(xyz, 1, idx.unsqueeze(-1).expand(-1, -1, 3))
    packed = _capi.ball_query(xyz, _capi.rows_strides(xyz), centres, 2048, [0.1, 0.2, 0.4], [32, 64, 128]).cpu().numpy()
    assert packed.shape == (2, 512, 224)
    assert np.array_equal(packed[:, :, :32], g["ball_r0.1"])
    assert np.array_equal(packed[:, :, 32:96], g["ball_r0.2"])
    assert np.array_equal(packed[:, :, 96:], g["ball_r0.4"])


def test_ball_query_edge_cases(golden):
    g = golden("edge")
    same = dev(g["same_xyz"])
    assert np.array_equal(e2h.query_ball_point(0.2, 8, same, same[:, :4].contiguous()).cpu().numpy(), g["same_ball"])
    gx = dev(g["grid_xyz"])
    gc = torch.stack([gx[b, torch.from_numpy(g["grid_fps"][b, :24]).to(DEV)] for b in range(2)])
    assert np.array_equal(e2h.query_ball_point(0.5, 16, gx, gc).cpu().numpy(), g["grid_ball_r0.5_k16"])
    ox = dev(g["odd_xyz"])
    oc = torch.stack([ox[b, torch.from_numpy(g["odd_fps"][b]).to(DEV)] for b in range(2)])
    for r, k in [(0.3, 16), (0.7, 48), (1e-3, 4), (4.0, 301)]:
        got = e2h.query_ball_point(r, k, ox, oc).cpu().numpy()
        assert np.array_equal(got, g["odd_ball_r%g_k%d" % (r, k)]), (r, k)
    got = e2h.query_ball_point(0.2, 4, ox, dev(g["far_centres"])).cpu().numpy()
    assert np.array_equal(got, g["far_ball_r0.2_k4"])          # no neighbour: sentinel N everywhere


def test_square_distance_bitwise(golden):
    g = golden("fps_ball")
    xyz = g["xyz"][:1]
    centres = xyz[:, g["fps_idx"][0, :8].astype(np.int64)]
    got = e2h.square_distance(dev(centres), dev(xyz)).cpu().numpy()[0]
    assert np.array_equal(got.view(np.uint32), g["sqdist_w0_first8"].view(np.uint32))


@pytest.mark.parametrize("n,s,radii,ks", [(2048, 128, [0.4, 0.8], [64, 128]), (512, 128, [0.4, 0.8], [64, 128]),
                                          (16384, 512, [0.1, 0.2, 0.4], [32, 64, 128]), (1000, 77, [0.25], [20])])
def test_ball_query_vs_c_oracle(n, s, radii, ks):
    b = 2
    ev = synth.make_windows(b, n, seed=70 + n)
    xyz = np.ascontiguousarray(ev[:, :3].transpose(0, 2, 1))
    start = synth.make_start_indices(b, n, seed=1)
    fidx = c_oracle.fps(xyz, s, start)
    centres = np.stack([xyz[i, fidx[i]] for i in range(b)])
    xd = dev(xyz)
    packed = _capi.ball_query(xd, _capi.rows_strides(xd), dev(centres), n, radii, ks).cpu().numpy()
    off = 0
    for r, k in zip(radii, ks):
        want = c_oracle.ball_query(r, k, xyz, centres)
        assert np.array_equal(packed[:, :, off:off + k], want), (r, k)
        off += k


# ------------------------------------------------------------------ gather / transpose / MLP ----
def test_index_points_and_gather():
    torch.manual_seed(0)
    B, N, D, S, K = 2, 300, 7, 20, 6
    feats = torch.randn(B, N, D, device=DEV)
    xyz_cf = torch.randn(B, 3, N, device=DEV)
    idx = torch.randint(0, N, (B, S, K), device=DEV)
    got = e2h.index_points(feats, idx)
    want = torch.stack([feats[b][idx[b]] for b in range(B)])
    assert torch.equal(got, want)
    centres = torch.randn(B, S, 3, device=DEV)
    ld = 12
    out = torch.full((B * S * K, ld), float("nan"), device=DEV)
    _capi.group_gather(xyz_cf, _capi.cf_strides(xyz_cf), feats, D, centres, idx.int(), 0, B, N, S, K, out, ld)
    xyz_rows = xyz_cf.permute(0, 2, 1)
    rel = torch.stack([xyz_rows[b][idx[b]] for b in range(B)]) - centres.view(B, S, 1, 3)
    want = torch.cat([want, rel, torch.zeros(B, S, K, ld - D - 3, device=DEV)], -1).view(-1, ld)
    assert torch.equal(out, want)


def test_transpose_roundtrip_and_offsets():
    x = torch.randn(3, 37, 70, device=DEV)[:, 2:35, :]           # strided view [3,33,70]
    rows = torch.empty(3, 70, 40, device=DEV).fill_(-1)
    _capi.transpose(x, (x.stride(0), x.stride(1), x.stride(2)), 3, 33, 70, rows, 70 * 40, 40, 5)
    assert torch.equal(rows[:, :, 5:38], x.permute(0, 2, 1))
    assert (rows[:, :, :5] == -1).all() and (rows[:, :, 38:] == -1).all()


def _torch_mlp_rows(x, convs, pool):
    h = x
    for (w, b, g, be, m, v) in convs:
        h = torch.relu((h @ w.t() + b - m) / torch.sqrt(v + 1e-5) * g + be)
    return h if not pool else h.view(-1, pool, h.shape[-1]).max(1).values


PRECISION_TOL = {"fp32": 1e-5, "tf32x3": 1e-5, "bf16": 1e-2}


@pytest.fixture(params=["fp32", "tf32x3", "bf16"])
def precision(request):
    old = e2h.get_mlp_precision()
    e2h.set_mlp_precision(request.param)
    yield request.param
    e2h.set_mlp_precision(old)


@pytest.mark.parametrize("M,cin,widths,pool", [
    (1000, 8, [32, 32, 64], 0), (64 * 32, 8, [32, 32, 64], 32), (40 * 64, 323, [128, 196, 256], 64),
    (6 * 128, 515, [256, 512, 1024], 128), (5 * 256, 19, [40], 256), (24 * 12, 7, [130], 12), (9 * 20, 5, [33, 17], 20),
    (300 * 128 + 128, 64, [96, 128], 128), (777, 100, [300, 48], 0),
    (1000, 40, [96, 768], 0), (3 * 384, 16, [64, 128], 384), (2000, 33, [64, 32], 0), (1536, 257, [128], 64),
    (32 * 37, 20, [48, 80], 32)])
def test_linear_relu_stack_vs_fp64(M, cin, widths, pool, precision):
    rs = np.random.RandomState(M + cin)
    spec = dict(kind="all", in_channel=cin, mlp=widths)
    st = synth.random_state_for(spec, seed=cin)
    layers_np = [tuple(st[k % j] for k in ("mlp_convs.%d.weight", "mlp_convs.%d.bias", "mlp_bns.%d.weight",
                                           "mlp_bns.%d.bias", "mlp_bns.%d.running_mean", "mlp_bns.%d.running_var"))
                 for j in range(len(widths))]
    x = rs.randn(M, cin).astype(np.float32)
    ld = (cin + 3) // 4 * 4
    xd = torch.zeros(M, ld, device=DEV)
    xd[:, :cin] = dev(x)
    layers = []
    for (w, b, g, be, m, v) in layers_np:
        wt, bias = _capi.fold_conv_bn(dev(w.reshape(w.shape[0], -1)), dev(b), dev(g), dev(be), dev(m), dev(v), 1e-5)
        layers.append({"wt": wt, "bias": bias, "cin": w.shape[1], "cout": w.shape[0], "packed": {}})
    rows_out = M // pool if pool else M
    out = torch.zeros(rows_out, widths[-1], device=DEV)
    from ev2hands_b200.pointnet2_utils import _mlp_rows
    _mlp_rows(xd, M, ld, layers, pool, out, widths[-1], 0)
    layers_t = [tuple(torch.from_numpy(np.asarray(t, dtype=np.float64).reshape(t.shape[0], -1) if i == 0
                                       else np.asarray(t, dtype=np.float64)) for i, t in enumerate(l))
                for l in layers_np]
    want = _torch_mlp_rows(torch.from_numpy(x).double(), layers_t, pool)
    tol = PRECISION_TOL[precision]
    assert rel_err(out, want) <= tol
    if pool and M <= 4096:   # cross-check the C fp64 yardstick on the same rows
        ref64 = c_oracle.mlp_max_f64(x.reshape(-1, pool, cin), layers_np)
        assert rel_err(out, ref64) <= tol


# ------------------------------------------------------------------ modules ---------------------
def _encoder_with(seeds):
    enc = e2h.SetAbstractionEncoder()
    for n, s in zip(("sa1", "sa2", "sa3"), seeds):
        load_numpy_state(getattr(enc, n), synth.random_state_for(synth.ENCODER_SPECS[n], seed=int(s)))
    return enc.to(DEV).eval()


def test_encoder_golden(golden, precision):
    g = golden("encoder")
    FEAT_TOL = PRECISION_TOL[precision]
    enc = _encoder_with(g["weight_seeds"])
    events = dev(g["events"])
    with torch.no_grad():
        out, lv = enc(events, fps_starts=(torch.from_numpy(g["start_sa1"]), torch.from_numpy(g["start_sa2"])),
                      return_levels=True)
    assert np.array_equal(enc.sa1.last_fps_idx.cpu().numpy(), g["fps_sa1"])
    assert np.array_equal(enc.sa2.last_fps_idx.cpu().numpy(), g["fps_sa2"])
    ball2 = enc.sa2.last_ball_idx.cpu().numpy()
    assert np.array_equal(ball2[:, :, :64], g["ball_sa2_r0.4"]) and np.array_equal(ball2[:, :, 64:], g["ball_sa2_r0.8"])
    assert np.array_equal(lv["l1_xyz"].cpu().numpy(), g["l1_xyz"])
    assert np.array_equal(lv["l2_xyz"].cpu().numpy(), g["l2_xyz"])
    assert lv["l1_points"].shape == (2, 320, 512) and lv["l2_points"].shape == (2, 512, 128) and out.shape == (2, 1024)
    assert rel_err(lv["l1_points"][0], g["l1_points_w0"]) <= FEAT_TOL
    assert rel_err(lv["l2_points"][0], g["l2_points_w0"]) <= FEAT_TOL
    assert rel_err(out, g["l3_points"][:, :, 0]) <= FEAT_TOL


def test_regressor_golden(golden, precision):
    g = golden("regressor")
    FEAT_TOL = PRECISION_TOL[precision]
    reg = e2h.RegressorSetAbstraction()
    for n, s in zip(("sa1", "sa2"), g["weight_seeds"]):
        load_numpy_state(getattr(reg, n), synth.random_state_for(synth.REGRESSOR_SPECS[n], seed=int(s)))
    reg = reg.to(DEV).eval()
    events = dev(g["events"])
    with torch.no_grad():
        l1_xyz, l1_points = reg.sa1(events[:, :3, :], dev(g["hand_feats"]), fps_start=torch.from_numpy(g["start_sa1"]))
        _, out = reg.sa2(l1_xyz, l1_points)
    assert np.array_equal(l1_xyz.cpu().numpy(), g["r1_xyz"])
    assert rel_err(l1_points[0], g["r1_points_w0"]) <= FEAT_TOL
    assert rel_err(out, g["r2_points"]) <= FEAT_TOL


def test_encoder_vs_torch_oracle_fresh_inputs():
    seeds = (31, 32, 33)
    enc = _encoder_with(seeds)
    ev = synth.make_windows(3, 2048, seed=2024)
    starts = (torch.from_numpy(synth.make_start_indices(3, 2048, 5)), torch.from_numpy(synth.make_start_indices(3, 512, 6)))
    with torch.no_grad():
        got = enc(dev(ev), fps_starts=starts)
        states = {n: synth.random_state_for(synth.ENCODER_SPECS[n], seed=s) for n, s in zip(("sa1", "sa2", "sa3"), seeds)}
        want, aux = sa_oracle.encoder_forward(states, synth.ENCODER_SPECS, torch.from_numpy(ev),
                                              {"sa1": starts[0], "sa2": starts[1]}, return_aux=True)
    assert np.array_equal(enc.sa1.last_fps_idx.cpu().numpy(), aux["sa1"]["fps_idx"].numpy())
    assert np.array_equal(enc.sa1.last_ball_idx.cpu().numpy(), torch.cat(aux["sa1"]["ball_idx"], -1).numpy())
    assert np.array_equal(enc.sa2.last_ball_idx.cpu().numpy(), torch.cat(aux["sa2"]["ball_idx"], -1).numpy())
    assert rel_err(got, want[:, :, 0]) <= FEAT_TOL


def test_random_start_consumes_cpu_generator_like_reference():
    # without explicit starts the module must draw torch.randint(0, N, (B,)) from the CPU
    # generator, once per Msg layer, in call order (pointnet2_utils.py:75)
    enc = _encoder_with((1, 2, 3))
    ev = dev(synth.make_windows(2, 2048, seed=8))
    torch.manual_seed(123)
    s1 = torch.randint(0, 2048, (2,), dtype=torch.long)
    s2 = torch.randint(0, 512, (2,), dtype=torch.long)
    after = torch.randint(0, 10 ** 6, (1,))
    torch.manual_seed(123)
    with torch.no_grad():
        a = enc(ev)
    assert torch.equal(torch.randint(0, 10 ** 6, (1,)), after)
    with torch.no_grad():
        b = enc(ev, fps_starts=(s1, s2))
    assert torch.equal(a, b)


def test_results_do_not_depend_on_sharding_or_chunking(monkeypatch):
    enc = _encoder_with((4, 5, 6))
    ev = dev(synth.make_windows(6, 2048, seed=77))
    s1 = torch.from_numpy(synth.make_start_indices(6, 2048, 1))
    s2 = torch.from_numpy(synth.make_start_indices(6, 512, 2))
    with torch.no_grad():
        whole = enc(ev, fps_starts=(s1, s2))
        parts = torch.cat([enc(ev[i:i + 2], fps_starts=(s1[i:i + 2], s2[i:i + 2])) for i in (0, 2, 4)])
    assert torch.equal(whole, parts)
    from ev2hands_b200 import pointnet2_utils as pu
    monkeypatch.setattr(pu, "_WORKSPACE_BYTES", 48 << 20)       # forces several chunks per scale
    with torch.no_grad():
        chunked = enc(ev, fps_starts=(s1, s2))
    assert torch.equal(whole, chunked)


def test_row_chaining_between_layers_and_side_stream(monkeypatch, precision):
    """The encoder's inference path hands each layer's point-major rows to the next and runs sa2's FPS + ball
    query on a second stream; the module-by-module calls of the reference's API take the same shortcut through
    the record riding on the returned tensor.  All of it must give the same results as feeding plain
    channel-first tensors, and an in-place edit of the tensor must drop the shortcut."""
    from ev2hands_b200 import encoder as enc_mod
    tol = PRECISION_TOL[precision]
    enc = _encoder_with((7, 8, 9))
    ev = dev(synth.make_windows(3, 2048, seed=99))
    s1 = torch.from_numpy(synth.make_start_indices(3, 2048, 3))
    s2 = torch.from_numpy(synth.make_start_indices(3, 512, 4))
    with torch.no_grad():
        fast, lv = enc(ev, fps_starts=(s1, s2), return_levels=True)
        monkeypatch.setattr(enc_mod, "_GEOM_STREAM", False)
        one_stream = enc(ev, fps_starts=(s1, s2))
        assert torch.equal(fast, one_stream)
        # module by module, the way TEHNet.forward calls them (TEHNet.py:172-181): shortcut through the riding record
        l1_xyz, l1_points = enc.sa1(ev[:, :3, :], ev, fps_start=s1)
        assert getattr(l1_points, "_ev2h_rows", None) is not None
        l2_xyz, l2_points = enc.sa2(l1_xyz, l1_points, fps_start=s2)
        _, l3 = enc.sa3(l2_xyz, l2_points)
        assert torch.equal(l1_points, lv["l1_points"]) and torch.equal(l2_points, lv["l2_points"])
        assert torch.equal(l3.squeeze(-1), fast)
        # plain tensors (no record): the layers transpose them themselves; same values up to the summation order
        # of sa3's first layer (its input channels arrive as [xyz | points] instead of [points | xyz])
        p1 = l1_points.clone()
        l2_xyz_b, l2_points_b = enc.sa2(l1_xyz.clone(), p1, fps_start=s2)
        assert torch.equal(l2_xyz_b, l2_xyz) and torch.equal(l2_points_b, l2_points)
        _, l3_b = enc.sa3(l2_xyz_b, l2_points_b.clone())
        assert rel_err(l3_b, l3) <= tol
        # an in-place edit makes the record stale: the edited tensor is what must be consumed
        l1_points.mul_(0.5)
        _, l2_half = enc.sa2(l1_xyz, l1_points, fps_start=s2)
        _, l2_want = enc.sa2(l1_xyz, l1_points.clone(), fps_start=s2)
        assert torch.equal(l2_half, l2_want) and not torch.equal(l2_half, l2_points)


def test_full_size_properties_batch64():
    """BASELINE config 2 (B=64, N=2048): size-independent properties instead of an oracle run."""
    B, N = 64, 2048
    enc = _encoder_with((7, 8, 9))
    ev = dev(synth.make_windows(B, N, seed=1234 + 2))
    s1 = torch.from_numpy(synth.make_start_indices(B, N, 0))
    s2 = torch.from_numpy(synth.make_start_indices(B, 512, 1))
    with torch.no_grad():
        out, lv = enc(ev, fps_starts=(s1, s2), return_levels=True)
    assert out.shape == (B, 1024) and torch.isfinite(out).all() and (out >= 0).all()
    fidx = enc.sa1.last_fps_idx.long()
    assert torch.equal(fidx[:, 0].cpu(), s1)
    xyz = ev[:, :3, :].permute(0, 2, 1).contiguous()
    centres = torch.gather(xyz, 1, fidx.unsqueeze(-1).expand(-1, -1, 3))
    # FPS never re-picks a location until all distinct locations are used: selected points are distinct
    # coordinates as long as the running min-distance is positive; check distinctness of the first 256
    c = centres[:, :256]
    same = (c[:, :, None, :] == c[:, None, :, :]).all(-1)
    assert int(same.sum()) == B * 256                                  # only the diagonal
    # ball query: every listed neighbour is inside the radius under the reference's own distance
    # expression, lists are ascending until the padding starts, padding repeats the first entry
    ball = enc.sa1.last_ball_idx.long()
    sq = e2h.square_distance(centres[:4], xyz[:4])                      # [4,512,2048]
    off = 0
    for r, k in zip([0.1, 0.2, 0.4], [32, 64, 128]):
        nb = ball[:4, :, off:off + k]
        dn = torch.gather(sq, 2, nb)
        assert (dn <= _capi.radius_sq_f32(r)).all()
        inside = (sq <= _capi.radius_sq_f32(r)).sum(-1)
        n_real = inside.clamp(max=k)
        ar = torch.arange(k, device=DEV).view(1, 1, k)
        real = ar < n_real.unsqueeze(-1)
        inc = (nb[:, :, 1:] > nb[:, :, :-1]) | ~real[:, :, 1:]
        assert inc.all()
        assert torch.equal(torch.where(real, nb, nb[:, :, :1].expand_as(nb)), nb)
        off += k
    # windows 0..3 of the batch agree with running them alone (no cross-window leakage)
    with torch.no_grad():
        alone = enc(ev[:4], fps_starts=(s1[:4], s2[:4]))
    assert torch.equal(out[:4], alone)


# ------------------------------------------------------------------ training path ---------------
def test_group_max_forward_backward_vs_torch():
    torch.manual_seed(1)
    x = torch.randn(2, 9, 16, 11, device=DEV)
    x[0, 0, :, 0] = 0.0                         # all-equal column: first index wins, like torch.max
    x[1, 3, 5, 2] = x[1, 3, 7, 2] = 9.0         # duplicated maximum
    xa = x.clone().requires_grad_(True)
    xb = x.clone().requires_grad_(True)
    from ev2hands_b200.pointnet2_utils import _GroupMax
    ya = _GroupMax.apply(xa)
    yb = xb.max(dim=2).values
    assert torch.equal(ya, yb)
    g = torch.randn_like(ya)
    ya.backward(g)
    yb.backward(g)
    assert torch.equal(xa.grad, xb.grad)


@pytest.fixture
def strict_fp32():
    """stock torch ops as an fp32 reference: cuDNN / cuBLAS may otherwise run convolutions and GEMMs in plain tf32"""
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def test_train_mode_forward_backward_matches_torch_autograd(strict_fp32):
    torch.manual_seed(0)
    m = e2h.PointNetSetAbstractionMsg(32, [0.4, 0.8], [8, 16], 6, [[16, 24], [16, 32]]).to(DEV).train()
    B, N = 3, 256
    ev = dev(synth.make_windows(B, N, seed=5))
    xyz = ev[:, :3, :]
    feats = torch.randn(B, 6, N, device=DEV, requires_grad=True)
    start = torch.from_numpy(synth.make_start_indices(B, N, 3))
    new_xyz, out = m(xyz, feats, fps_start=start)
    loss = (out * torch.linspace(0.5, 1.5, out.numel(), device=DEV).view_as(out)).sum()
    loss.backward()
    got = {n: p.grad.clone() for n, p in m.named_parameters()}
    got_in = feats.grad.clone()
    got_rm = m.bn_blocks[0][0].running_mean.clone()

    # the same computation with stock torch ops on the same indices
    import copy
    ref = copy.deepcopy(m)
    for bnb in ref.bn_blocks:
        for bn in bnb:
            bn.reset_running_stats()
    ref.zero_grad()
    feats2 = feats.detach().clone().requires_grad_(True)
    xyz_rows = xyz.permute(0, 2, 1)
    centres = new_xyz.permute(0, 2, 1)
    ball = m.last_ball_idx.long()
    pooled, off = [], 0
    for i, K in enumerate([8, 16]):
        gi = ball[:, :, off:off + K]
        fr = feats2.permute(0, 2, 1)
        gp = torch.stack([fr[b][gi[b]] for b in range(B)])
        gx = torch.stack([xyz_rows[b][gi[b]] for b in range(B)]) - centres.view(B, 32, 1, 3)
        h = torch.cat([gp, gx], -1).permute(0, 3, 2, 1)
        for conv, bn in zip(ref.conv_blocks[i], ref.bn_blocks[i]):
            h = torch.relu(bn(conv(h)))
        pooled.append(h.max(2).values)
        off += K
    out2 = torch.cat(pooled, 1)
    assert rel_err(out, out2) <= 1e-5
    (out2 * torch.linspace(0.5, 1.5, out2.numel(), device=DEV).view_as(out2)).sum().backward()
    ref_grads = dict((n, p.grad) for n, p in ref.named_parameters())
    for n, g in ref_grads.items():
        if n.startswith("conv_blocks") and n.endswith(".bias"):
            # a bias in front of a train-mode BatchNorm cancels in (x - mean): its exact gradient is zero and what
            # either side computes is rounding noise of its own summation order - compare it with the scale of the
            # layer's weight gradient instead of with the other side's noise
            scale = float(ref_grads[n[:-4] + "weight"].abs().max())
            assert float(got[n].abs().max()) <= 1e-3 * scale and float(g.abs().max()) <= 1e-3 * scale, n
        else:
            assert rel_err(got[n], g) <= 1e-4, n
    assert rel_err(got_in, feats2.grad) <= 1e-4
    assert rel_err(got_rm, ref.bn_blocks[0][0].running_mean) <= 1e-5


# ------------------------------------------------------------------ long windows (config 5) ------
def test_long_window_16k_fp32_vs_bf16_and_oracle_indices():
    """BASELINE config 5 shape (16384-event windows, small batch here): indices bit-exact against the
    C oracle, 3xTF32 features within 1e-5 of the exact-fp32 CUDA path, bf16 variant within 1e-2."""
    B, N = 3, 16384
    enc = _encoder_with((11, 12, 13))
    ev_np = synth.make_windows(B, N, seed=555)
    ev = dev(ev_np)
    s1 = torch.from_numpy(synth.make_start_indices(B, N, 2))
    s2 = torch.from_numpy(synth.make_start_indices(B, 512, 3))
    outs = {}
    old = e2h.get_mlp_precision()
    try:
        for prec in ("fp32", "tf32x3", "bf16"):
            e2h.set_mlp_precision(prec)
            with torch.no_grad():
                outs[prec] = enc(ev, fps_starts=(s1, s2))
            if prec == "fp32":
                xyz = np.ascontiguousarray(ev_np[:, :3].transpose(0, 2, 1))
                fidx = c_oracle.fps(xyz, 512, s1.numpy())
                assert np.array_equal(enc.sa1.last_fps_idx.cpu().numpy(), fidx)
                centres = np.stack([xyz[b, fidx[b]] for b in range(B)])
                ball = enc.sa1.last_ball_idx.cpu().numpy()
                off = 0
                for r, k in zip([0.1, 0.2, 0.4], [32, 64, 128]):
                    assert np.array_equal(ball[:, :, off:off + k], c_oracle.ball_query(r, k, xyz, centres)), r
                    off += k
    finally:
        e2h.set_mlp_precision(old)
    assert rel_err(outs["tf32x3"], outs["fp32"]) <= 1e-5
    assert rel_err(outs["bf16"], outs["fp32"]) <= 1e-2


# ---- decoder: feature propagation (SURVEY 8f row N1) -------------------------------------------------------

def _decoder_with(seeds):
    dec = e2h.FeaturePropagationDecoder()
    for n, s in zip(("fp3", "fp2", "fp1"), seeds):
        load_numpy_state(getattr(dec, n), synth.random_state_for(synth.DECODER_SPECS[n], seed=int(s)))
    return dec.to(DEV).eval()


def test_decoder_golden(golden, precision):
    """fp3 -> fp2 -> fp1 against the reference's own outputs: 3-NN indices bit-exact, weights and features
    within the precision's bar."""
    e, g = golden("encoder"), golden("decoder")
    FEAT_TOL = PRECISION_TOL[precision]
    dec = _decoder_with(g["weight_seeds"])
    f1, f2, f3 = (dev(a) for a in synth.decoder_test_features(2, seed=int(g["feature_seed"])))
    ev = dev(e["events"])
    with torch.no_grad():
        d0, d1, d2 = dec(ev[:, :3, :], dev(e["l1_xyz"]), dev(e["l2_xyz"]), dev(e["l3_xyz"]), f1, f2, f3, return_levels=True)
    for tag, fp in (("fp2", dec.fp2), ("fp1", dec.fp1)):
        assert np.array_equal(fp.last_idx.cpu().numpy(), g[tag + "_idx"].astype(np.int32))
        assert rel_err(fp.last_weight, g[tag + "_weight"]) <= 1e-6
    assert rel_err(d2, g["d2"]) <= FEAT_TOL
    assert rel_err(d1[:, :, ::2], g["d1_every2"]) <= FEAT_TOL
    assert rel_err(d0[:, :, ::16], g["d0_every16"]) <= FEAT_TOL


def test_three_nn_matches_c_free_oracle_on_ragged_sizes():
    """3-NN + weights against the torch oracle for sizes that are not multiples of the CTA / tile sizes,
    a strided (non-contiguous) query view, and exact duplicates among the sources (ties keep the lower index)."""
    rs = np.random.RandomState(5)
    for B, N, S in ((1, 1, 3), (2, 130, 7), (3, 257, 1025), (1, 2048, 512)):
        q = rs.rand(B, 5, N).astype(np.float32)
        src = rs.rand(B, 3, S).astype(np.float32)
        if S >= 7:
            src[:, :, 5] = src[:, :, 2]                      # duplicate source point
        qd = dev(q)[:, :3, :]                                # strided view, like xyz[:, :3, :] in the model
        idx, w = _capi.three_nn(qd, dev(src))
        want_i, want_w = sa_oracle.three_nn_weights(torch.from_numpy(q[:, :3, :]).permute(0, 2, 1).contiguous(),
                                                    torch.from_numpy(src).permute(0, 2, 1).contiguous())
        wi = want_i.numpy()
        gi = idx.cpu().numpy().astype(np.int64)
        if not np.array_equal(gi, wi):                      # only exact ties may be ordered differently by torch's sort
            d = sa_oracle.pairwise_sqdist(torch.from_numpy(q[:, :3, :]).permute(0, 2, 1).contiguous(),
                                          torch.from_numpy(src).permute(0, 2, 1).contiguous()).numpy()
            bad = np.argwhere(gi != wi)
            for b, n, k in bad:
                assert d[b, n, gi[b, n, k]] == d[b, n, wi[b, n, k]]
        assert rel_err(w, want_w.numpy()) <= 1e-6


def test_feature_propagation_train_mode_matches_eval_formulation():
    """The training (autograd) path and the CUDA path are the same function: compare them in eval mode with
    gradients enabled vs disabled."""
    dec = _decoder_with((7, 8, 9))
    rs = np.random.RandomState(3)
    xyz1, xyz2 = dev(rs.rand(2, 3, 300).astype(np.float32)), dev(rs.rand(2, 3, 40).astype(np.float32))
    p1, p2 = dev(rs.randn(2, 320, 300).astype(np.float32)), dev(rs.randn(2, 256, 40).astype(np.float32))
    with torch.no_grad():
        fast = dec.fp2(xyz1, xyz2, p1, p2)
    p1g = p1.clone().requires_grad_(True)
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False          # cuDNN would otherwise run the Conv1d stack in plain tf32
    try:
        slow = dec.fp2(xyz1, xyz2, p1g, p2)
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert slow.requires_grad
    assert rel_err(fast, slow.detach().cpu().numpy()) <= 1e-5


# ---- row compaction: skipping the padded duplicate neighbours must not change a single bit ------------------

def test_compacted_rows_are_bit_identical_to_dense(precision):
    import ev2hands_b200.pointnet2_utils as pu
    if precision == "fp32":
        pytest.skip("the fp32 path is layer by layer, not the fused kernel")
    enc = _encoder_with((41, 42, 43))
    ev = dev(synth.make_windows(5, 2048, seed=77))
    starts = (torch.from_numpy(synth.make_start_indices(5, 2048, 8)), torch.from_numpy(synth.make_start_indices(5, 512, 9)))
    outs = {}
    old = (pu._COMPACT, pu._DEDUP)
    try:
        for flags in ((False, False), (True, False), (True, True)):       # dense / compacted / compacted + duplicate points once
            pu._COMPACT, pu._DEDUP = flags
            with torch.no_grad():
                l3, lv = enc(ev, fps_starts=starts, return_levels=True)
            outs[flags] = (l3.cpu().numpy(), lv["l1_points"].cpu().numpy(), lv["l2_points"].cpu().numpy())
    finally:
        pu._COMPACT, pu._DEDUP = old
    for flags in ((True, False), (True, True)):
        for a, b in zip(outs[(False, False)], outs[flags]):
            assert np.array_equal(a, b)


def test_first_occurrence_and_deduplicated_ball_query():
    rs = np.random.RandomState(9)
    B, N, S = 3, 900, 40
    base = rs.rand(B, 300, 8).astype(np.float32)
    base[:, :, 7] = 0
    pick = rs.randint(0, 300, size=(B, N))
    pts8 = np.stack([base[b][pick[b]] for b in range(B)])                 # sampling with replacement: many exact copies
    first = _capi.first_occurrence(dev(pts8)).cpu().numpy()
    want_first = np.zeros((B, N), dtype=np.uint8)
    for b in range(B):
        seen = set()
        for n in range(N):
            key = pts8[b, n].tobytes()
            if key not in seen:
                seen.add(key); want_first[b, n] = 1
    assert np.array_equal(first, want_first)
    xyz = np.ascontiguousarray(pts8[:, :, 4:7].transpose(0, 2, 1))
    centres = np.ascontiguousarray(pts8[:, :S, 4:7])
    Ks, radii = [8, 32], [0.2, 0.45]
    xd = dev(xyz)
    idx, uniq, ucnt = _capi.ball_query_uniq(xd, _capi.cf_strides(xd), dev(centres), N, radii, Ks, dev(first))
    idx2 = _capi.ball_query(xd, _capi.cf_strides(xd), dev(centres), N, radii, Ks)
    assert torch.equal(idx, idx2)                                       # the reference list is unchanged
    idx_h, uniq_h, ucnt_h = idx.cpu().numpy(), uniq.cpu().numpy(), ucnt.cpu().numpy()
    k_off = 0
    for i, K in enumerate(Ks):
        for b in range(B):
            for s in range(S):
                blk = idx_h[b, s, k_off:k_off + K]
                real = len(np.unique(blk))                               # ascending + padded with the first: distinct = real hits
                hits = blk[:real]
                want = [int(h) for h in hits if want_first[b, h]]
                assert ucnt_h[i, b, s] == len(want)
                assert list(uniq_h[b, s, k_off:k_off + len(want)]) == want
        k_off += K


def test_compaction_tables_match_a_numpy_restatement():
    rs = np.random.RandomState(2)
    B, N, S = 3, 700, 50
    xyz = rs.rand(B, 3, N).astype(np.float32)
    xyz[:, :, 10] = 5.0                                             # a far-away centre: alone in its ball
    centres_idx = np.stack([np.concatenate([[10], rs.choice(N, S - 1, replace=False)]) for _ in range(B)])
    centres = np.stack([xyz[b][:, centres_idx[b]].T for b in range(B)]).astype(np.float32)
    Ks = [8, 32, 64]
    xd = dev(xyz)
    idx, cnt = _capi.ball_query(xd, _capi.cf_strides(xd), dev(centres), N, [0.05, 0.15, 0.3], Ks, with_counts=True)
    rowmaps, blockgroups, n_rows = _capi.group_compact(idx, cnt, N, Ks)
    idx_h, cnt_h, n_rows_h = idx.cpu().numpy(), cnt.cpu().numpy(), n_rows.cpu().numpy()
    k_off = 0
    for i, K in enumerate(Ks):
        # counts: number of distinct leading entries before the padding (= entries != first after position 0, + 1)
        blk_all = idx_h[:, :, k_off:k_off + K]
        want_cnt = np.array([[len(np.unique(blk_all[b, s])) for s in range(S)] for b in range(B)])
        assert np.array_equal(cnt_h[i], want_cnt)
        # groups are appended in no particular order: rebuild {group: rows} from the tables and compare per group
        total = int(n_rows_h[i])
        rm_h, bg_h = rowmaps[i].cpu().numpy()[:total], blockgroups[i].cpu().numpy()[:total // 8]
        assert total % 8 == 0
        got = {}
        for blk, g in enumerate(bg_h):
            got.setdefault(int(g), []).extend(rm_h[8 * blk:8 * blk + 8].tolist())
        # every group's blocks are contiguous
        changes = 1 + int((bg_h[1:] != bg_h[:-1]).sum())
        assert changes == len(got) == B * S
        want_total = 0
        for g in range(B * S):
            b, s = divmod(g, S)
            c = max(int(want_cnt[b, s]), 1)
            rows = (c + 7) // 8 * 8
            want_total += rows
            assert got[g] == [b * N + int(blk_idx) for blk_idx in (blk_all[b, s, [k if k < c else 0 for k in range(rows)]])]
        assert total == want_total
        k_off += K


def test_ball_query_with_in_kernel_compaction_matches_the_two_step_tables():
    """ev2h_ball_query_compact_f32 = ball query + ev2h_group_compact_i32 in one kernel: same index lists, and the same
    set of rows per group (groups land in the list in no particular order in both)."""
    rs = np.random.RandomState(12)
    B, N, S = 2, 1500, 70
    base = rs.rand(B, 500, 8).astype(np.float32)
    base[:, :, 7] = 0
    pts8 = np.stack([base[b][rs.randint(0, 500, size=N)] for b in range(B)])
    xyz = np.ascontiguousarray(pts8[:, :, 4:7].transpose(0, 2, 1))
    centres = np.ascontiguousarray(pts8[:, :S, 4:7])
    Ks, radii = [16, 64, 128], [0.1, 0.3, 0.6]
    xd, cd = dev(xyz), dev(centres)
    strides = _capi.cf_strides(xd)
    for dedup in (False, True):
        first = _capi.first_occurrence(dev(pts8)) if dedup else None
        idx, rowmaps, blockgroups, n_rows = _capi.ball_query_compact(xd, strides, cd, N, radii, Ks, first)
        if dedup:
            idx2, lists, cnt = _capi.ball_query_uniq(xd, strides, cd, N, radii, Ks, first)
        else:
            idx2, cnt = _capi.ball_query(xd, strides, cd, N, radii, Ks, with_counts=True)
            lists = idx2
        assert torch.equal(idx, idx2)
        rm2, bg2, n2 = _capi.group_compact(lists, cnt, N, Ks)
        assert torch.equal(n_rows, n2)
        for i in range(len(Ks)):
            total = int(n_rows[i])
            def per_group(rm, bg):
                rm, bg = rm.cpu().numpy()[:total], bg.cpu().numpy()[:total // 8]
                d = {}
                for blk, g in enumerate(bg):
                    d.setdefault(int(g), []).extend(rm[8 * blk:8 * blk + 8].tolist())
                return d
            assert per_group(rowmaps[i], blockgroups[i]) == per_group(rm2[i], bg2[i])


# ------------------------------------------------------------------ event windows (SURVEY 8f N3) ----
def _window_case(golden, case):
    g = golden("windows")
    return (g[case + "_events"], g[case + "_starts"], g[case + "_counts"], g[case + "_idx"], g[case + "_windows"], g[case + "_M"])


@pytest.mark.parametrize("case,mode", [("stream", "stream"), ("erpc", "erpc"), ("erpct", "erpc"), ("erpcpad", "erpc")])
def test_event_windows_golden(golden, case, mode):
    """ev2h_window_aggregate_f64 + ev2h_window_sample_f32 against what the reference's own dataset classes
    produced from the same raw events and the same draw: bit for bit ("erpct": where equal mean times leave
    the reference's unstable argsort a choice, time and every untied point)."""
    from oracle import window_oracle as wo
    ev, starts, counts, idx, want, M = _window_case(golden, case)
    wb = e2h.EventWindowBuilder(mode)
    got = wb(torch.from_numpy(ev).to(DEV), starts, counts, sample_idx=torch.from_numpy(idx), check=True)
    assert np.array_equal(wb.last_n_pixels.cpu().numpy(), M)
    got = got.cpu().numpy()
    assert got.shape == want.shape
    if case == "erpct":
        for b, (s, c) in enumerate(zip(starts, counts)):
            rec = wo.aggregate(ev[s:s + c], mode)
            tt = rec[:, 2]
            u, cn = np.unique(tt, return_counts=True)
            keep = ~np.isin(tt, u[cn > 1])[idx[b]]
            assert np.array_equal(got[b, 2], want[b, 2]) and np.array_equal(got[b][:, keep], want[b][:, keep])
        # and all of it against the oracle, whose sort is stable like the kernel's
        assert np.array_equal(got, wo.build_windows(ev, starts, counts, idx, mode))
    else:
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_event_windows_draw_like_the_reference(golden):
    """without explicit indices the builder draws np.random.choice(M, N) per window from numpy's global generator"""
    ev, starts, counts, idx, want, M = _window_case(golden, "stream")
    wb = e2h.EventWindowBuilder("stream")
    np.random.seed(5)                     # the seed tests/golden/make_window_golden.py used
    got = wb(torch.from_numpy(ev).to(DEV), starts, counts)
    assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32))
    # sampling=False (erpc.py:219-226): every pixel once, then the missing n_events - M drawn
    ev, starts, counts, idx, want, M = _window_case(golden, "erpcpad")
    wb = e2h.EventWindowBuilder("erpc", sampling=False)
    np.random.seed(8)
    got = wb(torch.from_numpy(ev).to(DEV), starts, counts)
    assert np.array_equal(got.cpu().numpy().view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("mode,n_max", [("stream", 16384), ("stream", 700), ("erpc", 4096), ("erpc", 33)])
def test_event_windows_ragged_vs_oracle(mode, n_max):
    """ragged batches up to the largest supported window, overlapping windows, hot pixels (long runs), a single
    event, negative and huge timestamps - records and windows against the oracle, bit for bit"""
    from oracle import window_oracle as wo
    rs = np.random.RandomState(n_max)
    ev = synth.make_raw_events(3 * n_max + 50, seed=n_max, t0=-2.5e5 if mode == "stream" else 7.0e9, duration=6.0e5,
                               extra_columns=2 if mode == "erpc" else 0)
    ev[10:10 + n_max // 3, :2] = (17, 200)                  # a hot pixel: one long run
    ev[5, 3] = 2.0                                          # polarity that is neither 0 nor 1 counts as negative
    starts = np.array([0, 7, n_max, 2 * n_max + 49, 3])
    counts = np.array([n_max, max(1, n_max // 2), n_max - 1, 1, 2])
    wb = e2h.EventWindowBuilder(mode, n_events=777)
    rec, n_pix, n_bad = wb.aggregate(torch.from_numpy(ev).to(DEV), starts, counts)
    want_rec = [wo.aggregate(ev[s:s + c], mode) for s, c in zip(starts, counts)]
    assert n_pix.cpu().tolist() == [r.shape[0] for r in want_rec] and int(n_bad.sum()) == 0
    for b, r in enumerate(want_rec):
        assert np.array_equal(rec[b, :r.shape[0]].cpu().numpy().view(np.uint32), r.view(np.uint32)), b
    idx = np.stack([rs.randint(0, r.shape[0], size=777) for r in want_rec])
    got = wb.sample(rec, n_pix, n_bad, torch.from_numpy(idx)).cpu().numpy()
    want = wo.build_windows(ev, starts, counts, idx, mode)
    assert np.array_equal(got, want, equal_nan=True)        # the 1-event window is NaN in t (0/0) there too
    assert np.isnan(got[3, 2]).all() and not np.isnan(got[[0, 1, 2]]).any()
    if mode == "stream":        # ("erpc" at 7e9 ns: the two events' mean times are one float32, NaN like the reference)
        assert not np.isnan(got[4]).any()


def test_event_windows_errors_and_out_of_sensor_events():
    ev = synth.make_raw_events(300, seed=3)
    ev[7, 0] = 346.0          # one column past the sensor
    ev[9, 1] = -1.0
    wb = e2h.EventWindowBuilder("stream", n_events=64)
    d = torch.from_numpy(ev).to(DEV)
    rec, n_pix, n_bad = wb.aggregate(d, [0], [300])
    assert n_bad.cpu().tolist() == [2]
    with pytest.raises(IndexError):
        wb(d, [0], [300], check=True)
    with pytest.raises(IndexError):
        wb.aggregate(d, [200], [101])
    with pytest.raises(RuntimeError):
        wb.aggregate(torch.from_numpy(ev), [0], [300])              # host tensor: no CPU path
    with pytest.raises(RuntimeError, match="exceed"):
        e2h.EventWindowBuilder("erpc").aggregate(torch.zeros((5000, 4), dtype=torch.float64, device=DEV), [0], [5000])
    bad_idx = torch.full((1, 64), 10 ** 6, dtype=torch.int64)
    wb.sample(rec, n_pix, n_bad, bad_idx)
    assert int(n_bad[0]) == 2 + 64


def test_event_windows_feed_the_encoder(golden):
    """raw events -> windows -> encoder, all on the device: same features as the encoder on the reference's window"""
    ev, starts, counts, idx, want, M = _window_case(golden, "stream")
    enc = _encoder_with((1, 2, 3))
    wb = e2h.EventWindowBuilder("stream")
    wins = wb(torch.from_numpy(ev).to(DEV), starts, counts, sample_idx=torch.from_numpy(idx))
    s1 = torch.from_numpy(synth.make_start_indices(3, 2048, 0))
    s2 = torch.from_numpy(synth.make_start_indices(3, 512, 1))
    with torch.no_grad():
        a = enc(wins, fps_starts=(s1, s2))
        b = enc(dev(want), fps_starts=(s1, s2))
    assert torch.equal(a, b)


def test_event_windows_sharded_equal_the_whole_batch():
    """sharding.shard_windows: every rank builds its windows from its own slice of the event table; the union is
    bit-identical to the unsharded batch (the draws are made for the global batch and sliced with the windows)."""
    from ev2hands_b200 import sharding
    ev = synth.make_raw_events(9000, seed=31)
    starts = np.array([0, 300, 900, 1500, 1501, 2500, 1900, 6000, 6100])
    counts = np.array([2048, 700, 2600, 900, 10, 1500, 64, 2999, 2048])
    wb = e2h.EventWindowBuilder("stream", n_events=512)
    rec, n_pix, n_bad = wb.aggregate(torch.from_numpy(ev).to(DEV), starts, counts)
    m = n_pix.cpu().numpy()
    idx = np.stack([np.random.RandomState(b).randint(0, m[b], size=512) for b in range(len(m))])
    whole = wb.sample(rec, n_pix, n_bad, torch.from_numpy(idx)).cpu().numpy()
    for world in (2, 4):
        parts = []
        for rank in range(world):
            row_lo, row_hi, ls, lc, (lo, hi) = sharding.shard_windows(starts, counts, rank, world)
            local = torch.from_numpy(ev[row_lo:row_hi]).to(DEV)            # the only rows this rank uploads
            parts.append(wb(local, ls, lc, sample_idx=torch.from_numpy(idx[lo:hi]), check=True).cpu().numpy())
        assert np.array_equal(np.concatenate(parts), whole)


def test_event_windows_full_size_properties_batch1024():
    """config-3-sized batch (1024 half-overlapping windows of 2048 events): size-independent properties instead
    of an oracle run - pixel counts against numpy, every output point is one of its window's pixels with that
    pixel's event counts, x / y / t normalised into [-1, 1] with t touching both ends."""
    B, n, N = 1024, 2048, 2048
    ev = synth.make_raw_events(B * n // 2 + n, seed=41, duration=2.0e3 * (B // 2 + 1))
    starts, counts = np.arange(B) * (n // 2), np.full(B, n)
    wb = e2h.EventWindowBuilder("stream", n_events=N)
    np.random.seed(123)
    out = wb(torch.from_numpy(ev).to(DEV), starts, counts, check=True).cpu().numpy()
    m = wb.last_n_pixels.cpu().numpy()
    pix = (ev[:, 1].astype(np.int64) * 346 + ev[:, 0].astype(np.int64))
    assert out.shape == (B, 5, N) and int(wb.last_n_bad.sum()) == 0
    assert np.abs(out[:, :3]).max() <= 1.0 and (out[:, 2].min(1) == -1.0).all() and (out[:, 2].max(1) == 1.0).all()
    for b in range(0, B, 37):
        w_pix = pix[starts[b]:starts[b] + n]
        uniq, cnt = np.unique(w_pix, return_counts=True)
        assert m[b] == uniq.size
        # invert the normalisation: 2 * (v / size) - 1 in float32
        gx = (2 * (np.arange(346, dtype=np.float32) / np.float32(346)) - 1).astype(np.float32)
        gy = (2 * (np.arange(260, dtype=np.float32) / np.float32(260)) - 1).astype(np.float32)
        xi, yi = np.searchsorted(gx, out[b, 0]), np.searchsorted(gy, out[b, 1])
        assert np.array_equal(gx[xi], out[b, 0]) and np.array_equal(gy[yi], out[b, 1])
        got_pix = yi.astype(np.int64) * 346 + xi
        pos = np.searchsorted(uniq, got_pix)
        assert np.array_equal(uniq[pos], got_pix)                        # a pixel of this window
        assert np.array_equal(out[b, 3] + out[b, 4], cnt[pos].astype(np.float32))   # with that pixel's event count
    for b in range(B):
        assert m[b] == np.unique(pix[starts[b]:starts[b] + n]).size
