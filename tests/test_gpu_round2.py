"""Round-2 parity tests of the CUDA path (through the C ABI): the holes VERDICT r01 listed.

  * config 5 (N = 16384) and config 2 (B = 64) FEATURES against the oracle, not against the kernels themselves
  * sample_and_group / the sampled PointNetSetAbstraction (SURVEY 8a row a5) against the reference's outputs
  * the module-by-module call sequence of TEHNet.forward (TEHNet.py:172-181) with tensors edited between layers
  * the oracle run on the GPU (cuBLAS rounding) against the CPU oracle and the kernels (SURVEY 8c caveat 4)
  * training step at the model's shapes against the reference's own autograd (golden from the reference)
  * CUDA-graph capture refuses host-drawn FPS start indices; start indices are range checked
All tests here need a GPU."""
import json
import os

import numpy as np
import pytest
import torch

import ev2hands_b200 as e2h
from ev2hands_b200 import _capi, synth
from ev2hands_b200.encoder import GraphedForward, load_numpy_state
from oracle import c_oracle, sa_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FEAT_TOL = 1e-5     # max|got - want| <= FEAT_TOL * max|want| per tensor (fp32-level paths)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def rel_err(got, want):
    got = got.detach().cpu().double().numpy() if torch.is_tensor(got) else np.asarray(got, dtype=np.float64)
    want = want.detach().cpu().double().numpy() if torch.is_tensor(want) else np.asarray(want, dtype=np.float64)
    return np.abs(got - want).max() / max(np.abs(want).max(), 1e-30)


def _states(seeds):
    return {n: synth.random_state_for(synth.ENCODER_SPECS[n], seed=int(s)) for n, s in zip(("sa1", "sa2", "sa3"), seeds)}


def _encoder_with(seeds):
    enc = e2h.SetAbstractionEncoder()
    for n, st in _states(seeds).items():
        load_numpy_state(getattr(enc, n), st)
    return enc.to(DEV).eval()


def _record(name, payload):
    """keep a measured outcome next to the run (gpurun_out/ travels back from the GPU box)"""
    d = os.path.join(ROOT, "gpurun_out")
    try:
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, name), "w") as f:
            json.dump(payload, f, indent=1)
    except OSError:
        pass


# ------------------------------------------------------------------ config 5: features vs the oracle ---------
@pytest.mark.parametrize("prec,tol", [("fp32", 1e-5), ("tf32x3", 1e-5), ("bf16", 1e-2)])
def test_long_window_16k_features_vs_oracle(prec, tol):
    """BASELINE config 5 shape (16384-event windows): encoder features of the CUDA path against the torch-CPU
    oracle run window by window (SURVEY 8c caveat 2), every level, not CUDA against CUDA."""
    B, N = 2, 16384
    seeds = (11, 12, 13)
    enc = _encoder_with(seeds)
    ev_np = synth.make_windows(B, N, seed=556)
    s1 = torch.from_numpy(synth.make_start_indices(B, N, 2))
    s2 = torch.from_numpy(synth.make_start_indices(B, 512, 3))
    old = e2h.get_mlp_precision()
    try:
        e2h.set_mlp_precision(prec)
        with torch.no_grad():
            got, lv = enc(dev(ev_np), fps_starts=(s1, s2), return_levels=True)
    finally:
        e2h.set_mlp_precision(old)
    states = _states(seeds)
    for b in range(B):
        with torch.no_grad():
            want, aux = sa_oracle.encoder_forward(states, synth.ENCODER_SPECS, torch.from_numpy(ev_np[b:b + 1]),
                                                  {"sa1": s1[b:b + 1], "sa2": s2[b:b + 1]}, return_aux=True)
        assert np.array_equal(enc.sa1.last_fps_idx[b].cpu().numpy(), aux["sa1"]["fps_idx"][0].numpy())
        assert np.array_equal(enc.sa1.last_ball_idx[b].cpu().numpy(), torch.cat(aux["sa1"]["ball_idx"], -1)[0].numpy())
        assert np.array_equal(enc.sa2.last_ball_idx[b].cpu().numpy(), torch.cat(aux["sa2"]["ball_idx"], -1)[0].numpy())
        assert rel_err(lv["l1_points"][b], aux["l1_points"][0]) <= tol, ("l1", b)
        assert rel_err(lv["l2_points"][b], aux["l2_points"][0]) <= tol, ("l2", b)
        assert rel_err(got[b], want[0, :, 0]) <= tol, ("l3", b)


# ------------------------------------------------------------------ config 2: B = 64, windows spread over the batch ----
def test_batch64_spread_windows_vs_oracle():
    """BASELINE config 2 (B = 64, N = 2048) with the bench's inputs: 8 windows spread over the batch are compared
    with the oracle (indices bit-exact, features 1e-5) - the full batch ran through the kernels in one go."""
    B, N = 64, 2048
    seeds = (100, 101, 102)
    enc = _encoder_with(seeds)
    ev_np = synth.make_windows(B, N, seed=1234 + 2)
    s1 = torch.from_numpy(synth.make_start_indices(B, N, 0))
    s2 = torch.from_numpy(synth.make_start_indices(B, 512, 1))
    with torch.no_grad():
        got = enc(dev(ev_np), fps_starts=(s1, s2))
    sel = torch.tensor([0, 9, 18, 27, 36, 45, 54, 63])
    states = _states(seeds)
    with torch.no_grad():
        want, aux = sa_oracle.encoder_forward(states, synth.ENCODER_SPECS, torch.from_numpy(ev_np)[sel],
                                              {"sa1": s1[sel], "sa2": s2[sel]}, return_aux=True)
    assert np.array_equal(enc.sa1.last_fps_idx[sel.to(DEV)].cpu().numpy(), aux["sa1"]["fps_idx"].numpy())
    assert np.array_equal(enc.sa1.last_ball_idx[sel.to(DEV)].cpu().numpy(), torch.cat(aux["sa1"]["ball_idx"], -1).numpy())
    assert np.array_equal(enc.sa2.last_fps_idx[sel.to(DEV)].cpu().numpy(), aux["sa2"]["fps_idx"].numpy())
    assert np.array_equal(enc.sa2.last_ball_idx[sel.to(DEV)].cpu().numpy(), torch.cat(aux["sa2"]["ball_idx"], -1).numpy())
    for j, b in enumerate(sel.tolist()):
        assert rel_err(got[b], want[j, :, 0]) <= FEAT_TOL, b


# ------------------------------------------------------------------ a5: sample_and_group, sampled SA ----------
def test_sample_and_group_golden(golden):
    """sample_and_group (pointnet2_utils.py:110-138) against the reference's own outputs; the start index is
    drawn from the CPU generator like the reference does."""
    g = golden("sampled")
    ev = g["events"]
    xyz = dev(ev[:, :3].transpose(0, 2, 1))
    pts = dev(ev.transpose(0, 2, 1))
    torch.manual_seed(21)
    new_xyz, new_points, grouped_xyz, fps_idx = e2h.sample_and_group(48, 0.3, 16, xyz, pts, returnfps=True)
    assert np.array_equal(fps_idx.cpu().numpy(), g["fps_idx"].astype(np.int64))
    assert np.array_equal(new_xyz.cpu().numpy(), g["new_xyz"])
    assert np.array_equal(grouped_xyz.cpu().numpy(), g["grouped_xyz"])
    assert np.array_equal(new_points.cpu().numpy(), g["new_points"])          # gathers and one subtraction: bitwise
    torch.manual_seed(22)
    _, np_points = e2h.sample_and_group(48, 0.3, 16, xyz, None)
    assert np.array_equal(np_points.cpu().numpy(), g["new_points_nopoints"])
    all_xyz, all_points = e2h.sample_and_group_all(xyz, pts)
    assert all_xyz.shape == (2, 1, 3) and not all_xyz.any()
    assert torch.equal(all_points, torch.cat([xyz, pts], -1).view(2, 1, 512, 8))


@pytest.mark.parametrize("prec,tol", [("fp32", 1e-5), ("tf32x3", 1e-5)])
def test_sampled_set_abstraction_golden(golden, prec, tol):
    """PointNetSetAbstraction with group_all=False (pointnet2_utils.py:176-202), eval mode, against the reference."""
    g = golden("sampled")
    m = e2h.PointNetSetAbstraction(npoint=48, radius=0.3, nsample=16, in_channel=5 + 3, mlp=[16, 32], group_all=False)
    load_numpy_state(m, synth.random_sa_state("mlp_convs.{j}", "mlp_bns.{j}", [[16, 32]], [8], seed=int(g["weight_seed"])))
    m = m.to(DEV).eval()
    ev = dev(g["events"])
    old = e2h.get_mlp_precision()
    try:
        e2h.set_mlp_precision(prec)
        torch.manual_seed(23)                       # the module draws the start index itself (CPU generator)
        with torch.no_grad():
            new_xyz, new_points = m(ev[:, :3, :], ev)
    finally:
        e2h.set_mlp_precision(old)
    assert np.array_equal(new_xyz.cpu().numpy(), g["module_xyz"])
    assert new_points.shape == (2, 32, 48)
    assert rel_err(new_points, g["module_points"]) <= tol


def test_sampled_set_abstraction_train_mode_matches_eval_with_batch_stats(golden):
    """train-mode path of the sampled SA layer (gather + scatter-add backward kernels, PyTorch conv/BN) against the
    same computation in stock torch ops on the kernel's indices."""
    g = golden("sampled")
    torch.manual_seed(3)
    m = e2h.PointNetSetAbstraction(npoint=48, radius=0.3, nsample=16, in_channel=5 + 3, mlp=[16, 32], group_all=False).to(DEV).train()
    ev = dev(g["events"])
    feats = ev.clone().requires_grad_(True)
    start = torch.from_numpy(g["start_module"])
    old = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        new_xyz, out = m(ev[:, :3, :].detach(), feats, fps_start=start)
        out.square().sum().backward()
        import copy
        ref = copy.deepcopy(m)
        for bn in ref.mlp_bns:
            bn.reset_running_stats()
        ref.zero_grad()
        xyz_rows = ev[:, :3, :].permute(0, 2, 1)
        fidx = e2h.farthest_point_sample(xyz_rows.contiguous(), 48, start=start)
        centres = torch.gather(xyz_rows, 1, fidx.unsqueeze(-1).expand(-1, -1, 3))
        ball = e2h.query_ball_point(0.3, 16, xyz_rows.contiguous(), centres.contiguous())
        f2 = ev.clone().requires_grad_(True)
        fr = f2.permute(0, 2, 1)
        gp = torch.stack([fr[b][ball[b]] for b in range(2)])
        gx = torch.stack([xyz_rows[b][ball[b]] for b in range(2)]) - centres.view(2, 48, 1, 3)
        h = torch.cat([gx, gp], -1).permute(0, 3, 2, 1)              # reference order here: [rel_xyz, points] (:128)
        for conv, bn in zip(ref.mlp_convs, ref.mlp_bns):
            h = torch.relu(bn(conv(h)))
        out2 = h.max(2).values
        out2.square().sum().backward()
    finally:
        torch.backends.cudnn.allow_tf32 = old
    assert torch.equal(new_xyz, centres.permute(0, 2, 1))
    assert rel_err(out, out2) <= 1e-5
    assert rel_err(feats.grad, f2.grad) <= 1e-4
    for (n, p), (_, q) in zip(m.named_parameters(), ref.named_parameters()):
        assert rel_err(p.grad, q.grad) <= 1e-4, n


# ------------------------------------------------------------------ the call sequence of TEHNet.forward --------
def _oracle_levels(states, ev_np, s1, s2):
    with torch.no_grad():
        want, aux = sa_oracle.encoder_forward(states, synth.ENCODER_SPECS, torch.from_numpy(ev_np), {"sa1": s1, "sa2": s2},
                                              return_aux=True)
    return want[:, :, 0], aux


@pytest.mark.parametrize("between", ["as_is", "contiguous", "clone", "scaled_copy", "to_same_device"])
def test_module_by_module_calls_like_tehnet(between):
    """TEHNet.forward (TEHNet.py:172-181) calls sa1, sa2, sa3 one by one on channel-first tensors.  Whatever the
    caller does to l1_points / l2_points between the layers - nothing, .contiguous(), .clone(), a new tensor, .to() -
    the next layer must see exactly the tensor it is handed: the row record riding on the layer output either survives
    (same tensor object, unmodified) or the layer falls back to transposing the channel-first tensor."""
    seeds = (41, 42, 43)
    enc = _encoder_with(seeds)
    ev_np = synth.make_windows(2, 2048, seed=321)
    s1 = torch.from_numpy(synth.make_start_indices(2, 2048, 7))
    s2 = torch.from_numpy(synth.make_start_indices(2, 512, 8))
    xyz = dev(ev_np)
    scale = 1.0
    from ev2hands_b200 import pointnet2_utils as pu
    pu.ROW_SHORTCUT.update(hit=0, stale=0, none=0)
    with torch.no_grad():
        l0_xyz = xyz[:, :3, :]
        l1_xyz, l1_points = enc.sa1(l0_xyz, xyz, fps_start=s1)
        if between == "contiguous":
            l1_points = l1_points.contiguous()          # already contiguous: the same object comes back
        elif between == "clone":
            l1_points = l1_points.clone()
        elif between == "scaled_copy":
            l1_points, scale = l1_points * 0.5, 0.5
        elif between == "to_same_device":
            l1_points = l1_points.to(DEV)
        l2_xyz, l2_points = enc.sa2(l1_xyz, l1_points, fps_start=s2)
        if between == "clone":
            l2_points = l2_points.clone()
        l3_xyz, l3_points = enc.sa3(l2_xyz, l2_points)
    assert l3_xyz.shape == (2, 3, 1) and l3_points.shape == (2, 1024, 1)
    states = _states(seeds)
    if scale == 1.0:
        want, aux = _oracle_levels(states, ev_np, s1, s2)
        assert rel_err(l1_points, aux["l1_points"]) <= FEAT_TOL
        assert rel_err(l2_points, aux["l2_points"]) <= FEAT_TOL
        assert rel_err(l3_points[:, :, 0], want) <= FEAT_TOL
    else:
        with torch.no_grad():
            o1 = sa_oracle.sa_msg_forward(states["sa1"], synth.ENCODER_SPECS["sa1"], torch.from_numpy(ev_np[:, :3]),
                                          torch.from_numpy(ev_np), s1)
            o2 = sa_oracle.sa_msg_forward(states["sa2"], synth.ENCODER_SPECS["sa2"], o1[0], o1[1] * 0.5, s2)
            o3 = sa_oracle.sa_all_forward(states["sa3"], synth.ENCODER_SPECS["sa3"], o2[0], o2[1])
        assert rel_err(l2_points, o2[1]) <= FEAT_TOL
        assert rel_err(l3_points, o3[1]) <= FEAT_TOL
    # the shortcut is taken exactly when the very tensor a layer produced comes back unmodified
    expect_hits = {"as_is": 2, "contiguous": 2, "to_same_device": 2, "clone": 0, "scaled_copy": 1}[between]
    assert pu.ROW_SHORTCUT["hit"] == expect_hits, pu.ROW_SHORTCUT


def test_mhlnes_in_place_write_to_l0_xyz():
    """MHLNES branch (TEHNet.py:176-177): l0_xyz is a VIEW of the input and its last channel is overwritten in place
    with the mean of channels 3.. before sa1 runs; the kernels read that view through its strides."""
    seeds = (44, 45, 46)
    enc = _encoder_with(seeds)
    ev_np = synth.make_windows(2, 2048, seed=322)
    s1 = torch.from_numpy(synth.make_start_indices(2, 2048, 9))
    s2 = torch.from_numpy(synth.make_start_indices(2, 512, 10))
    xyz = dev(ev_np)
    with torch.no_grad():
        l0_points = xyz
        l0_xyz = xyz[:, :3, :]
        l0_xyz[:, -1, :] = xyz[:, 3:, :].mean(1)
        l1_xyz, l1_points = enc.sa1(l0_xyz, l0_points, fps_start=s1)
        l2_xyz, l2_points = enc.sa2(l1_xyz, l1_points, fps_start=s2)
        _, l3_points = enc.sa3(l2_xyz, l2_points)
    ev_ref = torch.from_numpy(ev_np.copy())
    ev_ref[:, 2, :] = ev_ref[:, 3:, :].mean(1)
    assert torch.equal(xyz.cpu(), ev_ref)                 # same in-place arithmetic on both sides (mean of 2 values)
    want, aux = _oracle_levels(_states(seeds), ev_ref.numpy(), s1, s2)
    assert np.array_equal(enc.sa1.last_fps_idx.cpu().numpy(), aux["sa1"]["fps_idx"].numpy())
    assert rel_err(l1_points, aux["l1_points"]) <= FEAT_TOL
    assert rel_err(l3_points[:, :, 0], want) <= FEAT_TOL


# ------------------------------------------------------------------ the oracle on the GPU (cuBLAS rounding) ----
def test_oracle_on_gpu_agrees_with_cpu_oracle_and_kernels(golden):
    """SURVEY 8c caveat 4: the reference's own ops on the B200 (square_distance = cuBLAS sgemm with K = 3) against the
    CPU (MKL) outputs the goldens hold, and against the kernels.  FPS has no matrix product and must agree exactly;
    for the ball query the number of differing entries is recorded (and asserted to be zero when it is)."""
    g = golden("fps_ball")
    xyz = dev(g["xyz"])
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        fps_gpu = sa_oracle.fps(xyz, 512, torch.from_numpy(g["start"]).to(DEV))
        centres = sa_oracle.take_rows(xyz, fps_gpu)
        sq_gpu = sa_oracle.pairwise_sqdist(centres[:1, :8], xyz[:1])[0]
        report = {"fps_equal_cpu_oracle": bool(np.array_equal(fps_gpu.cpu().numpy(), g["fps_idx"].astype(np.int64)))}
        sq_bits_equal = bool(np.array_equal(sq_gpu.cpu().numpy().view(np.uint32), g["sqdist_w0_first8"].view(np.uint32)))
        report["sqdist_bits_equal_cpu_oracle"] = sq_bits_equal
        report["sqdist_max_abs_diff"] = float(np.abs(sq_gpu.cpu().numpy() - g["sqdist_w0_first8"]).max())
        for r, k in zip([0.1, 0.2, 0.4], [32, 64, 128]):
            ball_gpu = sa_oracle.ball_query(r, k, xyz, centres).cpu().numpy()
            kern = e2h.query_ball_point(r, k, xyz, centres).cpu().numpy()
            want = g["ball_r%g" % r].astype(np.int64)
            assert np.array_equal(kern, want)                                      # kernels == CPU reference, always
            report["ball_r%g_entries_differing_gpu_oracle_vs_cpu" % r] = int((ball_gpu != want).sum())
            report["ball_r%g_groups_differing" % r] = int((ball_gpu != want).any(-1).sum())
            report["ball_r%g_entries" % r] = int(want.size)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    _record("gpu_oracle_crosscheck.json", report)
    print("gpu-oracle cross-check:", json.dumps(report))
    assert report["fps_equal_cpu_oracle"]
    # cuBLAS may round the K = 3 product differently from MKL: membership may flip for pairs within 1 ulp of r^2, never more
    for r in (0.1, 0.2, 0.4):
        assert report["ball_r%g_groups_differing" % r] <= 0.001 * 2 * 512


# ------------------------------------------------------------------ training at the model's shapes -------------
@pytest.mark.parametrize("tensor_core_gemms", ["", "dgrad", "all"])
def test_train_step_at_model_shapes_matches_reference_autograd(golden, tensor_core_gemms, monkeypatch):
    """sa2 of the model (D = 320 feature channels, K = 64 / 128, S = 128) in train mode: forward with batch-statistics
    BatchNorm and backward through max-pool (arg-max route) and the grouping gather (scatter-add with heavy
    contention: every point is a neighbour of most centres) against the REFERENCE module's own autograd on CPU
    (tests/golden/train_sa2.npz, made by make_golden.py from the unmodified reference).  fp32 GEMMs over rows, and
    the input-gradient GEMMs on the tensor cores (EV2H_TRAIN_TC=dgrad): strict bars.  Tensor-core forward as well
    (EV2H_TRAIN_TC=1): forward at the same bar, gradients at 1e-2 - the weight gradients in front of a batch-statistics
    BatchNorm are differences of large sums and amplify the forward's 2e-6."""
    import ev2hands_b200.pointnet2_utils as pu
    monkeypatch.setattr(pu, "_TRAIN_TC", tensor_core_gemms)
    gtol = 1e-2 if tensor_core_gemms == "all" else 2e-4
    g = golden("train_sa2")
    m = e2h.PointNetSetAbstractionMsg(128, [0.4, 0.8], [64, 128], 320, [[128, 128, 256], [128, 196, 256]])
    load_numpy_state(m, synth.random_state_for(synth.ENCODER_SPECS["sa2"], seed=int(g["weight_seed"])))
    m = m.to(DEV).train()
    ev = dev(g["events"])
    feats = dev(np.random.RandomState(int(g["feats_seed"])).randn(2, 320, 512).astype(np.float32)).requires_grad_(True)
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        new_xyz, out = m(ev[:, :3, :], feats, fps_start=torch.from_numpy(g["start"]))
        lw = torch.from_numpy(np.linspace(0.5, 1.5, out.numel(), dtype=np.float32)).view_as(out).to(DEV)
        (out * lw).sum().backward()
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    assert np.array_equal(new_xyz.detach().cpu().numpy(), g["new_xyz"])
    assert rel_err(out[:, ::4, ::4], g["out_every4"]) <= 2e-5
    assert rel_err(feats.grad[:, :, ::8], g["grad_feats_every8"]) <= gtol
    grads = dict(m.named_parameters())
    for key in g:
        if key.startswith("grad.") and not (key.endswith(".bias") and ".conv_blocks." in "." + key):
            assert rel_err(grads[key[5:]].grad, g[key]) <= gtol, key
    # a convolution bias in front of a batch-statistics BatchNorm has an exactly zero gradient (the mean is subtracted):
    # both sides hold rounding noise only, orders of magnitude below the weight gradients
    wmax = float(np.abs(g["grad.conv_blocks.1.1.weight"]).max())
    assert float(grads["conv_blocks.1.2.bias"].grad.abs().max()) <= 1e-3 * wmax and float(np.abs(g["grad.conv_blocks.1.2.bias"]).max()) <= 1e-3 * wmax
    assert rel_err(m.bn_blocks[0][0].running_mean, g["running_mean_0_0"]) <= 1e-5
    assert rel_err(m.bn_blocks[1][2].running_var, g["running_var_1_2"]) <= 1e-5


# ------------------------------------------------------------------ FPS start indices: capture and range -------
def test_graph_capture_refuses_host_start_indices():
    enc = _encoder_with((1, 2, 3))
    ev = dev(synth.make_windows(2, 2048, seed=8))
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        GraphedForward(lambda e, a, b: enc(e, fps_starts=(a, b)), ev, torch.zeros(2, dtype=torch.long), torch.zeros(2, dtype=torch.long))
    # a captured forward that would draw the start indices itself is refused inside the capture
    with torch.no_grad():
        enc(ev)                                               # warm: weights folded outside the capture
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="capture"):
        with torch.no_grad(), torch.cuda.graph(graph):
            enc(ev)
    torch.cuda.synchronize()
    # with device-resident starts the graph replays and follows refilled start indices
    s1 = torch.from_numpy(synth.make_start_indices(2, 2048, 1)).to(DEV)
    s2 = torch.from_numpy(synth.make_start_indices(2, 512, 2)).to(DEV)
    with torch.no_grad():
        gf = GraphedForward(lambda e, a, b: enc(e, fps_starts=(a, b)), ev, s1, s2)
        a = gf(ev, s1, s2).clone()
        t1 = torch.from_numpy(synth.make_start_indices(2, 2048, 5)).to(DEV)
        b = gf(ev, t1, s2).clone()
        want_b = enc(ev, fps_starts=(t1, s2))
        want_a = enc(ev, fps_starts=(s1, s2))
    assert torch.equal(a, want_a) and torch.equal(b, want_b) and not torch.equal(a, b)


def test_fps_start_index_out_of_range():
    xyz = dev(synth.make_windows(2, 256, seed=3)[:, :3].transpose(0, 2, 1))
    with pytest.raises(IndexError):
        e2h.farthest_point_sample(xyz, 16, start=torch.tensor([0, 256]))
    with pytest.raises(IndexError):
        e2h.farthest_point_sample(xyz, 16, start=torch.tensor([-1, 3]))
    # device-resident starts cannot be checked without a sync: the kernel clamps them instead of reading out of bounds
    got = e2h.farthest_point_sample(xyz, 16, start=torch.tensor([5, 999], device=DEV))
    want = e2h.farthest_point_sample(xyz, 16, start=torch.tensor([5, 255]))
    assert torch.equal(got, want)
    with pytest.raises(RuntimeError, match="requires_grad"):
        enc = _encoder_with((1, 2, 3))
        ev = dev(synth.make_windows(1, 2048, seed=8)).requires_grad_(True)
        enc.sa1(ev[:, :3, :], ev.detach())


# ------------------------------------------------------------------ nn.DataParallel re-entrancy ----------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_data_parallel_two_replicas_match_single_device():
    """train.py:68 wraps the model in nn.DataParallel: one Python thread per GPU drives replicas of the same module
    objects concurrently.  Eval forward over 2 devices must equal the single-device result bit for bit."""
    enc = _encoder_with((51, 52, 53))
    ev = dev(synth.make_windows(6, 2048, seed=91))
    s1 = torch.from_numpy(synth.make_start_indices(6, 2048, 1)).to(DEV)
    s2 = torch.from_numpy(synth.make_start_indices(6, 512, 2)).to(DEV)

    class Wrap(torch.nn.Module):
        def __init__(self, enc):
            super().__init__()
            self.enc = enc

        def forward(self, ev, a, b):
            return self.enc(ev, fps_starts=(a, b))

    w = Wrap(enc)
    with torch.no_grad():
        want = w(ev, s1, s2)
        dp = torch.nn.DataParallel(w, device_ids=[0, 1])
        for _ in range(3):                               # repeated: caches are built by concurrent threads the first time
            got = dp(ev, s1, s2)
            assert torch.equal(got, want)


# ------------------------------------------------------------------ config 4: the whole training step ---------
def test_tehnet_training_step_runs_end_to_end(monkeypatch):
    """BASELINE configs[3] at a small batch: forward in train mode through the whole network (kernels for FPS, ball
    query, gather, max-pool; cuDNN conv/BN), criterion, backward, bucketed reducer, Adam - every parameter receives a
    finite gradient inside the flat buffer and the loss moves."""
    monkeypatch.setenv("ERPC", "1")
    from ev2hands_b200 import tehnet, trainer
    torch.manual_seed(0)
    net = tehnet.TEHNet(n_pose_params=6).to(DEV).train()
    hands = tehnet.create_standin_mano_layers(DEV)
    opt = torch.optim.Adam(net.parameters(), lr=1e-3)
    red = trainer.BucketedGradReducer(net.parameters(), n_buckets=4)
    batch = tehnet.make_training_batch(3, 2048, seed=1, device=DEV)
    losses_seen = []
    for _ in range(3):
        b = {k: (dict(v) if isinstance(v, dict) else v) for k, v in batch.items()}
        loss, parts = trainer.train_step(net, hands, b, opt, red, tehnet.training_losses)
        losses_seen.append(float(loss))
        assert torch.isfinite(loss)
    assert torch.isfinite(red.flat).all()
    n_with_grad = sum(int(p.grad is not None and p.grad.abs().sum() > 0) for p in net.parameters())
    n_all = sum(1 for _ in net.parameters())
    # conv biases in front of a batch-statistics BatchNorm have exactly zero gradients; everything else must learn
    assert n_with_grad >= 0.6 * n_all, (n_with_grad, n_all)
    assert losses_seen[-1] != losses_seen[0]
    red.remove()
    # eval mode of the same network: the fused inference kernels, finite outputs of the reference's shapes
    net.eval()
    with torch.no_grad():
        out = net(batch["events"], hands)
    assert out["class_logits"].shape == (3, 4, 2048) and out["left"]["vertices"].shape == (3, 778, 3)
    assert out["right"]["j3d"].shape == (3, 21, 3) and torch.isfinite(out["class_logits"]).all()


# ------------------------------------------------------------------ N2: classifier + query convolutions + attention ----
def _tehnet_with_heads(golden_heads, monkeypatch):
    monkeypatch.setenv("ERPC", "1")
    from ev2hands_b200 import tehnet
    net = tehnet.TEHNet(n_pose_params=6)
    st = synth.random_head_state(seed=int(golden_heads["weight_seed"]))
    res = net.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in st.items()}, strict=False)
    assert not res.unexpected_keys
    return net.to(DEV).eval()


@pytest.mark.parametrize("prec,tol", [("tf32x3", 1e-5), ("bf16", 1e-2)])
def test_heads_golden(golden, monkeypatch, prec, tol):
    """SURVEY 8f row N2: the segmentation classifier, both query convolutions (3-tap Conv1d gathered by the kernel's
    loaders, BatchNorm after the ReLU in the epilogue) and the class-wise attention, against the reference's own
    modules (tests/golden/heads.npz, TEHNet.py:188-192)."""
    g = golden("heads")
    net = _tehnet_with_heads(g, monkeypatch)
    feat = dev(np.random.RandomState(int(g["feature_seed"])).randn(2, 256, 2048).astype(np.float32))
    old = e2h.get_mlp_precision()
    try:
        e2h.set_mlp_precision(prec)
        with torch.no_grad():
            seg, left, right = net._heads_cuda(feat)
    finally:
        e2h.set_mlp_precision(old)
    assert seg.shape == (2, 4, 2048) and left.shape == (2, 4, 2048) and right.shape == (2, 4, 2048)
    assert rel_err(seg, g["seg_out"]) <= tol
    assert rel_err(left, g["left_features"]) <= tol
    assert rel_err(right, g["right_features"]) <= tol


def test_heads_kernels_vs_torch_modules_on_odd_shapes(monkeypatch):
    """conv1d_tc and class_attention against the PyTorch modules they replace, sequence lengths that are not a
    multiple of the 128-row tile (the convolution's zero padding must follow the SEQUENCE, not the tile)."""
    torch.manual_seed(5)
    B, N, Cin, Cout = 3, 200, 64, 96
    x = torch.randn(B, Cin, N, device=DEV)
    conv = torch.nn.Conv1d(Cin, Cout, 3, 1, 1).to(DEV)
    from ev2hands_b200 import tehnet
    rows = x.permute(0, 2, 1).contiguous().view(B * N, Cin)
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            want = torch.relu(conv(x)) * 1.5 - 0.25
        L = tehnet._pack_conv1d(conv.weight.detach().double(), conv.bias.detach().double(), _capi.TC_F16X3)
        L["mode"] = _capi.TC_F16X3
        post = (torch.full((Cout,), 1.5, device=DEV), torch.full((Cout,), -0.25, device=DEV))
        got = tehnet._conv_rows(rows, B * N, Cin, L, N, relu=True, post=post)
        assert rel_err(got.view(B, N, -1)[:, :, :Cout].permute(0, 2, 1), want) <= 1e-5
        key, val, qry = torch.randn(B, 4, N, device=DEV), torch.randn(B, 64, N, device=DEV), torch.randn(B, 64, N, device=DEV)
        want_a = tehnet.AttentionBlock()(key, val, qry)
        r = lambda t: t.permute(0, 2, 1).contiguous().view(B * N, -1)      # noqa: E731
        got_a = _capi.class_attention(r(key), 4, r(qry), 64, r(val), 64, B, N, 4, 64, 64 ** -0.5)
        assert rel_err(got_a, want_a) <= 1e-5
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


# ------------------------------------------------------------------ fp16-split numeric range flag ---------------
def test_fp16_split_overflow_raises_the_range_flag():
    """the default fp32-level mode splits operands into fp16 pairs: an activation beyond the fp16 range must not pass
    silently - the fused kernel raises a device flag that check_numeric_range() reads and clears"""
    enc = _encoder_with((61, 62, 63))
    ev = dev(synth.make_windows(2, 2048, seed=77))
    s1 = torch.from_numpy(synth.make_start_indices(2, 2048, 1))
    s2 = torch.from_numpy(synth.make_start_indices(2, 512, 2))
    from ev2hands_b200 import pointnet2_utils as pu
    if pu._fused_mode(_capi.TC_TF32X3) != _capi.TC_F16X3:
        pytest.skip("the fp16 split is not the selected fp32-level arithmetic (EV2H_SPLIT)")
    e2h.check_numeric_range(DEV)                               # clear
    with torch.no_grad():
        ok_out = enc(ev, fps_starts=(s1, s2))
    assert torch.isfinite(ok_out).all() and e2h.check_numeric_range(DEV)
    big = ev.clone()
    big[:, 3:, :] *= 3.0e6                                     # event counts far outside any real window: layer-1 outputs ~1e6
    with torch.no_grad():
        enc(big, fps_starts=(s1, s2))
    assert not e2h.check_numeric_range(DEV)                    # flagged ...
    assert e2h.check_numeric_range(DEV)                        # ... and cleared by the read


# ------------------------------------------------------------------ pipelined front end ------------------------
def test_pipelined_sampling_and_ball_query_are_bit_identical(monkeypatch):
    """the sampling cut into ranges (resumable kernel) with the ball query of each finished range on a side stream
    must give exactly the indices, centres and features of one sampling launch followed by one ball query"""
    from ev2hands_b200 import pointnet2_utils as pu
    enc = _encoder_with((71, 72, 73))
    ev = dev(synth.make_windows(5, 2048, seed=99))
    s1 = torch.from_numpy(synth.make_start_indices(5, 2048, 3))
    s2 = torch.from_numpy(synth.make_start_indices(5, 512, 4))
    outs = {}
    for splits in (0, 2, 4):
        monkeypatch.setattr(pu, "_FPS_SPLITS", splits)
        with torch.no_grad():
            out, lv = enc(ev, fps_starts=(s1, s2), return_levels=True)
        torch.cuda.synchronize()
        outs[splits] = (out.clone(), enc.sa1.last_fps_idx.clone(), enc.sa1.last_ball_idx.clone(), lv["l1_xyz"].clone(), lv["l1_points"].clone())
    for splits in (2, 4):
        for a, b in zip(outs[0], outs[splits]):
            assert torch.equal(a, b), splits
    # the C-ABI range entry alone, odd split points, against the C oracle
    xyz = np.ascontiguousarray(synth.make_windows(3, 1000, seed=5)[:, :3].transpose(0, 2, 1))
    start = synth.make_start_indices(3, 1000, 7)
    want = c_oracle.fps(xyz, 100, start)
    xd = dev(xyz)
    idx = torch.empty((3, 100), dtype=torch.int32, device=DEV)
    rows = torch.empty((3, 100, 3), dtype=torch.float32, device=DEV)
    best = torch.empty((3, 1000), dtype=torch.float32, device=DEV)
    cur = torch.empty((3,), dtype=torch.int32, device=DEV)
    sd = torch.from_numpy(start).to(DEV)
    for lo, hi in ((0, 1), (1, 37), (37, 99), (99, 100)):
        _capi.fps_range(xd, _capi.rows_strides(xd), sd, 3, 1000, 100, lo, hi, best, cur, idx, rows, None)
    assert np.array_equal(idx.cpu().numpy(), want)
    assert torch.equal(rows, torch.gather(xd, 1, idx.long().unsqueeze(-1).expand(-1, -1, 3)))


# ------------------------------------------------------------------ FPS kernels for long windows -------------
def _long_window_cases():
    rs = np.random.RandomState(5)
    ev = synth.make_windows(3, 16384, seed=71)                          # clustered, ~40 % exact copies: ties everywhere
    yield "events16384", np.ascontiguousarray(ev[:, :3].transpose(0, 2, 1)), 512
    ev = synth.make_windows(2, 9000, seed=72)                           # ragged length: padded positions in the last buckets
    yield "events9000", np.ascontiguousarray(ev[:, :3].transpose(0, 2, 1)), 300
    ev = synth.make_windows(2, 5000, seed=73, mode="uniform")
    yield "uniform5000", np.ascontiguousarray(ev[:, :3].transpose(0, 2, 1)), 700
    lattice = rs.randint(0, 12, size=(2, 12000, 3)).astype(np.float32) / 4.0   # 1728 distinct points: equal distances between
    yield "lattice12000", lattice, 2000                                        # DIFFERENT points, and more samples than points
    flat = np.zeros((1, 6000, 3), np.float32)
    flat[..., 0] = rs.rand(1, 6000).astype(np.float32)                         # degenerate extent on two axes
    yield "line6000", flat, 64
    same = np.full((1, 4500, 3), 0.25, np.float32)                             # one point 4500 times
    yield "same4500", same, 16


@pytest.mark.parametrize("name,xyz,s", list(_long_window_cases()), ids=lambda v: v if isinstance(v, str) else "")
def test_fps_long_window_kernels_agree_with_the_oracle(name, xyz, s):
    """exhaustive, cluster and spatially pruned kernels (ev2h_fps_variant_f32) all return the C oracle's indices"""
    b, n = xyz.shape[:2]
    start = synth.make_start_indices(b, n, seed=n)
    want = c_oracle.fps(xyz, s, start)
    x = dev(xyz)
    for variant in (1, 2, 3, 0):
        idx, rows, cf = _capi.fps(x, _capi.rows_strides(x), torch.from_numpy(start), b, n, s, variant=variant)
        got = idx.cpu().numpy()
        assert np.array_equal(got, want), "variant %d differs from the oracle at %s" % (variant, np.argwhere(got != want)[:3])
        picked = torch.gather(x, 1, idx.long().unsqueeze(-1).expand(-1, -1, 3))
        assert torch.equal(rows, picked) and torch.equal(cf, picked.permute(0, 2, 1))


def test_fps_pruned_kernel_with_non_finite_coordinates_matches_the_exhaustive_kernel():
    ev = synth.make_windows(2, 8000, seed=74)
    xyz = np.ascontiguousarray(ev[:, :3].transpose(0, 2, 1))
    xyz[0, 17, 1] = np.inf
    xyz[1, 4000, 0] = np.nan
    x = dev(xyz)
    start = torch.from_numpy(synth.make_start_indices(2, 8000, seed=3))
    a = _capi.fps(x, _capi.rows_strides(x), start, 2, 8000, 128, variant=1)[0]
    b = _capi.fps(x, _capi.rows_strides(x), start, 2, 8000, 128, variant=3)[0]
    assert torch.equal(a, b)


def test_tensor_core_layer_kernel_over_millions_of_rows():
    """the training path runs ev2h_linear_tc over B*S*K ~ 2 M rows (110 tiles per CTA instead of the inference path's
    handful): a loader-group hand-shake that could miss a barrier phase once in ~10^5 tiles showed up only there
    (fixed: stage ownership).  Many tiles, three arithmetic modes, result checked on a sample."""
    from ev2hands_b200 import pointnet2_utils as pu
    torch.manual_seed(0)
    M = 1 << 20
    for cin, cout, mode in ((64, 96, _capi.TC_F16X3), (96, 64, _capi.TC_TF32_BF16C), (8, 32, _capi.TC_F16X3), (196, 256, _capi.TC_TF32X3)):
        x = torch.randn(M, cin, device=DEV)
        w = torch.randn(cin, cout, device=DEV) / cin ** 0.5
        packed = pu._pack_dense(w, mode)
        b = torch.zeros(((cout + 127) // 128 * 128,), device=DEV)
        y = torch.empty(M, cout, device=DEV)
        for _ in range(12):
            _capi.linear_tc_no_relu(x, M, cin, cin, packed, b, cout, y, cout, 0, mode)
        torch.cuda.synchronize()
        ref = x[-4096:].double() @ w.double()
        assert float((y[-4096:].double() - ref).abs().max() / ref.abs().max()) < 1e-5


# ------------------------------------------------------------------ ball query: more edge cases vs the C oracle ----
@pytest.mark.parametrize("n,s,mode,radii,ks", [
    (16384, 100, "uniform", [0.4, 0.1, 0.2], [128, 32, 64]),        # radii in any order
    (9000, 77, "events", [0.25], [24]),                              # ragged length, one radius
    (7000, 64, "events", [0.3, 0.3], [16, 48]),                      # equal radii
    (6500, 40, "events", [1e-4, 5.0], [8, 200]),                     # nothing but the centre / the whole window
])
def test_ball_query_radius_lists_and_ragged_lengths_vs_c_oracle(n, s, mode, radii, ks):
    b = 3
    ev = synth.make_windows(b, n, seed=200 + n, mode=mode)
    xyz = np.ascontiguousarray(ev[:, :3].transpose(0, 2, 1))
    fidx = c_oracle.fps(xyz, s, synth.make_start_indices(b, n, seed=5))
    centres = np.stack([xyz[i, fidx[i]] for i in range(b)])
    xd = dev(xyz)
    packed, cnt = _capi.ball_query(xd, _capi.rows_strides(xd), dev(centres), n, radii, ks, with_counts=True)
    packed, cnt = packed.cpu().numpy(), cnt.cpu().numpy()
    off = 0
    for j, (r, k) in enumerate(zip(radii, ks)):
        want = c_oracle.ball_query(r, k, xyz, centres)
        assert np.array_equal(packed[:, :, off:off + k], want), (r, k)
        real = (want != n).sum(-1)
        # the reference pads with copies of the first neighbour: the real count is the number of distinct entries
        distinct = np.array([[len(set(want[w, c])) for c in range(s)] for w in range(b)])
        assert np.array_equal(cnt[j], np.where(real == 0, 0, distinct)), (r, k)
        off += k


# ------------------------------------------------------------------ duplicate flags for long windows -----------------
@pytest.mark.parametrize("n", [4097, 9000, 16384])
def test_first_occurrence_on_long_windows(n):
    rs = np.random.RandomState(n)
    base = rs.rand(2, n // 3, 8).astype(np.float32)
    base[:, :, 7] = 0
    pick = rs.randint(0, n // 3, size=(2, n))
    pts8 = np.stack([base[b][pick[b]] for b in range(2)])                 # sampling with replacement: ~2/3 exact copies
    first = _capi.first_occurrence(dev(pts8)).cpu().numpy()
    want = np.zeros((2, n), dtype=np.uint8)
    for b in range(2):
        _, idx = np.unique(pts8[b].view(np.dtype((np.void, 32))).ravel(), return_index=True)
        want[b, idx] = 1
    assert np.array_equal(first, want)


def test_long_window_features_do_not_depend_on_duplicate_skipping(monkeypatch):
    """16384-event windows: the rows of exact copies of a point are skipped (round 2: the duplicate flags now cover long
    windows too); pooled features are bit-identical to evaluating them"""
    import ev2hands_b200.pointnet2_utils as pu
    enc = _encoder_with((21, 22, 23))
    ev = dev(synth.make_windows(2, 16384, seed=77))
    s1 = torch.from_numpy(synth.make_start_indices(2, 16384, 2))
    s2 = torch.from_numpy(synth.make_start_indices(2, 512, 3))
    outs = []
    for dedup in (True, False):
        monkeypatch.setattr(pu, "_DEDUP", dedup)
        with torch.no_grad():
            outs.append(enc(ev, fps_starts=(s1, s2)).clone())
    assert torch.equal(outs[0], outs[1])


@pytest.mark.parametrize("b,n,d", [(3, 2048, 5), (2, 777, 4), (2, 300, 0), (80, 16384, 5)])
def test_point_records_kernel(b, n, d):
    """ev2h_point_records_f32 = [features | xyz | 0] per point, from strided channel-first views; the last case has more
    points than one grid pass covers"""
    torch.manual_seed(n)
    ev = torch.randn(b, 7, n, device=DEV)
    pts = ev[:, 1:1 + d, :] if d else None
    xyz = ev[:, 2:5, :]
    got = _capi.point_records(pts, xyz, _capi.cf_strides(xyz))
    want = torch.zeros(b, n, 8, device=DEV)
    if d:
        want[:, :, :d] = pts.permute(0, 2, 1)
    want[:, :, d:d + 3] = xyz.permute(0, 2, 1)
    assert torch.equal(got, want)


def test_bench_prints_the_contract_line(tmp_path):
    """one short `bench.py` run through the driver's command line: ONE JSON line with the keys the contract names;
    --dump-outputs writes the features of the last timed step, the ones the checksum sums"""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "3",
                          "--no-configs", "--no-raw-events", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / "dump")],
                         capture_output=True, text=True, timeout=900, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "roofline", "e2e", "gpu_launches", "clocks"):
        assert key in d, key
    assert d["metric"] == "encoder event-windows/s" and d["n_gpus"] == 1 and d["steps"] == 3 and d["scaling"] == "weak"
    assert d["gpu_launches"] > 0 and d["value"] > 1000 and d["e2e"]["value"] > 1000
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    r = d["roofline"]
    assert r["bound"] == "tensor" and 0 < r["frac"] < 1 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-6
    assert abs(d["ms_per_step"] * d["value"] / 1e3 - 64) < 0.5          # 64 windows per step
    assert os.listdir(tmp_path / "dump") == ["features.npy"]
    feats = np.load(tmp_path / "dump" / "features.npy")
    assert feats.dtype == np.float32 and feats.shape == (64, 1024) and np.isfinite(feats).all()
    assert abs(feats.astype(np.float64).sum() - d["checksum"]) <= 1e-9 * max(abs(d["checksum"]), 1.0)


@pytest.mark.parametrize("m,cout,cin,ld_x", [(4096, 64, 8, 8), (100000, 96, 64, 64), (33333, 128, 323, 324), (5000, 196, 128, 128),
                                              (2048, 1024, 512, 512), (777, 32, 7, 8), (1500, 64, 515, 515), (64, 256, 256, 256)])
def test_weight_gradient_kernel(m, cout, cin, ld_x):
    """ev2h_wgrad_f32: dW = dY^T X over rows (the contraction runs over M), against fp64; strided and unaligned rows;
    deterministic"""
    torch.manual_seed(m)
    dy = torch.randn(m, cout, device=DEV) * torch.pow(10.0, -4 * torch.rand(m, 1, device=DEV))      # gradient-like dynamic range
    xbuf = torch.randn(m, ld_x, device=DEV)
    x = xbuf[:, :cin]
    got = _capi.wgrad(dy, x)
    want = dy.double().t() @ x.double()
    scale = (dy.double().abs().t() @ x.double().abs()).max()
    assert float((got.double() - want).abs().max() / scale) < 2e-6
    dw2, db = _capi.wgrad(dy, x, want_bias=True)
    assert torch.equal(got, dw2)
    assert float((db.double() - dy.double().sum(0)).abs().max() / dy.double().abs().sum(0).max()) < 2e-6
