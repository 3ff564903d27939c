"""Generate the golden vectors under tests/golden/ from the REAL reference.

Run in the build container only (it reads /root/reference, which does not exist
on the GPU box):

    python tests/golden/make_golden.py

The reference's ``model`` package cannot be imported normally (``model/__init__``
pulls in trimesh / manopth, absent here), so ``pointnet2_utils.py`` and
``TEHNet.py`` are loaded by file path under a stand-in package name.  Nothing is
copied: the reference code runs unmodified and only its outputs are saved.

Inputs come from ``ev2hands_b200.synth`` (numpy RandomState, portable) and are
stored alongside the outputs so the fixtures stay valid even if the generator
changes.  FPS start indices: the reference draws them with ``torch.randint`` on
the CPU generator (pointnet2_utils.py:75); we seed, draw the same numbers
ourselves, re-seed, and then call the reference so it re-draws them.
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from ev2hands_b200 import synth  # noqa: E402

REF_DIR = "/root/reference/src/Ev2Hands/model"


def load_reference():
    os.environ["ERPC"] = "1"     # dataset modules set this at import (erpc.py:20)
    pkg = types.ModuleType("refmodel")
    pkg.__path__ = [REF_DIR]
    sys.modules["refmodel"] = pkg
    mods = {}
    for name in ("pointnet2_utils", "TEHNet"):
        spec = importlib.util.spec_from_file_location("refmodel." + name, os.path.join(REF_DIR, name + ".py"))
        m = importlib.util.module_from_spec(spec)
        sys.modules["refmodel." + name] = m
        spec.loader.exec_module(m)
        mods[name] = m
    return mods["pointnet2_utils"], mods["TEHNet"]


def seeded_starts(seed, n_points, batch):
    torch.manual_seed(seed)
    s = torch.randint(0, n_points, (batch,), dtype=torch.long)
    torch.manual_seed(seed)      # the reference's own draw now returns the same numbers
    return s


def to_t(state):
    return {k: torch.from_numpy(np.asarray(v)) for k, v in state.items()}


def small_idx(a):
    a = np.asarray(a)
    return a.astype(np.int16) if a.max() < 32768 else a.astype(np.int32)


_ONLY = set(sys.argv[1:])      # e.g. `python make_golden.py decoder`: rewrite only decoder.npz
_savez = np.savez_compressed


def _savez_selected(path, **kw):
    if not _ONLY or os.path.basename(path)[:-4] in _ONLY:
        _savez(path, **kw)


np.savez_compressed = _savez_selected


def main():
    pu, th = load_reference()
    torch.set_num_threads(8)

    # ---- 1. FPS / square_distance / ball query on sa1-shaped windows ----------
    ev = synth.make_windows(2, 2048, seed=1234)
    xyz = torch.from_numpy(ev[:, :3].transpose(0, 2, 1).copy())
    start = seeded_starts(7, 2048, 2)
    fps_idx = pu.farthest_point_sample(xyz, 512)
    assert torch.equal(fps_idx[:, 0], start)
    centres = pu.index_points(xyz, fps_idx)
    out = {"xyz": xyz.numpy(), "start": start.numpy(), "fps_idx": small_idx(fps_idx.numpy()),
           "sqdist_w0_first8": pu.square_distance(centres[:1, :8], xyz[:1]).numpy()[0]}
    for r, k in zip([0.1, 0.2, 0.4], [32, 64, 128]):
        out["ball_r%g" % r] = small_idx(pu.query_ball_point(r, k, xyz, centres).numpy())
    np.savez_compressed(os.path.join(HERE, "fps_ball.npz"), **out)

    # ---- 2. edge cases ---------------------------------------------------------
    rs = np.random.RandomState(99)
    edge = {}
    # (a) every point identical
    same = np.tile(rs.rand(1, 1, 3).astype(np.float32), (1, 64, 1))
    st = seeded_starts(3, 64, 1)
    edge["same_xyz"], edge["same_start"] = same, st.numpy()
    edge["same_fps"] = pu.farthest_point_sample(torch.from_numpy(same), 16).numpy()
    edge["same_ball"] = pu.query_ball_point(0.2, 8, torch.from_numpy(same), torch.from_numpy(same[:, :4])).numpy()
    # (b) sample every point (S == N), coarse grid => many exact distance ties
    grid = (rs.randint(0, 5, size=(2, 96, 3)).astype(np.float32) / 4.0) * 2 - 1
    st = seeded_starts(4, 96, 2)
    edge["grid_xyz"], edge["grid_start"] = grid, st.numpy()
    g_fps = pu.farthest_point_sample(torch.from_numpy(grid), 96)
    edge["grid_fps"] = g_fps.numpy()
    g_c = pu.index_points(torch.from_numpy(grid), g_fps[:, :24])
    edge["grid_ball_r0.5_k16"] = pu.query_ball_point(0.5, 16, torch.from_numpy(grid), g_c).numpy()
    # (c) radii whose fp32 square rounds UP (0.3, 0.7) and a tiny radius that only
    #     ever contains the centre itself; N not a multiple of 32
    pts = (rs.rand(2, 301, 3).astype(np.float32) * 2 - 1)
    st = seeded_starts(5, 301, 2)
    edge["odd_xyz"], edge["odd_start"] = pts, st.numpy()
    o_fps = pu.farthest_point_sample(torch.from_numpy(pts), 40)
    edge["odd_fps"] = o_fps.numpy()
    o_c = pu.index_points(torch.from_numpy(pts), o_fps)
    for r, k in [(0.3, 16), (0.7, 48), (1e-3, 4), (4.0, 301)]:
        edge["odd_ball_r%g_k%d" % (r, k)] = pu.query_ball_point(r, k, torch.from_numpy(pts), o_c).numpy()
    # (d) centres that are NOT input points and have no neighbour: reference leaves N
    far = np.full((2, 2, 3), 50.0, dtype=np.float32)
    edge["far_centres"] = far
    edge["far_ball_r0.2_k4"] = pu.query_ball_point(0.2, 4, torch.from_numpy(pts), torch.from_numpy(far)).numpy()
    np.savez_compressed(os.path.join(HERE, "edge.npz"), **edge)

    # ---- 3. encoder sa1 -> sa2 -> sa3 with random weights ---------------------
    net = th.TEHNet(n_pose_params=6).eval()
    states = {n: synth.random_state_for(synth.ENCODER_SPECS[n], seed=100 + i)
              for i, n in enumerate(("sa1", "sa2", "sa3"))}
    for n in states:
        getattr(net, n).load_state_dict(to_t(states[n]), strict=True)
    events = torch.from_numpy(synth.make_windows(2, 2048, seed=1235))
    s1 = seeded_starts(11, 2048, 2)
    s2_probe = None
    with torch.no_grad():
        l0_xyz = events[:, :3, :]
        l1_xyz, l1_points = net.sa1(l0_xyz, events)
        # sa2 draws its own randint; capture it by seeding around the call
        s2 = seeded_starts(12, 512, 2)
        l2_xyz, l2_points = net.sa2(l1_xyz, l1_points)
        l3_xyz, l3_points = net.sa3(l2_xyz, l2_points)
    # recover index outputs by re-running the free functions on the same inputs
    xyz0 = l0_xyz.permute(0, 2, 1).contiguous()
    torch.manual_seed(11)
    f1 = pu.farthest_point_sample(xyz0, 512)
    assert torch.equal(pu.index_points(xyz0, f1).permute(0, 2, 1), l1_xyz)
    xyz1 = l1_xyz.permute(0, 2, 1).contiguous()
    torch.manual_seed(12)
    f2 = pu.farthest_point_sample(xyz1, 128)
    c2 = pu.index_points(xyz1, f2)
    assert torch.equal(c2.permute(0, 2, 1), l2_xyz)
    enc = {"events": events.numpy(), "start_sa1": s1.numpy(), "start_sa2": s2.numpy(),
           "fps_sa1": small_idx(f1.numpy()), "fps_sa2": small_idx(f2.numpy()),
           "ball_sa2_r0.4": small_idx(pu.query_ball_point(0.4, 64, xyz1, c2).numpy()),
           "ball_sa2_r0.8": small_idx(pu.query_ball_point(0.8, 128, xyz1, c2).numpy()),
           "l1_xyz": l1_xyz.numpy(), "l2_xyz": l2_xyz.numpy(), "l3_xyz": l3_xyz.numpy(),
           "l1_points_w0": l1_points[0].numpy(), "l2_points_w0": l2_points[0].numpy(),
           "l3_points": l3_points.numpy(), "weight_seeds": np.array([100, 101, 102])}
    np.savez_compressed(os.path.join(HERE, "encoder.npz"), **enc)

    # ---- 4. one hand regressor's sa1 -> sa2 ------------------------------------
    reg = net.left_mano_regressor
    rstates = {n: synth.random_state_for(synth.REGRESSOR_SPECS[n], seed=200 + i)
               for i, n in enumerate(("sa1", "sa2"))}
    for n in rstates:
        getattr(reg, n).load_state_dict(to_t(rstates[n]), strict=True)
    hand = torch.from_numpy(np.random.RandomState(77).randn(2, 4, 2048).astype(np.float32))
    s3 = seeded_starts(13, 2048, 2)
    with torch.no_grad():
        r1_xyz, r1_points = reg.sa1(l0_xyz, hand)
        r2_xyz, r2_points = reg.sa2(r1_xyz, r1_points)
    np.savez_compressed(os.path.join(HERE, "regressor.npz"), events=events.numpy(), hand_feats=hand.numpy(),
                        start_sa1=s3.numpy(), r1_xyz=r1_xyz.numpy(), r1_points_w0=r1_points[0].numpy(),
                        r2_points=r2_points.numpy(), weight_seeds=np.array([200, 201]))

    # ---- 5. decoder fp3 -> fp2 -> fp1 on the encoder's outputs (TEHNet.py:184-186) ----------
    dstates = {n: synth.random_state_for(synth.DECODER_SPECS[n], seed=300 + i) for i, n in enumerate(("fp3", "fp2", "fp1"))}
    for n in dstates:
        getattr(net, n).load_state_dict(to_t(dstates[n]), strict=True)
    # point features are seeded noise (regenerated by the tests, not stored); coordinates are the encoder's
    f1r, f2r, f3r = (torch.from_numpy(a) for a in synth.decoder_test_features(2, seed=55))
    with torch.no_grad():
        d2 = net.fp3(l2_xyz, l3_xyz, f2r, f3r)
        d1 = net.fp2(l1_xyz, l2_xyz, f1r, d2)
        d0 = net.fp1(l0_xyz, l1_xyz, None, d1)
        # the 3-NN tables of fp2 / fp1, recomputed with the reference's own functions (:294-301)
        nn_tabs = {}
        for tag, q, src in (("fp2", l1_xyz, l2_xyz), ("fp1", l0_xyz, l1_xyz)):
            dd, ii = pu.square_distance(q.permute(0, 2, 1).contiguous(), src.permute(0, 2, 1).contiguous()).sort(dim=-1)
            dd, ii = dd[:, :, :3], ii[:, :, :3]
            rc = 1.0 / (dd + 1e-8)
            nn_tabs[tag + "_idx"] = small_idx(ii.numpy())
            nn_tabs[tag + "_weight"] = (rc / torch.sum(rc, dim=2, keepdim=True)).numpy()
    np.savez_compressed(os.path.join(HERE, "decoder.npz"), d2=d2.numpy(), d1_every2=d1[:, :, ::2].numpy(),
                        d0_every16=d0[:, :, ::16].numpy(), weight_seeds=np.array([300, 301, 302]),
                        feature_seed=np.array(55), **nn_tabs)

    # ---- 6. sample_and_group / sampled (group_all=False) PointNetSetAbstraction (:110-138, :161-202) -----
    # not reached by the model (SURVEY 8a row a5); pinned for API completeness
    ev6 = synth.make_windows(2, 512, seed=1240)
    xyz6 = torch.from_numpy(ev6[:, :3].transpose(0, 2, 1).copy())
    pts6 = torch.from_numpy(ev6.transpose(0, 2, 1).copy())                  # [B,N,5]
    s6 = seeded_starts(21, 512, 2)
    g_xyz, g_points, g_grouped, g_fps = pu.sample_and_group(48, 0.3, 16, xyz6, pts6, returnfps=True)
    s6b = seeded_starts(22, 512, 2)
    g_xyz_np, g_points_np = pu.sample_and_group(48, 0.3, 16, xyz6, None)
    sa_s = pu.PointNetSetAbstraction(npoint=48, radius=0.3, nsample=16, in_channel=5 + 3, mlp=[16, 32], group_all=False).eval()
    st6 = synth.random_sa_state("mlp_convs.{j}", "mlp_bns.{j}", [[16, 32]], [8], seed=400)
    sa_s.load_state_dict(to_t(st6), strict=True)
    s6c = seeded_starts(23, 512, 2)
    with torch.no_grad():
        m_xyz, m_points = sa_s(torch.from_numpy(ev6[:, :3].copy()), torch.from_numpy(ev6))
    np.savez_compressed(os.path.join(HERE, "sampled.npz"), events=ev6, start=s6.numpy(), start_nopoints=s6b.numpy(),
                        start_module=s6c.numpy(), new_xyz=g_xyz.numpy(), new_points=g_points.numpy(),
                        grouped_xyz=g_grouped.numpy(), fps_idx=small_idx(g_fps.numpy()),
                        new_points_nopoints=g_points_np.numpy(), module_xyz=m_xyz.numpy(), module_points=m_points.numpy(),
                        weight_seed=np.array(400))

    # ---- 7. training step of the sa2-shaped module at the MODEL's shapes (D=320, K=64/128): forward in train mode
    # (batch-statistics BatchNorm), backward of a fixed linear loss; reference autograd on CPU --------------------
    torch.manual_seed(0)
    sa_t = pu.PointNetSetAbstractionMsg(128, [0.4, 0.8], [64, 128], 320, [[128, 128, 256], [128, 196, 256]]).train()
    st7 = synth.random_state_for(synth.ENCODER_SPECS["sa2"], seed=500)
    sa_t.load_state_dict(to_t(st7), strict=True)
    rs7 = np.random.RandomState(501)
    ev7 = synth.make_windows(2, 512, seed=1250)
    xyz7 = torch.from_numpy(ev7[:, :3].copy())
    feats7 = torch.from_numpy(rs7.randn(2, 320, 512).astype(np.float32)).requires_grad_(True)
    s7 = seeded_starts(31, 512, 2)
    t_xyz, t_out = sa_t(xyz7, feats7)
    lw = torch.from_numpy(np.linspace(0.5, 1.5, t_out.numel(), dtype=np.float32)).view_as(t_out)
    (t_out * lw).sum().backward()
    tr = {"events": ev7, "feats_seed": np.array(501), "start": s7.numpy(), "weight_seed": np.array(500),
          "new_xyz": t_xyz.detach().numpy(), "out_every4": t_out.detach().numpy()[:, ::4, ::4],
          "grad_feats_every8": feats7.grad.numpy()[:, :, ::8],
          "running_mean_0_0": sa_t.bn_blocks[0][0].running_mean.numpy(), "running_var_1_2": sa_t.bn_blocks[1][2].running_var.numpy()}
    for n, p in sa_t.named_parameters():
        if n in ("conv_blocks.0.0.weight", "conv_blocks.1.1.weight", "conv_blocks.1.2.bias", "bn_blocks.0.1.weight", "bn_blocks.1.0.bias"):
            tr["grad." + n] = p.grad.numpy()
    np.savez_compressed(os.path.join(HERE, "train_sa2.npz"), **tr)

    # ---- 8. the heads after the decoder (SURVEY 8f row N2): classifier, per-hand query convolutions, attention
    # (TEHNet.py:188-192) on seeded point features ---------------------------------------------------------------
    hst = synth.random_head_state(seed=600)
    missing = net.load_state_dict(to_t(hst), strict=False)
    assert not missing.unexpected_keys
    feat = torch.from_numpy(np.random.RandomState(66).randn(2, 256, 2048).astype(np.float32))
    with torch.no_grad():
        seg_out = net.classifier(feat)
        left_f = net.attention_block(seg_out, feat, net.left_query_conv(feat))
        right_f = net.attention_block(seg_out, feat, net.right_query_conv(feat))
        lq = net.left_query_conv(feat)
    np.savez_compressed(os.path.join(HERE, "heads.npz"), weight_seed=np.array(600), feature_seed=np.array(66),
                        seg_out=seg_out.numpy(), left_features=left_f.numpy(), right_features=right_f.numpy(),
                        left_query_every8=lq.numpy()[:, :, ::8])

    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)))




def dump_state_dict_layout():
    """Names and shapes of the reference modules' state_dicts (the checkpoint contract,
    demo.py:84 loads with strict=True) -> tests/golden/state_dict_layout.json."""
    import json
    _, th = load_reference()
    net = th.TEHNet(n_pose_params=6)
    out = {}
    for name in ("sa1", "sa2", "sa3"):
        out["encoder." + name] = {k: list(v.shape) for k, v in getattr(net, name).state_dict().items()}
    for name in ("sa1", "sa2"):
        out["regressor." + name] = {k: list(v.shape) for k, v in getattr(net.left_mano_regressor, name).state_dict().items()}
    out["fp1"] = {k: list(v.shape) for k, v in net.fp1.state_dict().items()}
    with open(os.path.join(HERE, "state_dict_layout.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    write_tehnet_layout(net)


def write_tehnet_layout(net):
    """The whole network's state_dict in order, one [name, shape, dtype] per line -> tests/golden/tehnet_layout.json."""
    import json
    rows = [json.dumps([k, list(v.shape), str(v.dtype).replace("torch.", "")]) for k, v in net.state_dict().items()]
    with open(os.path.join(HERE, "tehnet_layout.json"), "w") as f:
        f.write("[\n" + ",\n".join(rows) + "\n]\n")


if __name__ == "__main__":
    main()
    dump_state_dict_layout()
