"""CPU-side checks of the product package: the C-ABI library loads and exports what
include/ev2h.h declares, the drop-in modules keep the reference's checkpoint layout,
and nothing silently runs on the CPU."""
import ctypes
import json
import os

import numpy as np
import pytest
import torch

import ev2hands_b200 as e2h
from ev2hands_b200 import _capi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    L = _capi.lib()
    names = _capi.declared_symbols()
    assert len(names) >= 13 and "ev2h_fps_f32" in names
    for n in names:
        assert hasattr(L, n), "libev2h.so does not export %s" % n
    assert L.ev2h_version() >= 100
    # every declared compute entry has a ctypes signature (the binding covers the whole ABI)
    assert set(names) - {"ev2h_version", "ev2h_last_error", "ev2h_tc_packed_bytes", "ev2h_tc_packed_bytes_kc"} == set(_capi._SIGNATURES)


def test_bad_arguments_return_status_not_crash():
    L = _capi.lib()
    st = L.ev2h_fps_f32(None, 0, 0, 0, None, 1, 1, 1, None, None, None, None)
    assert st == 1
    assert b"null" in L.ev2h_last_error()
    st = L.ev2h_linear_relu_f32(ctypes.c_void_p(16), 8, 6, 6, ctypes.c_void_p(16), ctypes.c_void_p(16), 4, 0,
                                ctypes.c_void_p(16), 4, 0, None)
    assert st == 1 and b"multiple of 4" in L.ev2h_last_error()


def test_state_dict_layout_matches_reference():
    layout = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_layout.json")))
    enc = e2h.SetAbstractionEncoder()
    reg = e2h.RegressorSetAbstraction()
    for prefix, mod in (("encoder", enc), ("regressor", reg)):
        for name, child in mod.named_children():
            want = layout["%s.%s" % (prefix, name)]
            got = {k: list(v.shape) for k, v in child.state_dict().items()}
            assert got == want, (prefix, name)
    fp = e2h.PointNetFeaturePropagation(128, [128, 128, 256])
    assert {k: list(v.shape) for k, v in fp.state_dict().items()} == layout["fp1"]


def test_strict_load_of_reference_shaped_checkpoint():
    enc = e2h.SetAbstractionEncoder()
    for i, n in enumerate(("sa1", "sa2", "sa3")):
        st = synth.random_state_for(synth.ENCODER_SPECS[n], seed=100 + i)
        getattr(enc, n).load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in st.items()}, strict=True)


def test_no_cpu_fallback():
    enc = e2h.SetAbstractionEncoder().eval()
    with pytest.raises(RuntimeError, match="CUDA"):
        enc(torch.zeros(1, 5, 2048))
    with pytest.raises(RuntimeError, match="CUDA"):
        e2h.farthest_point_sample(torch.zeros(1, 64, 3), 8)


def test_feature_propagation_matches_oracle_formula():
    # the decoder block's training-path formulation (host logic) against a direct evaluation of its formula;
    # the module itself has no CPU path
    torch.manual_seed(0)
    fp = e2h.PointNetFeaturePropagation(6 + 5, [8]).eval()
    xyz1, xyz2 = torch.rand(2, 3, 20), torch.rand(2, 3, 7)
    p1, p2 = torch.rand(2, 6, 20), torch.rand(2, 5, 7)
    with pytest.raises(RuntimeError, match="no CPU path"):
        fp(xyz1, xyz2, p1, p2)
    with torch.no_grad():
        got = fp._forward_autograd(xyz1, xyz2, p1, p2)
    a, b = xyz1.permute(0, 2, 1), xyz2.permute(0, 2, 1)
    d = ((a[:, :, None] - b[:, None]) ** 2).sum(-1)
    dd, ii = d.topk(3, dim=-1, largest=False)
    w = 1 / (dd + 1e-8)
    w = w / w.sum(-1, keepdim=True)
    f2 = p2.permute(0, 2, 1)
    up = torch.stack([(f2[bi][ii[bi]] * w[bi][..., None]).sum(1) for bi in range(2)])
    h = torch.cat([p1.permute(0, 2, 1), up], -1).permute(0, 2, 1)
    with torch.no_grad():
        want = torch.relu(fp.mlp_bns[0](fp.mlp_convs[0](h)))
    assert torch.allclose(got, want, atol=1e-4)


def test_synthetic_windows_are_deterministic_and_event_like():
    a = synth.make_windows(3, 2048, seed=5)
    b = synth.make_windows(3, 2048, seed=5)
    assert np.array_equal(a, b) and a.shape == (3, 5, 2048) and a.dtype == np.float32
    assert np.abs(a[:, :3]).max() <= 1.0 + 1e-6
    # sampling with replacement leaves many exact duplicates (erpc.py:213)
    uniq = len({tuple(p) for p in a[0, :3].T})
    assert uniq < 0.8 * 2048
    assert (a[:, 3:] >= 0).all() and (a[:, 3:] == np.round(a[:, 3:])).all()


def test_event_window_builder_host_logic_and_no_cpu_path():
    """EventWindowBuilder (SURVEY 8f N3): argument checks happen on the host, nothing is computed without a GPU,
    and the C ABI rejects bad arguments with a status instead of crashing."""
    raw = torch.from_numpy(synth.make_raw_events(300, seed=3))
    wb = e2h.EventWindowBuilder("stream", n_events=64)
    with pytest.raises(RuntimeError, match="no CPU path"):
        wb(raw, [0], [300])
    with pytest.raises(IndexError):
        wb.aggregate(raw, [200], [101])
    with pytest.raises(RuntimeError, match="at least one event"):
        wb.aggregate(raw, [0], [0])
    with pytest.raises(RuntimeError, match="equally long"):
        wb.aggregate(raw, [0, 1], [10])
    with pytest.raises(ValueError):
        e2h.EventWindowBuilder("frames")
    L = _capi.lib()
    assert L.ev2h_window_aggregate_f64(None, 4, None, None, 1, 16, 346, 260, 0, None, None, None, None) == 1
    p = ctypes.c_void_p(64)
    assert L.ev2h_window_aggregate_f64(p, 4, p, p, 1, 5000, 346, 260, 1, p, p, p, None) == 2      # erpc: <= 4096 events
    assert b"exceed" in L.ev2h_last_error()
    assert L.ev2h_window_aggregate_f64(p, 4, p, p, 1, 16, 346, 260, 7, p, p, p, None) == 1 and b"mode" in L.ev2h_last_error()
    assert L.ev2h_window_aggregate_f64(p, 4, p, p, 1, 16, 4096, 4096, 0, p, p, p, None) == 1      # pixel number must fit the sort key
    assert L.ev2h_window_sample_f32(p, 16, p, p, 0, 64, 346, 260, p, p, None) == 1


def test_raw_event_stream_is_deterministic_and_sensor_shaped():
    a = synth.make_raw_events(4096, seed=9, t0=5.0, duration=1.0e4, extra_columns=2)
    b = synth.make_raw_events(4096, seed=9, t0=5.0, duration=1.0e4, extra_columns=2)
    assert np.array_equal(a, b) and a.shape == (4096, 6) and a.dtype == np.float64
    assert (np.diff(a[:, 2]) >= 0).all() and a[0, 2] >= 5.0
    assert (a[:, 0] >= 0).all() and (a[:, 0] < synth.SENSOR_W).all() and (a[:, 1] < synth.SENSOR_H).all()
    assert set(np.unique(a[:, 3])) <= {0.0, 1.0}
    u = synth.make_raw_events(2000, seed=1, duration=1.0e5, unique_times=True)
    assert np.unique(u[:, 2]).size == 2000


def test_header_is_plain_c_and_links_from_c(tmp_path):
    """include/ev2h.h must be consumable from C (the boundary is a C ABI, not a C++ or Python one): a C99 program
    that takes the address of every declared function links against libev2h.so, reports the version and gets a
    status + message (not a crash) for a bad call."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    names = [n for n in _capi.declared_symbols()]
    src = tmp_path / "abi.c"
    src.write_text(
        '#include <stdio.h>\n#include <string.h>\n#include "ev2h.h"\n'
        "int main(void) {\n"
        "    typedef void (*fn_t)(void);\n"
        "    fn_t fns[] = {" + ", ".join("(fn_t)%s" % n for n in names) + "};\n"
        "    size_t i, n = sizeof(fns) / sizeof(fns[0]);\n"
        "    for (i = 0; i < n; ++i) if (!fns[i]) return 2;\n"
        "    if (ev2h_fps_f32(NULL, 0, 0, 0, NULL, 1, 1, 1, NULL, NULL, NULL, NULL) != EV2H_ERR_BAD_ARGUMENT) return 3;\n"
        '    if (!strstr(ev2h_last_error(), "null")) return 4;\n'
        '    printf("%d %d\\n", ev2h_version(), (int)n);\n'
        "    return 0;\n}\n")
    exe = tmp_path / "abi"
    lib_dir = os.path.dirname(_capi.LIB_PATH)
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe),
                           "-L", lib_dir, "-l:libev2h.so", "-Wl,-rpath," + lib_dir])
    out = subprocess.check_output([str(exe)], text=True).split()
    assert int(out[0]) >= 100 and int(out[1]) == len(names)


# The original Ev2Hands project is not part of this repository: the test that runs its own TEHNet.py reads it from the
# checkout EV2HANDS_REFERENCE names and skips without one.
REF_MODEL_DIR = os.path.join(os.environ.get("EV2HANDS_REFERENCE", ""), "src", "Ev2Hands", "model")
HAVE_REF = bool(os.environ.get("EV2HANDS_REFERENCE")) and os.path.isdir(REF_MODEL_DIR)


def _load_tehnet(pkg_name, pointnet2_module=None):
    """TEHNet.py of the reference, loaded by path under a stand-in package (model/__init__ imports trimesh / manopth,
    absent here).  ``pointnet2_module`` given = the one-line change of INTEGRATION.md: TEHNet.py:6's
    ``from .pointnet2_utils import ...`` resolves to that module instead of the reference's file."""
    import importlib.util
    import sys
    import types
    pkg = types.ModuleType(pkg_name)
    pkg.__path__ = [REF_MODEL_DIR]
    sys.modules[pkg_name] = pkg
    if pointnet2_module is not None:
        sys.modules[pkg_name + ".pointnet2_utils"] = pointnet2_module
    spec = importlib.util.spec_from_file_location(pkg_name + ".TEHNet", os.path.join(REF_MODEL_DIR, "TEHNet.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[pkg_name + ".TEHNet"] = mod
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.skipif(not HAVE_REF, reason="needs a checkout of the original Ev2Hands project in EV2HANDS_REFERENCE")
def test_one_line_change_builds_the_real_tehnet_and_loads_its_checkpoint(monkeypatch):
    """SURVEY 7 step 6 / INTEGRATION.md: the UNMODIFIED reference TEHNet.py with line 6 pointed at ev2hands_b200
    constructs (TEHNet.__init__ :115-166, both MANORegressors :43-44 included), has the stock net's state_dict
    names and shapes, and loads the stock net's state_dict with strict=True (demo.py:84)."""
    monkeypatch.setenv("ERPC", "1")
    from ev2hands_b200 import pointnet2_utils as ours
    stock = _load_tehnet("refmodel_stock").TEHNet(n_pose_params=6)
    patched_mod = _load_tehnet("refmodel_patched", ours)
    patched = patched_mod.TEHNet(n_pose_params=6)
    for name in ("sa1", "sa2"):
        assert isinstance(getattr(patched, name), ours.PointNetSetAbstractionMsg)
        assert not isinstance(getattr(stock, name), ours.PointNetSetAbstractionMsg)
    assert isinstance(patched.sa3, ours.PointNetSetAbstraction) and isinstance(patched.fp1, ours.PointNetFeaturePropagation)
    assert isinstance(patched.left_mano_regressor.sa1, ours.PointNetSetAbstractionMsg)
    assert isinstance(patched.right_mano_regressor.sa2, ours.PointNetSetAbstraction)
    sd_stock, sd_new = stock.state_dict(), patched.state_dict()
    assert list(sd_stock.keys()) == list(sd_new.keys())
    assert {k: tuple(v.shape) for k, v in sd_stock.items()} == {k: tuple(v.shape) for k, v in sd_new.items()}
    assert {k: v.dtype for k, v in sd_stock.items()} == {k: v.dtype for k, v in sd_new.items()}
    res = patched.load_state_dict(sd_stock, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    for k, v in patched.state_dict().items():
        assert torch.equal(v, sd_stock[k]), k
    # and back: a checkpoint written by the patched net loads into the stock one
    stock.load_state_dict(patched.state_dict(), strict=True)
    # the patched net refuses to run on the CPU instead of silently falling back
    with pytest.raises(RuntimeError, match="CUDA"):
        patched.eval()(torch.zeros(1, 5, 2048), {"left": None, "right": None})


def test_tehnet_wiring_has_the_reference_checkpoint_layout_and_attention_matches(monkeypatch, golden):
    """ev2hands_b200.tehnet.TEHNet (the wiring the training configuration and rows N2 / N4 run on): the state_dict
    names in order, shapes and dtypes of the reference's TEHNet (tests/golden/tehnet_layout.json), a strict load of a
    checkpoint of that layout, and the classifier, query convolutions and AttentionBlock (TEHNet.py:9-27) equal to the
    reference's outputs on the CPU (tests/golden/heads.npz)."""
    monkeypatch.setenv("ERPC", "1")
    from ev2hands_b200 import tehnet
    with open(os.path.join(ROOT, "tests", "golden", "tehnet_layout.json")) as f:
        layout = [(k, tuple(s), d) for k, s, d in json.load(f)]
    ours = tehnet.TEHNet(n_pose_params=6)
    assert [(k, tuple(v.shape), str(v.dtype).replace("torch.", "")) for k, v in ours.state_dict().items()] == layout
    # the stored layout agrees with what the reference wrote or loaded itself: its modules' layouts
    # (state_dict_layout.json) and the decoder and head weights of the golden vectors
    shapes = {k: list(s) for k, s, _ in layout}
    parts = json.load(open(os.path.join(ROOT, "tests", "golden", "state_dict_layout.json")))
    g = golden("heads")
    head_state = synth.random_head_state(seed=int(g["weight_seed"]))
    for name, prefixes in (("encoder.sa1", ["sa1"]), ("encoder.sa2", ["sa2"]), ("encoder.sa3", ["sa3"]), ("fp1", ["fp1"]),
                           ("regressor.sa1", ["left_mano_regressor.sa1", "right_mano_regressor.sa1"]),
                           ("regressor.sa2", ["left_mano_regressor.sa2", "right_mano_regressor.sa2"])):
        for p in prefixes:
            assert {k[len(p) + 1:]: s for k, s in shapes.items() if k.startswith(p + ".")} == parts[name], p
    for n in ("fp3", "fp2"):
        want = {k: list(np.shape(v)) for k, v in synth.random_state_for(synth.DECODER_SPECS[n], seed=0).items()}
        assert {k[len(n) + 1:]: s for k, s in shapes.items() if k.startswith(n + ".")} == want, n
    assert all(shapes[k] == list(np.shape(v)) for k, v in head_state.items())
    gen = torch.Generator().manual_seed(1)
    ckpt = {k: (torch.randn(s, generator=gen) if d.startswith("float") else torch.randint(0, 100, s, generator=gen)).to(getattr(torch, d))
            for k, s, d in layout}
    ours.load_state_dict(ckpt, strict=True)
    assert all(torch.equal(v, ckpt[k]) for k, v in ours.state_dict().items())
    # the heads after the decoder, with the reference's golden weights and features
    res = ours.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in head_state.items()}, strict=False)
    assert not res.unexpected_keys
    ours.eval()
    feat = torch.from_numpy(np.random.RandomState(int(g["feature_seed"])).randn(2, 256, 2048).astype(np.float32))
    with torch.no_grad():
        seg = ours.classifier(feat)
        lq, rq = ours.left_query_conv(feat), ours.right_query_conv(feat)
        got = {"seg_out": seg, "left_query_every8": lq[:, :, ::8],
               "left_features": ours.attention_block(seg, feat, lq), "right_features": ours.attention_block(seg, feat, rq)}
    for name, t in got.items():
        want = torch.from_numpy(g[name])
        # same modules, same weights: equal up to the last bits another CPU's summation order may change
        assert torch.allclose(t, want, rtol=1e-5, atol=1e-6 * float(want.abs().max())), name


def test_standin_mano_layer_and_training_losses():
    """the MANO-shaped stand-in (parity unpinned, DESIGN.md) has MANO's interface and is differentiable; the criterion
    (losses.py:145-206 minus loss_interpen) gives finite terms with the reference's names"""
    from ev2hands_b200 import tehnet
    hands = tehnet.create_standin_mano_layers("cpu", n_cmps=6)
    B = 3
    go = torch.randn(B, 3, requires_grad=True)
    out = hands["left"](global_orient=go, hand_pose=torch.randn(B, 6), betas=torch.randn(B, 10), transl=torch.randn(B, 3))
    assert out.vertices.shape == (B, 778, 3) and out.joints.shape == (B, 21, 3)
    assert hands["left"].faces.shape == (1538, 3) and hands["left"].shapedirs.shape == (778, 3, 10)
    out.joints.sum().backward()
    assert torch.isfinite(go.grad).all() and go.grad.abs().sum() > 0
    # zero pose / shape / translation: the template, joints from the regressor
    z = hands["right"](global_orient=torch.zeros(1, 3), hand_pose=torch.zeros(1, 6) , betas=torch.zeros(1, 10), transl=torch.zeros(1, 3))
    again = hands["right"](global_orient=torch.zeros(1, 3), hand_pose=torch.zeros(1, 6), betas=torch.zeros(1, 10), transl=torch.ones(1, 3))
    assert torch.allclose(again.vertices, z.vertices + 1, atol=1e-6) and torch.allclose(again.joints, z.joints + 1, atol=1e-6)
    batch = tehnet.make_training_batch(B, 256, seed=3)
    assert batch["events"].shape == (B, 5, 256) and batch["class_logits"].shape == (B, 256) and batch["handedness"].shape == (B, 2)
    outs = {"class_logits": torch.randn(B, 4, 256, requires_grad=True)}
    for side in ("left", "right"):
        p = {"global_orient": torch.randn(B, 3), "hand_pose": torch.randn(B, 6), "betas": torch.randn(B, 10), "transl": torch.randn(B, 3)}
        o = hands[side](**p)
        outs[side] = dict(p, vertices=o.vertices, j3d=o.joints)
    losses = tehnet.training_losses(outs, batch, hands)
    assert set(losses) == {"loss_inter_shape", "loss_inter_transl", "loss_inter_j3d", "loss_global_orient", "loss_hand_pose",
                           "loss_rj3d", "loss_j3d", "loss_shape", "loss_transl", "loss_class_logits"}
    total = sum(losses.values())
    assert torch.isfinite(total)
    total.backward()
    assert outs["class_logits"].grad.abs().sum() > 0


def test_bench_reference_arm_prints_the_contract_line(tmp_path):
    """`bench.py --impl reference` (the arm the driver times beside ours) runs the oracle port on the host and prints ONE
    JSON line with the keys the driver reads; no GPU, no kernel of this repo.  --dump-outputs writes the last step's
    features; --steps below 1 is refused."""
    import json
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    bad = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "0"],
                         capture_output=True, text=True, timeout=600, cwd=root)
    assert bad.returncode != 0 and "--steps" in bad.stderr
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                          "--dump-outputs", str(tmp_path / "dump")], capture_output=True, text=True, timeout=600, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "encoder event-windows/s" and d["unit"] == "windows/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d.get("gpu_launches", 0) == 0
    assert os.listdir(tmp_path / "dump") == ["features.npy"]
    feats = np.load(tmp_path / "dump" / "features.npy")
    assert feats.dtype == np.float32 and feats.shape == (4, 1024) and np.isfinite(feats).all()


def test_bench_dump_keeps_a_fixed_sample_of_a_large_batch(tmp_path):
    """bench.py's --dump-outputs writer: a batch over the size budget is cut to the same seeded sample of windows every
    time, with the window numbers beside it, and the files stay within the budget."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    feats = np.random.RandomState(3).randn(500, 1024).astype(np.float32)
    for d in ("a", "b"):
        bench.dump_features(str(tmp_path / d), feats, budget=400_000)
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 400_000
    rows = np.load(tmp_path / "a" / "features_windows.npy")
    got = np.load(tmp_path / "a" / "features.npy")
    assert rows.dtype == np.float64 and len(rows) == len(got) > 0 and (np.diff(rows) > 0).all()
    assert np.array_equal(got, feats[rows.astype(np.int64)])
    for f in ("features.npy", "features_windows.npy"):
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes()
    bench.dump_features(str(tmp_path / "small"), feats[:8])
    assert os.listdir(tmp_path / "small") == ["features.npy"]
    assert np.array_equal(np.load(tmp_path / "small" / "features.npy"), feats[:8])
