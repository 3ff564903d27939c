#!/usr/bin/env python
"""Benchmark of the set-abstraction encoder hot path: event-windows per second.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One *step* is one forward of the encoder stack sa1 -> sa2 -> sa3 (TEHNet.py:172-181) over
one batch of synthetic event windows ([B, 5, 2048] float32, ev2hands_b200.synth).  At N=1
the workload is BASELINE.json configs[1] (64 windows on one B200); for N>1 every rank
processes its own 64 windows (weak scaling: windows are independent, no collective on the
inference path) and `value` is the total windows of all ranks divided by the slowest
rank's device time.

Printed JSON (one line, rank 0): the driver contract plus
  roofline      dominant kernel (the shared-MLP layers) against the measured tensor peak
  kernels       device ms per step and launches per step of every kernel of the path
  cpu_baseline  the oracle port of the reference encoder timed on the host cores
  e2e           the same metric through the public module API with host buffers
                (pinned H2D of the windows + D2H of the features inside the timed region)

--impl reference times the CPU oracle port of the reference (oracle/sa_oracle.py, the
reference's algorithm op for op; /root/reference itself does not exist on the GPU box).

--dump-outputs DIR writes the per-window features of the last timed step to DIR/features.npy
(float32 [B, 1024]; one features_rank<r>.npy per rank on several GPUs).  The inputs and weights
are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WINDOWS_PER_GPU = 64
N_POINTS = 2048
# dense multiply-accumulates per window of sa1+sa2+sa3 (SURVEY.md 8d), 2 flops each
MLP_MAC_PER_WINDOW = 4_468_080_640
ALGO_BYTES_PER_WINDOW = 1_900_000       # compulsory HBM traffic per window (SURVEY.md 8d)
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
DUMP_BYTES_MAX = 64_000_000             # --dump-outputs: all files of one run together


def dump_features(directory: str, feats: np.ndarray, name: str = "features", budget: int = DUMP_BYTES_MAX):
    """Writes feats [B, C] as <directory>/<name>.npy in float32.  A batch larger than the budget keeps a fixed, seeded
    sample of its windows (the same for every build), and <name>_windows.npy (float64) holds their numbers."""
    feats = np.ascontiguousarray(feats, dtype=np.float32)
    os.makedirs(directory, exist_ok=True)
    if feats.nbytes > budget - 4096:                       # 4 KiB for the .npy headers
        n_keep = (budget - 4096) // (feats[0].nbytes + 8)
        keep = np.sort(np.random.RandomState(0).choice(len(feats), n_keep, replace=False))
        np.save(os.path.join(directory, name + "_windows.npy"), keep.astype(np.float64))
        feats = feats[keep]
    np.save(os.path.join(directory, name + ".npy"), feats)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return {k: float(d[k]) for k in FALLBACK_PEAKS}, "measured"
        except Exception:
            pass
    return dict(FALLBACK_PEAKS), "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
            nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
            nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
            nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._halt.wait(self.period)

    def finish(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ----------------------------------------------------------------------------- CPU oracle arm ----
def oracle_states():
    from ev2hands_b200 import synth
    return {n: synth.random_state_for(synth.ENCODER_SPECS[n], seed=100 + i) for i, n in enumerate(("sa1", "sa2", "sa3"))}


def time_cpu_oracle(n_windows: int, reps: int, warmup: int, device: str = "cpu", threads: int | None = None):
    """Reference algorithm (oracle port) on the host - or, device="cuda", the same stock-PyTorch ops on the GPU,
    the comparator SURVEY.md 8d asks for since the reference ships no kernels: returns (windows/s, threads, seconds per rep,
    features [n_windows, 1024] of the last rep)."""
    from ev2hands_b200 import synth
    from oracle import sa_oracle
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    states = oracle_states()
    ev = torch.from_numpy(synth.make_windows(n_windows, N_POINTS, seed=1234 + 1)).to(device)
    starts = {"sa1": torch.from_numpy(synth.make_start_indices(n_windows, N_POINTS, 0)).to(device),
              "sa2": torch.from_numpy(synth.make_start_indices(n_windows, 512, 1)).to(device)}
    cuda = device != "cpu"
    old_tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    if cuda:                                     # fp32 arithmetic, like the reference on its own hardware
        torch.backends.cudnn.allow_tf32 = False
        torch.backends.cuda.matmul.allow_tf32 = False
    times = []
    with torch.no_grad():
        for i in range(warmup + reps):
            if cuda:
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            out = sa_oracle.encoder_forward(states, synth.ENCODER_SPECS, ev, starts)
            if cuda:
                torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_tf32
    return n_windows / (sum(times) / len(times)), threads, times, out.squeeze(-1)


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    sample = 4
    t0 = time.perf_counter()
    wps, threads, times, feats = time_cpu_oracle(sample, args.steps, max(1, min(args.warmup, 2)))
    if args.dump_outputs:
        dump_features(args.dump_outputs, feats.float().cpu().numpy())
    line = {
        "impl": "reference", "metric": "encoder event-windows/s", "value": wps, "unit": "windows/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * float(np.mean(times)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "encoder forward sa1->sa2->sa3, %d-window sample of the batch-64 workload per step, "
                               "N=2048 points/window, random-init weights, host CPU" % sample},
        "cpu_baseline": {"value": wps, "unit": "windows/s", "cores": threads, "kind": "port",
                         "sample": "%d windows per step x %d steps (oracle/sa_oracle.py, torch CPU)" % (sample, len(times))},
        "e2e": {"value": wps, "unit": "windows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line))
    return 0



# ----------------------------------------------------------------------------- secondary configs -
def mlp_kernel_ms(kern):
    n_, ms_ = 0, 0.0
    for kname in ("ev2h_linear_relu_f32", "ev2h_linear_relu_tc", "ev2h_linear_f32", "ev2h_linear_tc", "ev2h_sa_msg_fused_tc"):
        a, b = kern.get(kname, (0, 0.0))
        n_, ms_ = n_ + a, ms_ + b
    return n_, ms_


def time_encoder_config(enc, device, B_local, n_points, seed, rank, world, steps, flush, barrier, precision, graph=True):
    """One BASELINE config of the encoder forward on this rank's shard: `steps` timed steps (CUDA events per step, L2
    flushed between steps, graph replay when it captures) and an eager pass with events around every kernel.
    -> dict(ms_total, kern, graphed); the caller takes the max over ranks."""
    import ev2hands_b200 as e2h
    import ev2hands_b200.encoder as _enc_mod
    from ev2hands_b200 import _capi, sharding, synth
    from ev2hands_b200.encoder import GraphedForward
    old_prec = e2h.get_mlp_precision()
    e2h.set_mlp_precision(precision)
    try:
        ev_all = synth.make_windows(B_local * world, n_points, seed=seed)
        s1_all = synth.make_start_indices(B_local * world, n_points, 0)
        s2_all = synth.make_start_indices(B_local * world, 512, 1)
        ev, s1, s2 = sharding.shard((torch.from_numpy(ev_all), torch.from_numpy(s1_all), torch.from_numpy(s2_all)), rank, world)
        ev, s1, s2 = ev.to(device), s1.to(device), s2.to(device)

        def fwd(e, a, b):
            with torch.no_grad():
                return enc(e, fps_starts=(a, b))

        graphed = None
        if graph:
            try:
                graphed = GraphedForward(fwd, ev, s1, s2)
            except Exception as exc:      # noqa: BLE001
                print("bench.py: capture failed for B=%d N=%d (%s); eager" % (B_local, n_points, exc), file=sys.stderr)
        run = (lambda: graphed(ev, s1, s2)) if graphed is not None else (lambda: fwd(ev, s1, s2))
        for _ in range(3):
            run()
        barrier()
        evs = []
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = run()
            b.record()
            evs.append((a, b))
        barrier()
        ms_total = float(sum(a.elapsed_time(b) for a, b in evs))
        geom_stream = _enc_mod._GEOM_STREAM
        _enc_mod._GEOM_STREAM = False
        _capi.LOG.reset(timing=True)
        try:
            for _ in range(steps):
                flush.zero_()
                fwd(ev, s1, s2)
            barrier()
            kern = _capi.LOG.totals_ms()
        finally:
            _capi.LOG.reset(timing=False)
            _enc_mod._GEOM_STREAM = geom_stream
        return {"ms_total": ms_total, "kern": kern, "graphed": graphed is not None, "checksum": float(out.double().sum().item())}
    finally:
        e2h.set_mlp_precision(old_prec)


def config_line(name, res, ms_total, B_global, n_points, steps, precision, peaks):
    n_mlp, mlp_ms = mlp_kernel_ms(res["kern"])
    world_share = res["world"]                             # kernel times are this rank's shard of the global batch
    ach = (2.0 * MLP_MAC_PER_WINDOW * (B_global // world_share) * steps) / (mlp_ms / 1e3) / 1e12 if mlp_ms > 0 else None
    geo = sum(res["kern"].get(k, (0, 0.0))[1] for k in ("ev2h_fps_f32", "ev2h_ball_query_f32", "ev2h_first_occurrence_u8"))
    tot_k = sum(v[1] for v in res["kern"].values())
    return {"workload": name, "global_windows": B_global, "windows_per_gpu": B_global // world_share, "points": n_points,
            "mlp": precision, "steps": steps, "ms_per_step": ms_total / steps, "value": B_global * steps / (ms_total / 1e3),
            "unit": "windows/s", "launch": "graph replay" if res["graphed"] else "eager",
            "roofline_frac": (ach / peaks["bf16_tflops"]) if ach else None, "mlp_tflops": ach,
            "fps_ball_share_of_kernel_time": (geo / tot_k) if tot_k > 0 else None,
            "kernels_ms_per_step": {k: v[1] / steps for k, v in sorted(res["kern"].items())}}


def time_training_config(device, rank, world, steps, barrier):
    """BASELINE configs[3]: full training step of the network (ev2hands_b200.tehnet.TEHNet: set abstraction, feature
    propagation, classifier, attention, both hand regressors; MANO LBS and the criterion in PyTorch - MANO is a
    MANO-shaped stand-in and loss_interpen is left out, both unavailable here), global batch 32 split over the ranks,
    per-replica BatchNorm statistics, gradients averaged with bucketed NCCL all-reduces launched from backward hooks,
    Adam.  -> dict of per-rank timings (ms) for the caller's max over ranks."""
    from ev2hands_b200 import sharding, tehnet, trainer
    os.environ.setdefault("ERPC", "1")
    old_tf32 = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    torch.backends.cudnn.allow_tf32 = False          # fp32 convolutions, like the reference on its own hardware
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        torch.manual_seed(0)                          # same initial weights on every rank
        net = tehnet.TEHNet(n_pose_params=6).to(device).train()
        hands = tehnet.create_standin_mano_layers(device, n_cmps=6)
        opt = torch.optim.Adam(net.parameters(), lr=1e-3)       # train.py:23,56
        red = trainer.BucketedGradReducer(net.parameters(), n_buckets=4)
        full = tehnet.make_training_batch(32, N_POINTS, seed=0)
        lo, hi = sharding.shard_bounds(32, rank, world)

        def cut(x):
            return {k: cut(v) for k, v in x.items()} if isinstance(x, dict) else x[lo:hi].to(device)
        batch = cut(full)
        n_params = sum(p.numel() for p in net.parameters())

        def step():
            b = {k: (dict(v) if isinstance(v, dict) else v) for k, v in batch.items()}      # the criterion adds fields
            return trainer.train_step(net, hands, b, opt, red, tehnet.training_losses)

        for _ in range(2):
            loss, _ = step()
        barrier()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            loss, _ = step()
        b_.record()
        barrier()
        step_ms = a.elapsed_time(b_) / steps
        # the exchange alone: one blocking all-reduce of the whole flat gradient buffer
        ar_ms = 0.0
        if world > 1:
            import torch.distributed as dist
            for _ in range(2):
                dist.all_reduce(red.flat)
            barrier()
            c, d = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c.record()
            for _ in range(5):
                dist.all_reduce(red.flat)
            d.record()
            barrier()
            ar_ms = c.elapsed_time(d) / 5
        out = {"step_ms": step_ms, "allreduce_ms": ar_ms, "grad_bytes": red.bytes, "params": n_params, "loss": float(loss.detach()),
               "buckets": len(red.buckets), "local_batch": hi - lo}
        red.remove()
        del net, opt, red
        torch.cuda.empty_cache()
        return out
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = old_tf32

# ----------------------------------------------------------------------------- GPU arm -----------
def build_encoder(device):
    import ev2hands_b200 as e2h
    from ev2hands_b200 import synth
    from ev2hands_b200.encoder import load_numpy_state
    enc = e2h.SetAbstractionEncoder()
    for i, n in enumerate(("sa1", "sa2", "sa3")):
        load_numpy_state(getattr(enc, n), synth.random_state_for(synth.ENCODER_SPECS[n], seed=100 + i))
    return enc.to(device).eval()


def run_ours(args):
    import torch.distributed as dist
    from ev2hands_b200 import _capi, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the ev2hands_b200 path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=device)
    if args.gpus != world and rank == 0:
        print("bench.py: --gpus %d but WORLD_SIZE=%d; using WORLD_SIZE" % (args.gpus, world), file=sys.stderr)

    B = args.windows_per_gpu
    import ev2hands_b200 as e2h
    e2h.set_mlp_precision(args.mlp)
    enc = build_encoder(device)
    # Every rank owns its shard of the global batch; starts are generated for the global batch
    # and sharded with the data so results do not depend on the shard count.
    ev_all = synth.make_windows(B * world, args.points, seed=1234 + 2)
    s1_all = synth.make_start_indices(B * world, args.points, 0)
    s2_all = synth.make_start_indices(B * world, 512, 1)
    from ev2hands_b200 import sharding
    ev_sh, s1_sh, s2_sh = sharding.shard((torch.from_numpy(ev_all), torch.from_numpy(s1_all), torch.from_numpy(s2_all)), rank, world)
    ev_host = ev_sh.contiguous().pin_memory()
    s1 = s1_sh.to(device)
    s2 = s2_sh.to(device)
    ev_dev = ev_host.to(device)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=device)     # > 126 MB L2

    def forward_resident(ev, a, b):
        with torch.no_grad():
            return enc(ev, fps_starts=(a, b))

    graphed = None
    if args.graph:
        # the ~35 launches of a step replayed as one CUDA graph (inputs resident, shapes fixed); eager if capture fails
        try:
            from ev2hands_b200.encoder import GraphedForward
            graphed = GraphedForward(forward_resident, ev_dev, s1, s2)
        except Exception as exc:      # noqa: BLE001
            print("bench.py: CUDA graph capture failed (%s); timing the eager path" % exc, file=sys.stderr)
            graphed = None

    def step_resident():
        if graphed is not None and not _capi.LOG.timing:
            return graphed(ev_dev, s1, s2)
        return forward_resident(ev_dev, s1, s2)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step_resident()
    barrier()

    # ---- instrumented pass (eager): per-kernel device time from CUDA events around every launch, same K steps,
    # same L2 flush; feeds the roofline (time of the MLP kernels) and the launch count
    # (one stream here, so that a kernel's bracket holds that kernel alone: the headline steps run sa2's FPS and
    # ball query on a second stream beside sa1's MLP kernels)
    import ev2hands_b200.encoder as _enc_mod
    geom_stream = _enc_mod._GEOM_STREAM
    _enc_mod._GEOM_STREAM = False
    _capi.LOG.reset(timing=True)
    barrier()
    for _ in range(args.steps):
        flush.zero_()
        forward_resident(ev_dev, s1, s2)
    barrier()
    launches = _capi.LOG.count
    kern = _capi.LOG.totals_ms()
    _capi.LOG.reset(timing=False)
    _enc_mod._GEOM_STREAM = geom_stream

    # ---- timed region: K steps, device time per step from CUDA events, L2 flushed between steps
    sampler = ClockSampler(physical_gpu_index(local_rank))
    sampler.start()
    evs = []
    barrier()
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = step_resident()
        b.record()
        evs.append((a, b))
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.finish()
    step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = float(sum(step_ms))
    # of the timed steps' result (fixed windows and FPS starts): taken now, because a replayed graph returns its static
    # output buffer and the end-to-end leg below overwrites it with the result of randomly drawn start indices
    headline_checksum = float(out.double().sum().item())
    if args.dump_outputs:
        dump_features(args.dump_outputs, out.float().cpu().numpy(), "features" if world == 1 else "features_rank%d" % rank,
                      DUMP_BYTES_MAX // world)

    # rows the fused kernel evaluated in the headline step / dense B*S*K rows, per scale (read now: the later legs run
    # other batch sizes through the same modules)
    comp = {}
    for name in ("sa1", "sa2"):
        m = getattr(enc, name)
        if getattr(m, "last_compact_rows", None) is not None:
            rows = m.last_compact_rows.cpu().tolist()
            comp[name] = [r / float(B * m.npoint * k) for r, k in zip(rows, m.nsample_list)]

    # ---- transparency: the same K steps with the row compaction switched off (every padded / duplicate neighbour
    # evaluated like the reference does; identical output bits), eager launches
    import ev2hands_b200.pointnet2_utils as _pu
    dense_ms = 0.0
    if _pu._COMPACT:
        _pu._COMPACT = False
        try:
            for _ in range(2):
                forward_resident(ev_dev, s1, s2)
            barrier()
            d_evs = []
            for _ in range(args.steps):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                out_dense = forward_resident(ev_dev, s1, s2)
                b.record()
                d_evs.append((a, b))
            barrier()
            dense_ms = float(sum(a.elapsed_time(b) for a, b in d_evs))
            dense_equal = bool(torch.equal(out_dense, out))
        finally:
            _pu._COMPACT = True

    # ---- end to end through the public API with host buffers: every step copies its windows from pinned host
    # memory, runs the forward (graph replay when captured, else eager; FPS start indices drawn on the host like the
    # reference does) and reads the per-window features back.  The copies run on their own stream, double buffered, so step i+1's upload overlaps
    # step i's kernels - as a serving loop would; the timed region is the whole loop (uploads, L2 flushes, kernels,
    # read-backs), one event pair around K steps.
    out_host = [torch.empty((B, 1024), dtype=torch.float32).pin_memory() for _ in range(2)]
    ev_stage = [torch.empty_like(ev_dev) for _ in range(2)]
    copy_stream = torch.cuda.Stream()

    # FPS start indices: drawn on the host like the reference (two torch.randint draws, pointnet2_utils.py:75) and
    # uploaded with the step's windows on the copy stream; the read-back of step i also runs on the copy stream, beside
    # the L2 flush of step i + 1 (the next replay waits for it: the graph's output buffer is static)
    h1_pin = [torch.empty((B,), dtype=torch.long).pin_memory() for _ in range(2)]
    h2_pin = [torch.empty((B,), dtype=torch.long).pin_memory() for _ in range(2)]
    h1_dev = [torch.empty((B,), dtype=torch.long, device=device) for _ in range(2)]
    h2_dev = [torch.empty((B,), dtype=torch.long, device=device) for _ in range(2)]

    def run_e2e(k):
        main = torch.cuda.current_stream()
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]
        done = [torch.cuda.Event() for _ in range(2)]
        read = [torch.cuda.Event() for _ in range(2)]

        def upload(i):
            j = i % 2
            if graphed is not None:
                if i >= 2:
                    ready[j].synchronize()                      # the pinned start buffers of step i - 2 have been uploaded
                torch.randint(0, args.points, (B,), dtype=torch.long, out=h1_pin[j])
                torch.randint(0, 512, (B,), dtype=torch.long, out=h2_pin[j])
            with torch.cuda.stream(copy_stream):
                if i >= 2:
                    copy_stream.wait_event(freed[j])          # the step that last read these buffers is done
                ev_stage[j].copy_(ev_host, non_blocking=True)
                if graphed is not None:
                    h1_dev[j].copy_(h1_pin[j], non_blocking=True)
                    h2_dev[j].copy_(h2_pin[j], non_blocking=True)
                ready[j].record(copy_stream)

        copy_stream.wait_stream(main)
        upload(0)
        for i in range(k):
            j = i % 2
            flush.zero_()
            if i + 1 < k:
                upload(i + 1)
            main.wait_event(ready[j])
            if graphed is not None:
                # the serving-loop API (ev2hands_b200.encoder.GraphedForward): the step's windows and start indices are
                # copied into the graph's input buffers, one replay
                if i >= 1:
                    main.wait_event(read[(i - 1) % 2])          # the previous output has left the static buffer
                o = graphed(ev_stage[j], h1_dev[j], h2_dev[j])
                freed[j].record(main)
                done[j].record(main)
                with torch.cuda.stream(copy_stream):
                    copy_stream.wait_event(done[j])
                    out_host[j].copy_(o, non_blocking=True)
                    read[j].record(copy_stream)
            else:
                with torch.no_grad():
                    o = enc(ev_stage[j])
                out_host[j].copy_(o, non_blocking=True)
                freed[j].record(main)
        main.wait_stream(copy_stream)                           # the last read-back is inside the timed region

    run_e2e(2)
    barrier()
    ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ea.record()
    run_e2e(args.steps)
    eb.record()
    barrier()
    e2e_ms = float(ea.elapsed_time(eb))

    # ---- optional secondary number: encoder + feature-propagation decoder (SURVEY 8f row N1), same timing rules
    dec_ms = 0.0
    if args.with_decoder:
        from ev2hands_b200.encoder import load_numpy_state
        dec = e2h.FeaturePropagationDecoder()
        for i, n in enumerate(("fp3", "fp2", "fp1")):
            load_numpy_state(getattr(dec, n), synth.random_state_for(synth.DECODER_SPECS[n], seed=300 + i))
        dec = dec.to(device).eval()
        l3_xyz = torch.zeros((B, 3, 1), dtype=torch.float32, device=device)

        def fwd_dec(ev_, s1_, s2_):
            with torch.no_grad():
                l3, lv = enc(ev_, fps_starts=(s1_, s2_), return_levels=True)
                return dec(ev_[:, :3, :], lv["l1_xyz"], lv["l2_xyz"], l3_xyz, lv["l1_points"], lv["l2_points"], l3.unsqueeze(-1))

        dec_graph = None
        if args.graph:
            try:                                   # one graph replay per step, like the headline (eager launches are host bound on some boxes)
                from ev2hands_b200.encoder import GraphedForward
                dec_graph = GraphedForward(fwd_dec, ev_dev, s1, s2)
            except Exception as exc:      # noqa: BLE001
                print("bench.py: decoder leg runs eager (%s)" % exc, file=sys.stderr)

        def step_dec():
            return dec_graph(ev_dev, s1, s2) if dec_graph is not None else fwd_dec(ev_dev, s1, s2)

        for _ in range(3):
            step_dec()
        barrier()
        d_evs = []
        for _ in range(args.steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            step_dec()
            b.record()
            d_evs.append((a, b))
        barrier()
        dec_ms = float(sum(a.elapsed_time(b) for a, b in d_evs))

    # ---- optional secondary number: raw events resident in HBM -> windows -> encoder features.  The N points of a
    # window are drawn on the host from numpy's generator exactly like the reference (one read-back of the pixel
    # counts per batch, np.random.choice per window), so this line includes that host work.
    raw_ms = raw_dev_ms = 0.0
    if args.from_raw_events and (args.points > 4096 or world > 1):
        # a 2048-event window has fewer occupied pixels than config 5 wants points; the scaling runs time the headline only
        args.from_raw_events = False
    if args.from_raw_events:
        try:
            import numpy as _np
            n_raw = 2048
            raw = synth.make_raw_events(B * n_raw // 2 + n_raw, seed=77, duration=2.0e3 * (B // 2 + 1))
            w_starts, w_counts = _np.arange(B) * (n_raw // 2), _np.full(B, n_raw)       # half-overlapping 2048-event windows
            raw_dev = torch.from_numpy(raw).to(device)
            wb = e2h.EventWindowBuilder("stream", n_events=args.points)
            fixed_idx = torch.from_numpy(_np.random.RandomState(5).randint(0, 1024, size=(B, args.points))).to(device)

            def step_raw(host_draw):
                with torch.no_grad():
                    return enc(wb(raw_dev, w_starts, w_counts, sample_idx=None if host_draw else fixed_idx), fps_starts=(s1, s2))

            for host_draw, slot in ((True, "raw_ms"), (False, "raw_dev_ms")):
                for _ in range(3):
                    step_raw(host_draw)
                barrier()
                r_evs = []
                for _ in range(args.steps):
                    flush.zero_()
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    step_raw(host_draw)
                    b.record()
                    r_evs.append((a, b))
                barrier()
                t = float(sum(a.elapsed_time(b) for a, b in r_evs))
                if slot == "raw_ms":
                    raw_ms = t
                else:
                    raw_dev_ms = t
        except Exception as exc:      # noqa: BLE001 - a secondary number must not take the headline down
            print("bench.py: raw-events leg failed (%s)" % exc, file=sys.stderr)
            raw_ms = raw_dev_ms = 0.0

    # ---- secondary configs of BASELINE.json, every line of the run (VERDICT r01 item 1): config 3 = 1024 windows
    # split over the ranks, config 5 = 16384-event windows, 256 split over the ranks, fp32-level and bf16 MLP;
    # and a sustained figure: the headline loop for >= 2 s with the clocks sampled
    cfg_res, sustained = {}, None
    if args.configs:
        plan = [("cfg3", max(1, 1024 // world), N_POINTS, args.mlp, min(args.steps, 5), 1234 + 3)]
        plan += [("cfg5_" + pr, max(1, 256 // world), 16384, pr, 3, 1234 + 5) for pr in dict.fromkeys((args.mlp, "bf16"))]
        for name, b_loc, n_pts, prec, k, seed in plan:
            try:
                r = time_encoder_config(enc, device, b_loc, n_pts, seed, rank, world, k, flush, barrier, prec, graph=args.graph)
            except Exception as exc:      # noqa: BLE001 - a secondary number must not take the headline down
                print("bench.py: %s failed (%s)" % (name, exc), file=sys.stderr)
                r = {"ms_total": 0.0, "kern": {}, "graphed": False, "checksum": 0.0}
            r.update(world=world, B_global=b_loc * world, n_points=n_pts, precision=prec, steps=k)
            cfg_res[name] = r
            torch.cuda.empty_cache()
        # sustained: the headline step for >= 2 s (one event pair around the loop, L2 flushed every step, clocks sampled)
        n_sus = int(min(4000, max(args.steps, 2200.0 / max(total_ms / args.steps, 0.05))))
        for _ in range(3):
            step_resident()
        sus_sampler = ClockSampler(physical_gpu_index(local_rank), period_s=0.02)
        barrier()
        sus_sampler.start()
        sa_, sb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sa_.record()
        for _ in range(n_sus):
            flush.zero_()
            step_resident()
        sb_.record()
        barrier()
        sustained = {"steps": n_sus, "ms_total": float(sa_.elapsed_time(sb_)), "clocks": sus_sampler.finish()}

    # whole-network inference (secondary): the reference's TEHNet.forward wiring in eval mode - encoder, decoder,
    # classifier + query convolutions + attention, both hand regressors' set abstraction + FC head, stand-in MANO layer
    full_ms = 0.0
    if args.configs:
        try:
            from ev2hands_b200 import tehnet as _th
            os.environ.setdefault("ERPC", "1")
            torch.manual_seed(0)
            fnet = _th.TEHNet(n_pose_params=6).to(device).eval()
            fhands = _th.create_standin_mano_layers(device)

            def full_step():
                with torch.no_grad():
                    return fnet(ev_dev, fhands)

            for _ in range(3):
                full_step()
            barrier()
            f_evs = []
            for _ in range(args.steps):
                flush.zero_()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                full_step()
                b.record()
                f_evs.append((a, b))
            barrier()
            full_ms = float(sum(a.elapsed_time(b) for a, b in f_evs))
            del fnet
        except Exception as exc:      # noqa: BLE001
            print("bench.py: full-network leg failed (%s)" % exc, file=sys.stderr)
            full_ms = 0.0
        full_ms = sharding.max_over_ranks([full_ms], device=device)[0]

    train_res = None
    if args.configs:
        try:
            train_res = time_training_config(device, rank, world, max(3, min(args.steps, 5)), barrier)
        except Exception as exc:      # noqa: BLE001
            print("bench.py: cfg4 (training step) failed (%s)" % exc, file=sys.stderr)
            train_res = None
        ok = sharding.max_over_ranks([0.0 if train_res is not None else 1.0], device=device)[0] == 0.0
        if ok:
            train_res["step_ms"], train_res["allreduce_ms"] = sharding.max_over_ranks([train_res["step_ms"], train_res["allreduce_ms"]], device=device)
        else:
            train_res = None

    # ---- max over ranks
    total_ms, e2e_ms, dec_ms, dense_ms, raw_ms, raw_dev_ms = sharding.max_over_ranks(
        [total_ms, e2e_ms, dec_ms, dense_ms, raw_ms, raw_dev_ms], device=device)
    cfg_names = sorted(cfg_res)
    if cfg_names:
        mx = sharding.max_over_ranks([cfg_res[n]["ms_total"] for n in cfg_names] + [sustained["ms_total"]], device=device)
        for n, v in zip(cfg_names, mx[:-1]):
            cfg_res[n]["ms_total_max"] = v
        sustained["ms_total"] = mx[-1]
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks, peak_kind = load_peaks()
    windows = B * world * args.steps
    value = windows / (total_ms / 1e3)
    mlp_n, mlp_ms = 0, 0.0
    for kname in ("ev2h_linear_relu_f32", "ev2h_linear_relu_tc", "ev2h_linear_f32", "ev2h_linear_tc", "ev2h_sa_msg_fused_tc"):
        n_, ms_ = kern.get(kname, (0, 0.0))
        mlp_n, mlp_ms = mlp_n + n_, mlp_ms + ms_
    mlp_flops_per_step = 2.0 * MLP_MAC_PER_WINDOW * B
    achieved_tflops = (mlp_flops_per_step * args.steps) / (mlp_ms / 1e3) / 1e12 if mlp_ms > 0 else None
    # the bench's timed region is a few ms long: burst peak applies (kernel timed in isolation)
    peak_tflops = peaks["bf16_tflops"]
    traffic = None
    prof = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    if os.path.exists(prof):
        try:
            traffic = json.load(open(prof)).get("mlp_dram_bytes_per_step")
        except Exception:
            traffic = None
    line = {
        "metric": "encoder event-windows/s", "value": value, "unit": "windows/s", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": {"fp32": "f32", "tf32x3": "f32 (split tf32 + bf16 corrections, fp32 accumulate)", "bf16": "bf16"}[args.mlp], "data": "synthetic",
        "config": {"workload": "encoder forward sa1->sa2->sa3 (TEHNet.py:172-181), %d windows per GPU, "
                               "N=%d points/window, 5 channels, random-init weights, eval mode" % (B, args.points),
                   "windows_per_gpu": B, "global_windows": B * world,
                   "mlp_path": {"fp32": "fp32 FFMA (CUDA cores)", "tf32x3": "tcgen05 3-product split x=hi+lo, w=hi+lo: tf32 hi*hi + two bf16 correction products (fp32-level accuracy)",
                                "bf16": "tcgen05 kind::f16 bf16 operands, fp32 accumulate"}[args.mlp],
                   "l2": "256 MiB buffer written between timed steps (L2 flush)",
                   "rows": "compacted: padded and exact-duplicate neighbours are evaluated once (bit-identical pooled features; EV2H_COMPACT=0 evaluates the dense groups, timed under compaction.dense_rows_eager)",
                   "launch": "one CUDA graph replay per step" if graphed is not None else "eager launches through the module API",
                   "kernel_times": "separate eager single-stream pass of the same K steps with CUDA events around every launch",
                   "streams": "sa2's FPS + ball query on a second stream beside sa1's MLP kernels" if geom_stream else "one stream",
                   "layout": "levels stay in point-major rows between layers; channel-first copies only on request"},
        "roofline": {"bound": "tensor", "achieved": achieved_tflops, "peak": peak_tflops, "unit": "TFLOP/s",
                     "frac": (achieved_tflops / peak_tflops) if achieved_tflops else None, "traffic": traffic,
                     "kernel": "%s (shared MLP, %d launches/step)" % ("linear_relu_kernel" if args.mlp == "fp32" else "sa_fused_tc_kernel + linear_tc_kernel", mlp_n // max(args.steps, 1)),
                     "peak_source": "%s bf16 dense (burst)" % peak_kind,
                     "algorithmic_flops_per_launch_set": mlp_flops_per_step,
                     "hbm_view": {"algorithmic_bytes_per_step": ALGO_BYTES_PER_WINDOW * B,
                                  "achieved_gbs_whole_step": ALGO_BYTES_PER_WINDOW * B * args.steps / (total_ms / 1e3) / 1e9,
                                  "peak_gbs": peaks["hbm_gbs"]}},
        "kernels": {k: {"launches_per_step": n / args.steps, "ms_per_step": ms / args.steps} for k, (n, ms) in sorted(kern.items())},
        "e2e": {"value": windows / (e2e_ms / 1e3), "unit": "windows/s", "ms_per_step": e2e_ms / args.steps,
                "h2d_bytes_per_step": int(ev_host.numel() * 4 + 2 * B * 8), "d2h_bytes_per_step": int(out_host[0].numel() * 4),
                "timed": "one event pair around K steps incl. uploads of the windows and the host-drawn FPS starts (copy stream, double buffered), "
                         "L2 flushes, " + ("graph replays (GraphedForward)" if graphed is not None else "eager forwards")
                         + ", read-backs (copy stream, beside the next step's L2 flush; the last one is waited for inside the region)"},
        "gpu_launches": launches, "clocks": clocks, "wall_s": wall,
        "checksum": headline_checksum,
    }
    # rows the fused kernel evaluates / dense B*S*K rows per scale: padded duplicate neighbours are skipped
    # (bit-identical pooled features); roofline.achieved counts the dense algorithmic FLOPs (SURVEY 8d)
    line["compaction"] = {"rows_evaluated_fraction": comp} if comp else None
    if comp and dense_ms > 0:
        line["compaction"]["dense_rows_eager"] = {"value": windows / (dense_ms / 1e3), "unit": "windows/s", "ms_per_step": dense_ms / args.steps,
                                                  "output_bits_equal": dense_equal}
    from ev2hands_b200 import pointnet2_utils as _pu2
    line["row_shortcut"] = dict(_pu2.ROW_SHORTCUT)      # levels handed over as rows (hit) vs transposed back (stale / none)
    line["transposes_per_step"] = kern.get("ev2h_transpose_f32", (0, 0.0))[0] / args.steps
    if cfg_res:
        cfgs = {}
        for n in sorted(cfg_res):
            r = cfg_res[n]
            if r["ms_total"] <= 0:
                cfgs[n] = {"failed": True}
                continue
            what = {"cfg3": "BASELINE configs[2]: encoder forward, batch 1024 split over the ranks, no collective"}.get(
                n, "BASELINE configs[4]: long-window stress, 16384-event windows, batch 256 split over the ranks")
            cfgs[n] = config_line(what, r, r["ms_total_max"], r["B_global"], r["n_points"], r["steps"], r["precision"], peaks)
        if "cfg5_bf16" in cfgs and ("cfg5_" + args.mlp) in cfgs and args.mlp != "bf16":
            a_, b_ = cfg_res["cfg5_" + args.mlp], cfg_res["cfg5_bf16"]
            cfgs["cfg5_bf16"]["checksum_rel_diff_vs_fp32_level"] = abs(a_["checksum"] - b_["checksum"]) / max(abs(a_["checksum"]), 1e-30)
        line["configs"] = cfgs
        mlp_share = mlp_ms / max(sum(v[1] for v in kern.values()), 1e-9)
        sus_ms = sustained["ms_total"]
        sus_tflops = (mlp_flops_per_step * sustained["steps"]) / (sus_ms * mlp_share / 1e3) / 1e12
        line["sustained"] = {"value": B * world * sustained["steps"] / (sus_ms / 1e3), "unit": "windows/s", "steps": sustained["steps"],
                             "seconds": sus_ms / 1e3, "ms_per_step": sus_ms / sustained["steps"], "clocks": sustained["clocks"],
                             "roofline_frac": sus_tflops / peaks["bf16_tflops_sustained"], "peak": peaks["bf16_tflops_sustained"],
                             "how": "the headline step repeated for >= 2 s, one event pair around the loop, L2 flushed every step; "
                                    "MLP time = loop time x the MLP kernels' share of the per-kernel pass (%.3f); peak = measured sustained bf16" % mlp_share}
    if full_ms > 0:
        line.setdefault("configs", {})["full_network_eval"] = {
            "workload": "TEHNet.forward wiring in eval mode (TEHNet.py:168-197): encoder + decoder + classifier + query convolutions + "
                        "attention + two hand regressors (set abstraction on the kernels, FC head and stand-in MANO layer in PyTorch), "
                        "%d windows per GPU, eager launches, host-drawn FPS starts" % B,
            "ms_per_step": full_ms / args.steps, "value": windows / (full_ms / 1e3), "unit": "windows/s"}
    if train_res is not None:
        line.setdefault("configs", {})["cfg4"] = {
            "workload": "BASELINE configs[3]: full training step (set abstraction + feature propagation + classifier + attention + two hand "
                        "regressors forward/backward on the GPU, MANO LBS + criterion in PyTorch), global batch 32 split over the ranks, "
                        "per-replica BatchNorm, bucketed NCCL gradient all-reduce from backward hooks, Adam",
            "global_batch": 32, "batch_per_gpu": train_res["local_batch"], "ms_per_step": train_res["step_ms"],
            "value": 32.0 / (train_res["step_ms"] / 1e3), "unit": "windows/s", "params": train_res["params"],
            "grad_allreduce_bytes": train_res["grad_bytes"], "grad_buckets": train_res["buckets"],
            "allreduce_us_alone": 1e3 * train_res["allreduce_ms"], "loss": train_res["loss"], "dtype": "f32 (TF32 off)",
            "stand_ins": "MANO layer = random MANO-shaped LBS (assets licence gated); criterion = losses.py:145-206 without loss_interpen "
                         "(mesh_intersection absent): parity of those two parts unpinned",
            "kernels": "FPS, ball query, grouping gather + scatter-add backward, input-gradient GEMMs of the 1x1 convolutions (tcgen05 layer "
                       "kernel, tf32 / bf16 split), weight + bias gradients (exact fp32, deterministic), forward GEMMs of layers with >= 96 "
                       "outputs (exact fp32): libev2h.so; narrower forward GEMMs: cuBLAS fp32; BatchNorm (batch statistics) / ReLU / max "
                       "over K: PyTorch; k = 3 convolutions of the heads: cuDNN"}
    if args.with_decoder:
        line["secondary"] = {"metric": "encoder + fp3/fp2/fp1 decoder event-windows/s (TEHNet.py:172-186)",
                             "value": windows / (dec_ms / 1e3), "unit": "windows/s", "ms_per_step": dec_ms / args.steps}
    if args.from_raw_events and raw_ms > 0 and raw_dev_ms > 0:
        line["from_raw_events"] = {
            "metric": "raw events (2048 per window, resident in HBM) -> windows -> encoder features, windows/s",
            "value": windows / (raw_ms / 1e3), "unit": "windows/s", "ms_per_step": raw_ms / args.steps,
            "draw": "host: pixel counts read back, np.random.choice per window like the reference (erpc.py:217)",
            "device_only": {"value": windows / (raw_dev_ms / 1e3), "unit": "windows/s", "ms_per_step": raw_dev_ms / args.steps,
                            "draw": "indices resident on the device"}}
    if world == 1 and not args.no_cpu_baseline and "from_raw_events" in line:
        # the reference's numpy recipe for the same windows on one host core (oracle/window_oracle.py, pinned bit for
        # bit to the reference's dataset classes): np.add.at grids, nonzero, draw, pc_normalize
        try:
            import numpy as _np
            from oracle import window_oracle as _wo
            raw_h = synth.make_raw_events(16 * 1024 + 2048, seed=77, duration=2.0e3 * 17)
            t0 = time.perf_counter()
            for w in range(16):
                r = _wo.aggregate(raw_h[w * 1024:w * 1024 + 2048], "stream")
                _wo.sample_normalize(r, _np.random.RandomState(w).randint(0, r.shape[0], size=args.points))
            line["from_raw_events"]["cpu_window_recipe"] = {"value": 16 / (time.perf_counter() - t0), "unit": "windows/s", "cores": 1,
                                                            "kind": "port", "sample": "16 windows of 2048 raw events, window construction only"}
        except Exception as exc:      # noqa: BLE001
            print("bench.py: CPU window recipe failed (%s)" % exc, file=sys.stderr)
    if world == 1 and not args.no_cpu_baseline:
        wps, threads, times, _ = time_cpu_oracle(4, 3, 1)
        line["cpu_baseline"] = {"value": wps, "unit": "windows/s", "cores": threads, "kind": "port",
                                "sample": "4 windows per run, 1 warm-up + 3 timed runs of oracle/sa_oracle.py (torch CPU, "
                                          "the reference's algorithm op for op)"}
        # BASELINE configs[0] (B = 1 on the host, the reference's own CPU-runnable case; BASELINE.md 3): min / median of
        # 5 runs after 2 warm-ups, all host threads and one thread
        try:
            cfg1 = {}
            for label, nthr in (("all_threads", os.cpu_count() or 1), ("one_thread", 1)):
                _, _, t1, _ = time_cpu_oracle(1, 5, 2, threads=nthr)
                cfg1[label] = {"threads": nthr, "windows_per_s_best": 1.0 / min(t1), "windows_per_s_median": 1.0 / float(np.median(t1)),
                               "ms_min": 1e3 * min(t1), "ms_median": 1e3 * float(np.median(t1))}
            line["cpu_baseline"]["cfg1_batch1"] = cfg1
        except Exception as exc:      # noqa: BLE001
            line["cpu_baseline"]["cfg1_batch1"] = {"unavailable": str(exc)[:200]}
        try:      # the same stock-PyTorch ops on this GPU (the reference ships no kernels): informational comparator
            gwps, _, _, _ = time_cpu_oracle(WINDOWS_PER_GPU, 2, 1, device="cuda")
            line["torch_gpu_baseline"] = {"value": gwps, "unit": "windows/s", "kind": "port",
                                          "sample": "64 windows per run (the workload's batch), 1 warm-up + 2 timed runs of oracle/sa_oracle.py on cuda:0 "
                                                    "(stock PyTorch fp32 ops, Python FPS loop, materialised distance matrices)"}
        except Exception as exc:      # noqa: BLE001
            line["torch_gpu_baseline"] = {"unavailable": str(exc)[:200]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1, got %d" % v)
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=10, help="timed steps of the headline")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the features the last timed step computed to DIR/features.npy (float32)")
    ap.add_argument("--windows-per-gpu", type=int, default=WINDOWS_PER_GPU)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", dest="configs", action="store_false",
                    help="skip the secondary configs (cfg3 / cfg5 / sustained) and time the headline only")
    ap.add_argument("--no-graph", dest="graph", action="store_false", help="time eager launches instead of a CUDA graph replay")
    ap.add_argument("--with-decoder", action="store_true", help="also time encoder + feature-propagation decoder (secondary number)")
    ap.add_argument("--from-raw-events", dest="from_raw_events", action="store_true", default=True,
                    help="also time raw events -> windows (EventWindowBuilder, SURVEY 8f N3) -> encoder (secondary number; default on)")
    ap.add_argument("--no-raw-events", dest="from_raw_events", action="store_false")
    ap.add_argument("--points", type=int, default=N_POINTS, help="events per window (2048 = the model's default; 16384 = config 5)")
    ap.add_argument("--mlp", choices=["fp32", "tf32x3", "bf16"], default=os.environ.get("EV2H_MLP", "tf32x3"),
                    help="arithmetic of the shared MLP: fp32 = CUDA-core FFMA, tf32x3 = tensor cores with fp32-level "
                         "accuracy (bar 1e-5), bf16 = tensor cores, bf16 operands (bar 1e-2)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
