"""Bit-exact envelope of the geometry kernels: farthest point sampling (csrc/fps.cu), the multi-radius ball query
and its in-kernel row compaction (csrc/ball_query.cu), the two-step compaction and the duplicate flags (csrc/compact.cu).

Every index these kernels produce decides which points a group holds, so a wrong one is not a small numerical error:
it must be caught where it happens.  The cases here reach every kernel instance the dispatch code can pick (derived from
its thresholds in `test_every_kernel_instance_is_reached`), on inputs chosen for ties, cancellation, degenerate extent,
underflow and non-finite coordinates, in the row layout and in the strided channel-first view the model passes:

* FPS and the ball query against the C oracle (oracle/sa_oracle_c.c), bit for bit;
* the inclusive radius rule on points built to lie exactly on fp32(r^2) and one ulp either side of it;
* float64 properties that hold whatever the rounding (they guard the oracle too), and the torch oracle
  (oracle/sa_oracle.py, the reference's own ops) against the C oracle on the small inputs;
* resumable sampling and range-wise compaction against their one-shot entries;
* duplicate flags against a bytes-based first occurrence.

Oracle results are cached per input inside the module; every kernel case runs once.
"""
import functools

import numpy as np
import pytest
import torch

from ev2hands_b200 import _capi, synth
from oracle import c_oracle, sa_oracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U = 2.0 ** -24                      # unit roundoff of fp32
LAYOUTS = ("rows", "cf")            # [B,N,3] rows, and the strided view ev[:, :3, :] of a [B,5,N] tensor


# ================================================================== inputs ==========================================
FINITE_KINDS = ("events", "uniform", "lattice", "offset", "clusters", "line", "plane", "same", "tiny", "subnormal",
                "signed_zero")
NONFINITE_KINDS = ("nan", "inf")
NO_BOUNDS = {"nan", "inf", "tiny", "subnormal"}          # relative float64 bounds do not hold there (non-finite, underflow)


def _nonfinite_positions(N):
    return sorted({0, N // 2, N - 1}), sorted({min(1, N - 1), N // 3, N - 1})


@functools.lru_cache(maxsize=None)
def make_xyz(kind, B, N, seed):
    """[B,N,3] float32 (read-only) of one input kind."""
    rs = np.random.RandomState(seed)
    if kind in ("events", "offset", "nan", "inf"):
        x = np.ascontiguousarray(synth.make_windows(B, N, seed=seed)[:, :3].transpose(0, 2, 1))
        if kind == "offset":                     # cancellation in p - c and |p|^2 ~ 3e6: many rounding ties
            x = x + np.float32(1e3)
        elif kind == "nan":
            pos, _ = _nonfinite_positions(N)
            for j, p in enumerate(pos):
                x[:, p, j % 3] = np.nan
        elif kind == "inf":
            _, pos = _nonfinite_positions(N)
            for j, p in enumerate(pos):
                x[:, p, j % 3] = np.inf
    elif kind == "uniform":
        x = np.ascontiguousarray(synth.make_windows(B, N, seed=seed, mode="uniform")[:, :3].transpose(0, 2, 1))
    elif kind == "lattice":                      # equal distances between different points, exactly representable
        x = rs.randint(-4, 5, size=(B, N, 3)) / np.float32(4.0)
    elif kind == "clusters":                     # two clusters 1e2 apart
        x = rs.uniform(-1, 1, size=(B, N, 3))
        x[rs.rand(B, N) < 0.5] += 100.0
    elif kind == "line":
        t = rs.uniform(-1, 1, size=(B, N, 1))
        x = np.array([0.1, -0.2, 0.3]) + t * np.array([0.6, -0.8, 0.0])
    elif kind == "plane":
        x = rs.uniform(-1, 1, size=(B, N, 3))
        x[..., 2] = 0.3
    elif kind == "same":
        x = np.broadcast_to(np.array([0.25, -0.5, 0.75]), (B, N, 3))
    elif kind == "tiny":                         # squares (~1e-46) underflow to 0: every distance ties at 0
        x = rs.uniform(-3e-23, 3e-23, size=(B, N, 3))
    elif kind == "subnormal":                    # squares ~1e-40 are subnormal: no flush to zero allowed
        x = rs.uniform(-1e-20, 1e-20, size=(B, N, 3))
    elif kind == "signed_zero":                  # +0.0 and -0.0 mixed with a few non-zero values
        x = rs.choice(np.array([0.0, -0.0, 0.0, -0.0, 0.5, -0.5]), size=(B, N, 3))
    else:
        raise ValueError(kind)
    x = np.ascontiguousarray(x, dtype=np.float32)
    x.setflags(write=False)
    return x


def to_device(xyz, layout, seed=0):
    """-> (tensor, strides) in the requested layout; the channel-first view keeps two extra channels beside xyz."""
    B, N, _ = xyz.shape
    if layout == "rows":
        t = torch.from_numpy(np.ascontiguousarray(xyz)).to(DEV)
        return t, _capi.rows_strides(t)
    ev = np.empty((B, 5, N), np.float32)
    ev[:, :3] = xyz.transpose(0, 2, 1)
    ev[:, 3:] = np.random.RandomState(seed).randint(0, 4, size=(B, 2, N))
    view = torch.from_numpy(ev).to(DEV)[:, :3, :]
    return view, _capi.cf_strides(view)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def gather_rows(xyz, idx):
    return np.stack([xyz[b][idx[b]] for b in range(xyz.shape[0])])


# ================================================================== oracles (cached per input) ======================
@functools.lru_cache(maxsize=None)
def oracle_fps(kind, B, N, seed, S, start):
    """C oracle FPS; a shorter sampling is a prefix of a longer one, so callers ask once for the longest."""
    return c_oracle.fps(make_xyz(kind, B, N, seed), S, np.array(start, np.int64))


@functools.lru_cache(maxsize=None)
def oracle_ball(kind, B, N, seed, centre_key, r, K):
    return c_oracle.ball_query(r, K, make_xyz(kind, B, N, seed), _CENTRES[centre_key])


_CENTRES = {}


def first_occurrence_np(pts8):
    """first[b, n] = 1 iff no earlier record of window b has the same 32 bytes."""
    B, N, _ = pts8.shape
    out = np.zeros((B, N), np.uint8)
    for b in range(B):
        _, idx = np.unique(np.ascontiguousarray(pts8[b]).view(np.dtype((np.void, 32))).ravel(), return_index=True)
        out[b, idx] = 1
    return out


def real_count(lst, N):
    """hits in one padded oracle list: its distinct leading entries (0 for the all-N sentinel of an empty ball)"""
    return 0 if lst[0] == N else len(np.unique(lst))


# ================================================================== kernel wrappers (return host arrays) =============
def k_fps(xyz, layout, start, S, variant=0):
    B, N, _ = xyz.shape
    x, st = to_device(xyz, layout, seed=N)
    idx, rows, cf = _capi.fps(x, st, torch.from_numpy(np.asarray(start, np.int64)), B, N, S, variant=variant)
    return idx.cpu().numpy(), rows.cpu().numpy(), cf.cpu().numpy()


def k_fps_ranges(xyz, layout, start, S, cuts):
    B, N, _ = xyz.shape
    x, st = to_device(xyz, layout, seed=N)
    sd = _capi.device_starts(torch.from_numpy(np.asarray(start, np.int64)), B, N, x.device)
    idx = torch.full((B, S), -7, dtype=torch.int32, device=DEV)
    rows = torch.full((B, S, 3), -7.0, device=DEV)
    cf = torch.full((B, 3, S), -7.0, device=DEV)
    best = torch.empty((B, N), device=DEV)
    cur = torch.empty((B,), dtype=torch.int32, device=DEV)
    for lo, hi in cuts:
        _capi.fps_range(x, st, sd, B, N, S, lo, hi, best, cur, idx, rows, cf)
    return idx.cpu().numpy(), rows.cpu().numpy(), cf.cpu().numpy()


def k_ball_all(xyz, layout, centres, radii, Ks, flags):
    """every ball-query entry on one input -> dict of host arrays"""
    B, N, _ = xyz.shape
    x, st = to_device(xyz, layout, seed=N + 1)
    c = torch.from_numpy(np.ascontiguousarray(centres)).to(DEV)
    out = {"plain": _capi.ball_query(x, st, c, N, radii, Ks).cpu().numpy()}
    idx, cnt = _capi.ball_query(x, st, c, N, radii, Ks, with_counts=True)
    out["idx"], out["cnt"] = idx.cpu().numpy(), cnt.cpu().numpy()
    fl = torch.from_numpy(flags).to(DEV)
    i2, uniq, ucnt = _capi.ball_query_uniq(x, st, c, N, radii, Ks, fl)
    out["uidx"], out["uniq"], out["ucnt"] = i2.cpu().numpy(), uniq.cpu().numpy(), ucnt.cpu().numpy()
    if all(k % 8 == 0 for k in Ks):
        for name, f in (("compact", None), ("compact_dedup", fl)):
            i3, rm, bg, nr = _capi.ball_query_compact(x, st, c, N, radii, Ks, f)
            out[name] = (i3.cpu().numpy(), [t.cpu().numpy() for t in rm], [t.cpu().numpy() for t in bg], nr.cpu().numpy())
    return out


def k_group_compact(lists, cnt, N, Ks):
    rm, bg, nr = _capi.group_compact(torch.from_numpy(np.ascontiguousarray(lists, np.int32)).to(DEV),
                                     torch.from_numpy(np.ascontiguousarray(cnt, np.int32)).to(DEV), N, Ks)
    return [t.cpu().numpy() for t in rm], [t.cpu().numpy() for t in bg], nr.cpu().numpy()


def k_compact_range(xyz, layout, centres, radii, Ks, flags, ranges):
    B, N, _ = xyz.shape
    S = centres.shape[1]
    x, st = to_device(xyz, layout, seed=N + 2)
    c = torch.from_numpy(np.ascontiguousarray(centres)).to(DEV)
    fl = None if flags is None else torch.from_numpy(flags).to(DEV)
    out = torch.full((B, S, sum(Ks)), -7, dtype=torch.int32, device=DEV)
    uniq = None if flags is None else torch.full_like(out, -7)
    rm = [torch.full((B * S * k,), -7, dtype=torch.int32, device=DEV) for k in Ks]
    bg = [torch.full((B * S * k // 8,), -7, dtype=torch.int32, device=DEV) for k in Ks]
    nr = torch.full((len(Ks),), 12345, dtype=torch.int32, device=DEV)
    for j, (lo, cnt) in enumerate(ranges):
        _capi.ball_query_compact_range(x, st, c, B, N, S, lo, cnt, j == 0, radii, Ks, out, fl, uniq, rm, bg, nr)
    return (out.cpu().numpy(), None if uniq is None else uniq.cpu().numpy(), [t.cpu().numpy() for t in rm],
            [t.cpu().numpy() for t in bg], nr.cpu().numpy())


def k_first(pts8):
    return _capi.first_occurrence(torch.from_numpy(np.ascontiguousarray(pts8)).to(DEV)).cpu().numpy()


def k_sqdist(centres, xyz):
    return _capi.square_distance(torch.from_numpy(np.ascontiguousarray(centres)).to(DEV),
                                 torch.from_numpy(np.ascontiguousarray(xyz)).to(DEV)).cpu().numpy()


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ================================================================== instances (fps_dispatch, ball_query_impl) =======
def fps_instance(N, variant, B, sms):
    """the kernel ev2h_fps_f32 / ev2h_fps_variant_f32 launches (fps.cu: fps_dispatch, default switches)"""
    for n_max, name in ((128, "fps<32,4,4>"), (256, "fps<64,4,4>"), (512, "fps<128,4,4>"), (1024, "fps<256,4,4>"),
                        (2048, "fps<256,8,8>"), (4096, "fps<512,8,8>")):
        if N <= n_max:
            return name
    if variant == 0:
        resident = B * (2 if N <= 8192 else 4) <= sms
        variant = 2 if resident and N > 8192 else 3
    if variant == 2:
        return "cluster<2>" if N <= 8192 else "cluster<4>"
    if variant == 3:
        return "pruned<16>" if N <= 8192 else "pruned<32>"
    return "fps<1024,8,8>" if N <= 8192 else "fps<1024,16,6>"


def fps_range_instance(N):
    for n_max, name in ((128, "range<32,4,4>"), (256, "range<64,4,4>"), (512, "range<128,4,4>"), (1024, "range<256,4,4>"),
                        (2048, "range<256,8,8>")):
        if N <= n_max:
            return name
    return "range<512,8,8>"


def uniq_slots(N):
    s = 8192
    while s < 2 * N:
        s *= 2
    return s


# ================================================================== §2 FPS against the C oracle =====================
FPS_NS = [1, 2, 31, 32, 33, 127, 128, 129, 200, 255, 256, 257, 511, 512, 513, 1023, 1024, 1025, 2047, 2048, 2049,
          4095, 4096, 4097, 8191, 8192, 8193, 16383, 16384]
_ROTATE = ("uniform", "lattice", "offset", "clusters", "line", "plane", "same", "tiny", "subnormal", "signed_zero")


def fps_plan(N):
    """(kind, B, S_max, [S ...], starts) per input at N; S_max = N + 7 runs once per window class, so S = N and S > N
    (all minima 0: the reference then picks index 0) are covered at every N"""
    i = FPS_NS.index(N)
    typ = max(1, min(512, N // 4))
    big = N > 4096
    kinds = ["events", _ROTATE[i % len(_ROTATE)], _ROTATE[(i + 5) % len(_ROTATE)], NONFINITE_KINDS[i % 2]]
    plan = []
    for j, kind in enumerate(kinds):
        if (big and j > 0) or (kind in ("tiny", "subnormal") and N > 1024):
            # long windows: one full-length sampling, the other kinds at S <= 512 (subnormal arithmetic is slow in the
            # oracle on the host)
            B, s_list = 3, [1, typ]
        else:
            B, s_list = (1, [1, typ, N, N + 7]) if big else (3, [1, typ, N, N + 7])
        rs = np.random.RandomState(1000 + N + j)
        starts = (N - 1,) if B == 1 else (0, N - 1, int(rs.randint(0, N)))
        plan.append((kind, B, sorted(set(s_list)), starts))
    return plan


def fps_property_f64(xyz, idx, n_steps):
    """at every step the chosen point's float64 distance to the centres so far is >= (1 - 16u) * the largest one"""
    x = xyz.astype(np.float64)
    for b in range(x.shape[0]):
        best = np.full(x.shape[1], np.inf)
        for s in range(min(n_steps, idx.shape[1]) - 1):
            c = x[b, idx[b, s]]
            best = np.minimum(best, ((x[b] - c) ** 2).sum(-1))
            chosen, top = best[idx[b, s + 1]], best.max()
            assert chosen >= (1.0 - 16 * U) * top, (b, s, chosen, top)


@pytest.mark.parametrize("N", FPS_NS)
def test_fps_matches_the_c_oracle_bit_for_bit(N):
    for kind, B, s_list, starts in fps_plan(N):
        xyz = make_xyz(kind, B, N, 7 + N)
        want_full = oracle_fps(kind, B, N, 7 + N, s_list[-1], starts)
        variants = (0, 1, 2, 3) if N > 4096 else (0,)
        for si, S in enumerate(s_list):
            want = want_full[:, :S]
            for li, layout in enumerate(LAYOUTS):
                for variant in variants:
                    if (si + li + variant) % 2 and len(variants) > 1 and S > 512:
                        continue                 # the full-length runs of long windows: each variant in one layout
                    idx, rows, cf = k_fps(xyz, layout, starts, S, variant)
                    where = (kind, S, layout, variant)
                    assert np.array_equal(idx, want), (where, np.argwhere(idx != want)[:3])
                    picked = gather_rows(xyz, want)
                    assert np.array_equal(bits(rows), bits(picked)), where
                    assert np.array_equal(bits(cf), bits(picked.transpose(0, 2, 1))), where
        if s_list[-1] > N and kind not in NONFINITE_KINDS:
            assert (want_full[:, N:] == 0).all(), kind        # all minima 0: the first index, as torch.max
        if kind not in NO_BOUNDS:
            fps_property_f64(xyz, want_full, 600)


def fps_batch_cases(sms):
    """both sides of the cluster kernel's residency threshold, and the cluster kernel where B * CS > SMs"""
    return [(16384, sms // 4, 96, (0, 2, 3)), (16384, sms // 4 + 1, 96, (0, 2, 3)), (8000, sms // 2 + 1, 96, (0, 1, 2, 3))]


def test_fps_batch_sizes_around_the_cluster_residency_threshold():
    sms = sm_count()
    for N, B, S, variants in fps_batch_cases(sms):
        xyz = make_xyz("events", B, N, 31)
        starts = tuple(int(s) for s in synth.make_start_indices(B, N, seed=B))
        want = oracle_fps("events", B, N, 31, S, starts)
        for layout, variant in zip(("rows", "cf", "rows", "cf"), variants):
            idx, rows, cf = k_fps(xyz, layout, starts, S, variant)
            assert np.array_equal(idx, want), (N, B, variant, fps_instance(N, variant, B, sms), np.argwhere(idx != want)[:3])
            picked = gather_rows(xyz, want)
            assert np.array_equal(bits(rows), bits(picked)) and np.array_equal(bits(cf), bits(picked.transpose(0, 2, 1)))


# ================================================================== §3 resumable FPS =================================
RANGE_NS = [33, 100, 250, 500, 1000, 2000, 4000]


@pytest.mark.parametrize("N", RANGE_NS)
def test_fps_in_ranges_equals_one_sampling(N):
    S = 40
    kinds = ("events", "lattice", "nan") if N >= 100 else ("same", "uniform")
    for j, kind in enumerate(kinds):
        B = 3
        xyz = make_xyz(kind, B, N, 50 + N)
        starts = (0, N - 1, int(np.random.RandomState(N).randint(0, N)))
        want = oracle_fps(kind, B, N, 50 + N, S, starts)
        for layout in LAYOUTS:
            one = k_fps(xyz, layout, starts, S)
            assert np.array_equal(one[0], want), (kind, layout)
            for cuts in ([(s, s + 1) for s in range(S)], [(0, 3), (3, 17), (17, 18), (18, 39), (39, 40)], [(0, S)]):
                got = k_fps_ranges(xyz, layout, starts, S, cuts)
                assert np.array_equal(got[0], one[0]), (kind, layout, cuts[:2])
                assert np.array_equal(bits(got[1]), bits(one[1])) and np.array_equal(bits(got[2]), bits(one[2])), (kind, layout)


# ================================================================== §4/§6/§7/§8 ball query ===========================
BQ_NS = [1, 5, 31, 33, 1000, 1023, 1024, 1025, 2049, 4097, 16384]
_RADII = {"events": [0.1, 0.2, 0.4, 0.8], "uniform": [0.1, 0.25, 0.5, 1.0], "offset": [0.1, 0.2, 0.4, 0.8],
          "lattice": [0.25, 0.5, 0.75, 1.0], "signed_zero": [0.25, 0.5, 0.5, 0.75], "clusters": [0.2, 1.0, 150.0, 0.5],
          "line": [0.05, 0.1, 0.3, 0.6], "plane": [0.1, 0.2, 0.4, 0.8], "same": [0.0, 1e-3, 0.2, 0.2],
          "tiny": [0.0, 1e-30, 0.1, 1e-20], "subnormal": [1e-21, 1e-20, 2e-20, 0.1],
          "nan": [0.1, 0.2, 0.4, 0.8], "inf": [0.1, 0.2, 0.4, 0.8]}


def bq_plan(N):
    """(kind, B, S, radii, Ks) per case at N: 1 to 4 radii in any order and with repeats, K <= N"""
    i = BQ_NS.index(N)
    s_cycle = (1, 31, 32, 33, 128, 512)
    k_pool = [k for k in (1, 8, 32, 128) if k <= N] or [1]
    kinds = ["events", _ROTATE[(2 * i) % len(_ROTATE)], _ROTATE[(2 * i + 1) % len(_ROTATE)], NONFINITE_KINDS[i % 2]]
    plan = []
    for j, kind in enumerate(kinds):
        rs = np.random.RandomState(300 + 10 * N + j)
        ns = 1 + (i + j) % 4
        radii = [float(r) for r in rs.choice(_RADII[kind], size=ns, replace=True)]
        if j % 2 == 0:
            eight = [k for k in k_pool if k % 8 == 0] or k_pool
            Ks = [int(k) for k in rs.choice(eight, size=ns)]
        else:
            Ks = [int(k) for k in rs.choice(k_pool, size=ns)]
        S = s_cycle[(i + j) % len(s_cycle)]
        B = 2 if N * S <= 4_000_000 else 1
        plan.append((kind, B, S, radii, Ks))
    return plan


def make_centres(kind, B, N, S, seed):
    """half picked from the window (a NaN / inf point among them where there is one), half anywhere in its box"""
    xyz = make_xyz(kind, B, N, seed)
    rs = np.random.RandomState(seed + S)
    pick = rs.randint(0, N, size=(B, S))
    if kind in NONFINITE_KINDS:
        pos = _nonfinite_positions(N)[0 if kind == "nan" else 1]
        n = min(len(pos), S)
        pick[:, :n] = pos[:n]
    c = gather_rows(xyz, pick).astype(np.float32)
    fin = np.where(np.isfinite(xyz), xyz, 0.0)
    lo, hi = fin.min(axis=1, keepdims=True), fin.max(axis=1, keepdims=True)
    free = (lo + (hi - lo) * rs.rand(B, S, 3)).astype(np.float32)
    half = np.arange(S) >= (S + 1) // 2
    c[:, half] = free[:, half]
    if kind == "inf":                           # centres of both signs on the axis of every +inf coordinate
        n = min(len(_nonfinite_positions(N)[1]), S)
        if n + 2 <= (S + 1) // 2:               # after the non-finite centres, before the free half
            c[:, n] = [0.0, 0.0, 0.0]
            c[:, n + 1] = [-0.5, -0.5, -0.5]
    return np.ascontiguousarray(c, np.float32)


def make_records(xyz, seed):
    """[B,N,8] records as the model builds them for sa1: [x, y, z, two extra channels | x, y, z]"""
    B, N, _ = xyz.shape
    rec = np.empty((B, N, 8), np.float32)
    rec[..., 0:3] = xyz
    rec[..., 3:5] = np.random.RandomState(seed).randint(0, 2, size=(B, N, 2))
    rec[..., 5:8] = xyz
    return rec


def check_index_range(lists, N, K):
    """every entry < N and >= 0, except an all-N list (the sentinel of an empty ball)"""
    lists = lists.reshape(-1, K)
    empty = (lists == N).all(-1)
    ok = (lists >= 0) & (lists < N)
    assert ok[~empty].all(), lists[~empty][~ok[~empty].all(-1)][:2]


def per_group(rm, bg, total):
    rm, bg = rm[:total], bg[:total // 8]
    d = {}
    for blk, g in enumerate(bg):
        d.setdefault(int(g), []).extend(rm[8 * blk:8 * blk + 8].tolist())
    return d


def numpy_rows(lists, cnt, B, N, S, K):
    """the compaction's row rule: per group its first max(cnt, 1) entries rounded up to 8 rows with copies of the first,
    global rows b * N + point, -1 everywhere for an empty ball"""
    want = {}
    for g in range(B * S):
        b, s = divmod(g, S)
        c = int(cnt[b, s])
        rows = (max(c, 1) + 7) // 8 * 8
        if c == 0:
            want[g] = [-1] * rows
        else:
            want[g] = [b * N + int(lists[b, s, k if k < c else 0]) for k in range(rows)]
    return want


def ball_property_f64(xyz, centres, r, lists, N, K):
    """each decision the list shows agrees with |q - p|^2 <= fp32(r^2) in float64 outside the first-order band of the
    expanded expression (the exact fp32 decisions inside it are pinned bitwise against the oracle)"""
    r2 = float(np.float32(float(r) ** 2))
    x, q = xyz.astype(np.float64), centres.astype(np.float64)
    for b in range(x.shape[0]):
        d64 = ((q[b][:, None, :] - x[b][None, :, :]) ** 2).sum(-1)
        scale = 2 * (np.abs(q[b]) @ np.abs(x[b]).T) + (q[b] ** 2).sum(-1)[:, None] + (x[b] ** 2).sum(-1)[None, :]
        band = np.abs(d64 - r2) <= 6 * U * scale
        for s in range(q.shape[1]):
            lst = lists[b, s]
            c = real_count(lst, N)
            limit = int(lst[c - 1]) if c == K else N - 1          # beyond the K-th hit the list says nothing
            inc = np.zeros(N, bool)
            inc[lst[:c]] = True
            pred = d64[s] <= r2
            bad = (inc != pred) & ~band[s]
            bad[limit + 1:] = False
            assert not bad.any(), (b, s, np.flatnonzero(bad)[:3], d64[s][bad][:3], r2)


# torch's matmul may round the K = 3 product of pairwise_sqdist differently from the C oracle's FMA chain at some shapes
# (the heads envelope met one in three_nn at S = 3, N = 5).  A ball-query disagreement between the two oracles must come
# from such a distance on the other side of r^2, and must be listed here (case, N, S, r, window, centre) and in DESIGN §2.
# None is known: every case of this file agrees.
KNOWN_TORCH_BQ_DISAGREEMENTS = set()


def torch_oracle_ball(label, xyz, centres, r, K, want):
    N = xyz.shape[1]
    got = sa_oracle.ball_query(r, K, torch.from_numpy(xyz), torch.from_numpy(centres)).numpy()
    if np.array_equal(got, want):
        return
    d_t = sa_oracle.pairwise_sqdist(torch.from_numpy(centres), torch.from_numpy(xyz)).numpy()
    d_c = c_oracle.sqdist(centres, xyz)
    r2 = np.float32(float(r) ** 2)
    for b, s in sorted({(int(b), int(s)) for b, s, _ in np.argwhere(got != want)}):
        flip = (~(d_t[b, s] > r2)) != (~(d_c[b, s] > r2))
        assert flip.any(), (label, N, b, s, "torch and C oracle lists differ without a distance across r^2")
        keep = ~flip                               # outside the flipped points both oracles list the same hits
        hits_t = [i for i in range(N) if keep[i] and not d_t[b, s, i] > r2]
        hits_c = [i for i in range(N) if keep[i] and not d_c[b, s, i] > r2]
        assert hits_t == hits_c
        key = (label, N, centres.shape[1], r, b, s)
        assert key in KNOWN_TORCH_BQ_DISAGREEMENTS, ("torch.matmul puts %d distance(s) across r^2: list the case" % flip.sum(), key)


@pytest.mark.parametrize("N", BQ_NS)
def test_ball_query_matches_the_c_oracle_bit_for_bit(N):
    for j, (kind, B, S, radii, Ks) in enumerate(bq_plan(N)):
        seed = 11 + N + j
        xyz = make_xyz(kind, B, N, seed)
        centres = make_centres(kind, B, N, S, seed)
        ckey = (kind, B, N, seed, S)
        _CENTRES[ckey] = centres
        flags = first_occurrence_np(make_records(xyz, seed))
        wants = [oracle_ball(kind, B, N, seed, ckey, r, K) for r, K in zip(radii, Ks)]
        got = check_ball_case(kind, xyz, centres, radii, Ks, LAYOUTS[j % 2], flags, wants, kind not in NO_BOUNDS)
        if kind in NONFINITE_KINDS and N > 1:
            nonfinite_rules(kind, xyz, centres, radii, Ks, got["idx"], N)
    if N <= 2048:
        for kind, B, S, radii, Ks in bq_plan(N):            # the torch oracle's FPS agrees exactly (no matmul in it)
            xyz = make_xyz(kind, B, N, 5)
            start = np.random.RandomState(N).randint(0, N, size=B)
            got = sa_oracle.fps(torch.from_numpy(xyz), min(N + 7, 300), torch.from_numpy(start)).numpy()
            assert np.array_equal(got, c_oracle.fps(xyz, min(N + 7, 300), start)), (kind, N)


def check_ball_case(label, xyz, centres, radii, Ks, layout, flags, wants, bounds):
    """every ball-query entry on one input against the oracle's lists `wants` (one per scale) -> the kernels' outputs"""
    B, N, _ = xyz.shape
    S = centres.shape[1]
    got = k_ball_all(xyz, layout, centres, radii, Ks, flags)
    where = (label, B, N, S, radii, Ks, layout)
    for name in ("plain", "idx", "uidx"):
        assert got[name].shape == (B, S, sum(Ks))
    off = 0
    for i, (r, K, want) in enumerate(zip(radii, Ks, wants)):
        for name in ("plain", "idx", "uidx"):
            blk = got[name][:, :, off:off + K]
            assert np.array_equal(blk, want), (where, name, r, np.argwhere(blk != want)[:3])
            check_index_range(blk, N, K)
        cnt = np.array([[real_count(want[b, s], N) for s in range(S)] for b in range(B)])
        assert np.array_equal(got["cnt"][i], cnt), (where, r)
        # the deduplicated list: the hits that are first occurrences, in index order
        for b in range(B):
            for s in range(S):
                hits = [int(h) for h in want[b, s, :cnt[b, s]] if flags[b, h]]
                assert got["ucnt"][i, b, s] == len(hits), (where, r, b, s)
                assert got["uniq"][b, s, off:off + len(hits)].tolist() == hits, (where, r, b, s)
        if bounds:
            ball_property_f64(xyz, centres, r, want, N, K)
        if N <= 2048:
            torch_oracle_ball(label, xyz, centres, r, K, want)
        off += K
    if "compact" in got:
        ucnt = got["ucnt"]
        cnt_all = np.stack([[[real_count(w[b, s], N) for s in range(S)] for b in range(B)] for w in wants])
        ulists = got["uniq"]
        for name, lists, counts in (("compact", np.concatenate(wants, -1), cnt_all), ("compact_dedup", ulists, ucnt)):
            i3, rm, bg, nr = got[name]
            assert np.array_equal(i3, np.concatenate(wants, -1)), (where, name)
            rm2, bg2, nr2 = k_group_compact(lists, counts, N, Ks)
            assert np.array_equal(nr, nr2), (where, name)
            off = 0
            for i, K in enumerate(Ks):
                total = int(nr[i])
                assert total % 8 == 0
                mine = per_group(rm[i], bg[i], total)
                assert mine == per_group(rm2[i], bg2[i], total), (where, name, i)
                assert mine == numpy_rows(lists[:, :, off:off + K], counts[i], B, N, S, K), (where, name, i)
                assert sum(len(v) for v in mine.values()) == total
                flat = rm[i][:total]
                assert ((flat >= 0) & (flat < B * N) | (flat == -1)).all()
                off += K
    return got


@pytest.mark.parametrize("N", [33, 1025, 2051])
def test_ball_query_padding_is_never_a_hit_for_an_infinite_centre(N):
    """the last word of a window whose tile is not a multiple of 32 points holds padding at 1e18; for a centre with a
    +inf coordinate its expanded distance is -inf + inf = NaN, which the inclusive rule would count as a hit.  Fewer real
    hits than K, so the list reaches past the last real point."""
    B = 1
    rs = np.random.RandomState(N)
    xyz = rs.uniform(-1.0, -0.1, size=(B, N, 3)).astype(np.float32)         # x < 0: no hit for a +inf-x centre
    few = rs.choice(N, 6, replace=False)
    xyz[0, few, 0] = rs.uniform(0.0, 1.0, 6).astype(np.float32)               # x >= 0: NaN distance, a hit
    p = int(few[0])
    xyz[0, p, 0] = np.inf
    centres = np.stack([xyz[:, p], xyz[:, N // 2], np.full((B, 3), np.inf, np.float32)], 1).astype(np.float32)
    radii, Ks = [0.3, 0.6], [32, 8]
    wants = [c_oracle.ball_query(r, K, xyz, centres) for r, K in zip(radii, Ks)]
    assert real_count(wants[0][0, 0], N) < 32 and real_count(wants[0][0, 2], N) < 32
    flags = first_occurrence_np(make_records(xyz, N))
    for layout in LAYOUTS:
        got = check_ball_case("inf_centre", xyz, centres, radii, Ks, layout, flags, wants, False)
        nonfinite_rules("inf", xyz, centres[:, :2], radii, Ks, got["idx"][:, :2], N)


def nonfinite_rules(kind, xyz, centres, radii, Ks, idx, N):
    """the reference's sqrdists > r**2 is False for NaN: NaN points are in every ball, NaN centres take every point;
    p with a +inf coordinate gives -2 q.p + |p|^2 = NaN (a hit) where that centre coordinate is >= 0, +inf (no hit) below"""
    B, S, _ = centres.shape
    off = 0
    for r, K in zip(radii, Ks):
        blk = idx[:, :, off:off + K]
        for b in range(B):
            for s in range(S):
                q = centres[b, s]
                lst = blk[b, s]
                c = real_count(lst, N)
                last = int(lst[c - 1]) if c else -1
                room = c < K
                if np.isnan(q).any():
                    assert lst.tolist() == list(range(K)), (b, s)
                    continue
                if not np.isfinite(q).all():
                    continue                     # a centre on an infinite point: checked against the oracle only
                for p in np.flatnonzero(~np.isfinite(xyz[b]).all(-1)):
                    pt = xyz[b, p]
                    if np.isnan(pt).any():
                        hit = True
                    else:
                        ax = int(np.flatnonzero(np.isinf(pt))[0])
                        hit = not (q[ax] < 0)
                    if hit and (room or p <= last):
                        assert p in lst[:c], (kind, b, s, p, q)
                    if not hit:
                        assert p not in lst[:c], (kind, b, s, p, q)
        off += K


def test_ball_query_nonfinite_points_and_centres():
    """a hand-built window: NaN point, +inf points on each axis, a NaN centre, centres of both signs and exact zeros"""
    B, N = 1, 64
    xyz = make_xyz("uniform", B, N, 3).copy()
    xyz[0, 5] = [np.nan, 0.1, 0.1]
    xyz[0, 9, 0] = np.inf
    xyz[0, 20, 1] = np.inf
    xyz[0, 40, 2] = np.inf
    centres = np.array([[[np.nan, 0, 0], [0.2, 0.3, 0.4], [-0.2, -0.3, -0.4], [0.0, -0.0, 0.0], [-0.0, 0.5, -0.5],
                         [0.5, -0.5, 0.5]]], np.float32)
    for layout in LAYOUTS:
        x, st = to_device(xyz, layout)
        got = _capi.ball_query(x, st, torch.from_numpy(centres).to(DEV), N, [0.3, 5.0], [N, 16]).cpu().numpy()
        off = 0
        for r, K in ((0.3, N), (5.0, 16)):
            want = c_oracle.ball_query(r, K, xyz, centres)
            assert np.array_equal(got[:, :, off:off + K], want), (layout, r)
            check_index_range(want, N, K)
            off += K
        full = got[0, :, :N]                  # K = N: the whole membership
        assert full[0].tolist() == list(range(N))                                  # NaN centre: every point
        for s in range(1, 6):
            mem = set(full[s].tolist())
            assert 5 in mem                                                          # NaN point: every ball
            for p, ax in ((9, 0), (20, 1), (40, 2)):
                assert (p in mem) == (not centres[0, s, ax] < 0), (s, p)


# ================================================================== §5 the radius boundary ===========================
BOUNDARY_RADII = [0.1, 0.2, 0.3, 1.0 / 3.0, 0.4, 0.8]


@functools.lru_cache(maxsize=None)
def boundary_points(r):
    """points whose oracle distance to their centre is exactly fp32(r^2) ('on'), the next float above ('above') or
    below ('below'): start from c + r v, |v| = 1, and nudge the coordinates by ulps until sqdist lands there"""
    r2 = np.float32(float(r) ** 2)
    targets = {"on": r2, "above": np.nextafter(r2, np.float32(np.inf)), "below": np.nextafter(r2, np.float32(0))}
    rs = np.random.RandomState(int(r * 1000))
    centres = np.array([[0.0, 0.0, 0.0], [0.25 * r, -0.125 * r, 0.0625 * r], [-0.0625 * r, 0.125 * r, -0.25 * r]], np.float32)
    pts = {k: [] for k in targets}
    owner = {k: [] for k in targets}

    def nudged(v, n):            # v and its n neighbours on either side, one ulp apart
        lo, hi = [v], [v]
        for _ in range(n):
            lo.append(np.nextafter(lo[-1], np.float32(-np.inf)))
            hi.append(np.nextafter(hi[-1], np.float32(np.inf)))
        return np.array(lo[:0:-1] + hi, np.float32)

    for ci, c in enumerate(centres):
        for _ in range(24):
            v = rs.normal(size=3)
            p0 = (c.astype(np.float64) + r * v / np.linalg.norm(v)).astype(np.float32)
            # every combination of +-6 ulps on the three coordinates
            cand = np.stack(np.meshgrid(*[nudged(p0[a], 6) for a in range(3)], indexing="ij"), -1).reshape(-1, 3)
            d = c_oracle.sqdist(c[None, None, :], cand[None])[0, 0]
            for kname, t in targets.items():
                hit = np.flatnonzero(d == t)[:2]
                pts[kname].extend(cand[hit])
                owner[kname].extend([ci] * len(hit))
    return centres, {k: np.array(v, np.float32).reshape(-1, 3) for k, v in pts.items()}, {k: np.array(v) for k, v in owner.items()}


@pytest.mark.parametrize("r", BOUNDARY_RADII, ids=lambda r: "r%.4g" % r)
def test_ball_query_radius_boundary_is_inclusive_in_fp32(r):
    centres, pts, owner = boundary_points(r)
    for k in ("on", "above", "below"):
        assert len(pts[k]) >= 32, (k, len(pts[k]))                   # the construction must not thin out
    r2 = np.float32(float(r) ** 2)
    allp = np.concatenate([pts["on"], pts["above"], pts["below"]])
    kind = np.array(["on"] * len(pts["on"]) + ["above"] * len(pts["above"]) + ["below"] * len(pts["below"]))
    own = np.concatenate([owner["on"], owner["above"], owner["below"]])
    perm = np.random.RandomState(1).permutation(len(allp))
    xyz, kind, own = allp[perm][None].copy(), kind[perm], own[perm]
    N = xyz.shape[1]
    C = centres[None].copy()
    d_or = c_oracle.sqdist(C, xyz)[0]
    d_k = k_sqdist(C, xyz)[0]
    assert np.array_equal(bits(d_k), bits(d_or))                      # the kernel's distances, bitwise
    for ci in range(3):
        mine = own == ci
        assert (d_or[ci][mine & (kind == "on")] == r2).all()
        assert (d_or[ci][mine & (kind == "above")] == np.nextafter(r2, np.float32(np.inf))).all()
        assert (d_or[ci][mine & (kind == "below")] == np.nextafter(r2, np.float32(0))).all()
    for layout in LAYOUTS:
        x, st = to_device(xyz, layout)
        got = _capi.ball_query(x, st, torch.from_numpy(C).to(DEV), N, [r], [N]).cpu().numpy()[0]
        assert np.array_equal(got[None], c_oracle.ball_query(r, N, xyz, C)), layout
        for ci in range(3):
            mem = set(got[ci].tolist())
            mine = own == ci
            for p in np.flatnonzero(mine & (kind != "above")):
                assert p in mem, (layout, ci, p, kind[p])                # on fp32(r^2) and below: inside
            for p in np.flatnonzero(mine & (kind == "above")):
                assert p not in mem, (layout, ci, p)                     # one ulp above: outside


# ================================================================== §9 compaction by range ==========================
@pytest.mark.parametrize("N,S,ranges", [(2049, 200, [(0, 64), (64, 32), (96, 96), (192, 8)]),
                                        (1000, 33, [(0, 32), (32, 1)]),
                                        (16384, 512, [(0, 160), (160, 320), (480, 32)])])
def test_compaction_by_range_equals_the_one_shot_tables(N, S, ranges):
    B = 2
    Ks, radii = [16, 64, 128, 8], [0.2, 0.4, 0.8, 0.1]
    for kind in ("events", "lattice"):
        seed = 90 + N
        xyz = make_xyz(kind, B, N, seed)
        centres = make_centres(kind, B, N, S, seed)
        fl = k_first(make_records(xyz, seed))
        for flags in (None, fl):
            x, st = to_device(xyz, "cf", seed=N + 2)
            c = torch.from_numpy(centres).to(DEV)
            f = None if flags is None else torch.from_numpy(flags).to(DEV)
            i1, rm1, bg1, nr1 = _capi.ball_query_compact(x, st, c, N, radii, Ks, f)
            i1, nr1 = i1.cpu().numpy(), nr1.cpu().numpy()
            rm1, bg1 = [t.cpu().numpy() for t in rm1], [t.cpu().numpy() for t in bg1]
            idx, uniq, rm, bg, nr = k_compact_range(xyz, "cf", centres, radii, Ks, flags, ranges)
            assert np.array_equal(idx, i1), (kind, flags is None)
            assert np.array_equal(nr, nr1), (kind, flags is None, nr, nr1)
            if flags is not None:
                _, u1, uc1 = _capi.ball_query_uniq(x, st, c, N, radii, Ks, f)
                u1, uc1 = u1.cpu().numpy(), uc1.cpu().numpy()
                off = 0
                for i, K in enumerate(Ks):
                    for b in range(B):
                        for s in range(S):
                            n = int(uc1[i, b, s])
                            assert np.array_equal(uniq[b, s, off:off + n], u1[b, s, off:off + n]), (kind, i, b, s)
                    off += K
            for i in range(len(Ks)):
                total = int(nr1[i])
                assert per_group(rm[i], bg[i], total) == per_group(rm1[i], bg1[i], total), (kind, i)


# ================================================================== §10 duplicate flags ==============================
DUP_NS = [1, 31, 4096, 4097, 8192, 8193, 16384]


def dup_inputs(N, seed):
    rs = np.random.RandomState(seed)
    yield "distinct", rs.rand(1, N, 8).astype(np.float32)
    yield "identical", np.broadcast_to(rs.rand(1, 1, 8).astype(np.float32), (1, N, 8)).copy()
    base = rs.rand(N // 3 + 1, 8).astype(np.float32)
    yield "two_thirds_copies", base[rs.randint(0, len(base), size=N)][None].copy()
    # pairs that differ in exactly one of the eight words (words 5-7 lie outside the hash of words 0-4)
    base = rs.rand((N + 1) // 2, 8).astype(np.float32)
    rec = np.repeat(base, 2, axis=0)[:N].copy()
    for j in range(1, N, 2):
        w = (j // 2) % 8
        rec[j, w] = np.nextafter(rec[j, w], np.float32(2.0))
    yield "one_word_apart", rec[None].copy()
    # pairs that differ only in the sign bit of one word: multiplying by an odd constant moves that bit to bit 31 alone,
    # which the slot mask drops, so both records always probe one chain and the full comparison must tell them apart
    base = rs.rand(N // 4 + 1, 8).astype(np.float32)
    rec = base[rs.randint(0, len(base), size=N)]
    flip = rs.randint(0, 8, size=N)
    neg = rs.rand(N) < 0.5
    rec[np.arange(N)[neg], flip[neg]] *= -1
    yield "one_sign_apart", rec[None].copy()
    # the same hashed words 0-4 everywhere, different xyz in words 5-7 (a record with D = 5 features), plus copies
    rec = np.broadcast_to(rs.rand(1, 8).astype(np.float32), (N, 8)).copy()
    rec[:, 5:8] = rs.randint(0, 64, size=(N, 3)) / np.float32(64)
    yield "hash_words_equal", rec[None].copy()
    # +0.0 and -0.0 are different records (the comparison is bitwise); NaN with one payload repeats, other payloads not
    rec = np.zeros((N, 8), np.float32)
    rec[:, 0] = np.where(rs.rand(N) < 0.5, np.float32(0.0), np.float32(-0.0))
    rec[:, 6] = np.where(rs.rand(N) < 0.5, np.float32(0.0), np.float32(-0.0))
    payload = (np.uint32(0x7fc00000) | rs.randint(0, 3, size=N).astype(np.uint32)).view(np.float32)
    rec[:, 3] = np.where(rs.rand(N) < 0.5, payload, np.float32(1.0))
    rec[:, 7] = np.where(rs.rand(N) < 0.3, np.uint32(0xffc00001).view(np.float32), np.float32(0.0))
    yield "signed_zero_nan_payloads", rec[None].copy()


@pytest.mark.parametrize("N", DUP_NS)
def test_duplicate_flags_match_a_bytes_based_first_occurrence(N):
    for name, pts8 in dup_inputs(N, 600 + N):
        want = first_occurrence_np(pts8)
        got = k_first(pts8)
        assert np.array_equal(got, want), (name, uniq_slots(N), np.flatnonzero(got[0] != want[0])[:4])
        if name == "signed_zero_nan_payloads" and N > 31:
            assert 2 < want.sum() < N
    # two windows of different contents in one launch
    a = next(dup_inputs(N, 1))[1]
    b2 = np.concatenate([a, a[:, ::-1]], 0)
    assert np.array_equal(k_first(b2), first_occurrence_np(b2))


def test_duplicate_flags_refuse_misaligned_records():
    buf = torch.zeros(2 * 64 * 8 + 1, device=DEV)
    view = buf[1:].view(2, 64, 8)                                    # 4 bytes past a 16-byte boundary
    with pytest.raises(RuntimeError, match="misaligned"):
        _capi.first_occurrence(view)
    assert torch.equal(_capi.first_occurrence(buf[:-1].view(2, 64, 8)), torch.tensor([[1] + [0] * 63] * 2, dtype=torch.uint8, device=DEV))


def test_duplicate_flags_time_when_all_hashed_words_are_equal():
    """16384 records whose hashed words agree: with a hash of fewer words than the record, every record probes one chain"""
    rec = dict(dup_inputs(16384, 5))["hash_words_equal"]
    x = torch.from_numpy(rec).to(DEV)
    _capi.first_occurrence(x)
    times = []
    for _ in range(5):                          # the least of five launches: a busy neighbour only adds time
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        got = _capi.first_occurrence(x)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b))
    ms = min(times)
    print("first_occurrence, N = 16384, hashed words equal: %.4f ms (%s)" % (ms, torch.cuda.get_device_name(0)))
    assert np.array_equal(got.cpu().numpy(), first_occurrence_np(rec))
    assert ms < 1.0, ms


# ================================================================== coverage =========================================
def test_every_kernel_instance_is_reached():
    """the instances the cases above launch, derived from the dispatch thresholds, cover every instance there is"""
    sms = sm_count()
    fps = set()
    for N in FPS_NS:
        for kind, B, s_list, starts in fps_plan(N):
            for v in ((0, 1, 2, 3) if N > 4096 else (0,)):
                fps.add(fps_instance(N, v, B, sms))
    for N, B, S, variants in fps_batch_cases(sms):
        fps.update(fps_instance(N, v, B, sms) for v in variants)
    assert fps == {"fps<32,4,4>", "fps<64,4,4>", "fps<128,4,4>", "fps<256,4,4>", "fps<256,8,8>", "fps<512,8,8>",
                   "fps<1024,8,8>", "fps<1024,16,6>", "cluster<2>", "cluster<4>", "pruned<16>", "pruned<32>"}, fps
    # the automatic choice on both sides of the residency line
    assert fps_instance(16384, 0, sms // 4, sms) == "cluster<4>" and fps_instance(16384, 0, sms // 4 + 1, sms) == "pruned<32>"
    assert {fps_range_instance(N) for N in RANGE_NS} == {"range<32,4,4>", "range<64,4,4>", "range<128,4,4>",
                                                         "range<256,4,4>", "range<256,8,8>", "range<512,8,8>"}
    scales = {len(radii) for N in BQ_NS for _, _, _, radii, _ in bq_plan(N)}
    assert scales == {1, 2, 3, 4}, scales                            # ball_query_kernel<1..4>
    assert any(all(k % 8 == 0 for k in Ks) and len(Ks) == 4 for N in BQ_NS for *_, Ks in bq_plan(N))
    assert {uniq_slots(N) for N in DUP_NS} == {8192, 16384, 32768}
    # entries: ev2h_ball_query_f32, _cnt_f32, _uniq_f32, _compact_f32 (k_ball_all) and _compact_range_f32 (k_compact_range)
    ks = {k for N in BQ_NS for *_, Ks in bq_plan(N) for k in Ks}
    ss = {S for N in BQ_NS for _, _, S, _, _ in bq_plan(N)}
    assert ks == {1, 8, 32, 128} and ss == {1, 31, 32, 33, 128, 512}, (ks, ss)
