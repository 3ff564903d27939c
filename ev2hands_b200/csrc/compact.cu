// Row compaction for the fused set-abstraction kernel.
//
// query_ball_point pads every group to K neighbours by repeating the first one (reference
// src/Ev2Hands/model/pointnet2_utils.py:104-106), and the shared MLP then evaluates those copies again
// (:253-257) although max-pooling cannot see them: max over {a, a, ..., b, c} = max over {a, b, c}.  On event
// windows most groups are far from full (17 % .. 89 % real neighbours per scale on the benchmark's data), so
// the fused kernel runs over a COMPACTED row list instead: per group its real neighbours, rounded up to a
// multiple of 8 rows with copies of the first one (8 rows = one UMMA core-matrix row block = the granularity
// of the pooled epilogue), groups back to back.  Results are bit-identical to the dense evaluation.
//
//   rowmap[r]        global point row (b*N + point) feeding compact row r, -1 for "no point" (empty ball)
//   blockgroup[r/8]  global group (b*S + centre) the 8-row block belongs to (defined for r < n_rows)
//   n_rows           total compact rows of the scale
#include "common.cuh"

namespace ev2h {

__device__ __forceinline__ int compact_rows(int cnt, int K) {
    cnt = cnt < 1 ? 1 : (cnt > K ? K : cnt);
    return (cnt + 7) & ~7;
}

struct CompactScales {
    int K[4], k_off[4];
    int32_t *rowmap[4];
    int32_t *blockgroup[4];
};

// lpg lanes per (group, scale) - 8, 16 or 32 for K <= 32, 64, 128.  A CTA reserves the rows of its groups with one
// atomic add on the scale's row counter, then every group writes its compact rows and block -> group entries.
// CTAs therefore land in the list in no particular order, which nothing depends on: every group's rows are contiguous, the block table says
// whose they are, and the pooled maximum does not care in which tile a group is evaluated.
__global__ void __launch_bounds__(256)
compact_fill_kernel(const int32_t *__restrict__ idx, int idx_ld, const int32_t *__restrict__ cnt, int G,
                    int N, int S, int32_t *__restrict__ n_rows, CompactScales prm) {
    const int sc = blockIdx.y;
    const int K = prm.K[sc];
    const int lpg = K <= 32 ? 8 : (K <= 64 ? 16 : 32);
    const int t = blockIdx.x * 256 + threadIdx.x;
    const int g = t / lpg, lane = t % lpg;
    const bool live = g < G;
    int c = 0, rows = 0;
    if (live) {
        c = cnt[(int64_t)sc * G + g];
        rows = compact_rows(c, K);
    }
    // one atomic add per CTA: block-wide exclusive scan of the group leaders' row counts
    __shared__ int warp_tot[8];
    __shared__ int cta_base;
    const int wl = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int mine = (live && lane == 0) ? rows : 0;
    int incl = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (wl >= d) incl += v;
    }
    if (wl == 31) warp_tot[wid] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        int tot = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w) { const int v = warp_tot[w]; warp_tot[w] = tot; tot += v; }
        cta_base = tot ? atomicAdd(n_rows + sc, tot) : 0;
    }
    __syncthreads();
    int off = cta_base + warp_tot[wid] + incl - mine;            // valid in the leader lane
    // the group's lanes are lpg consecutive lanes of one warp (lpg divides 32): broadcast the leader's offset
    off = __shfl_sync(0xffffffffu, off, wl & ~(lpg - 1));
    if (!live) return;
    const int real = c < 1 ? 1 : (c > K ? K : c);
    const int32_t *src = idx + (int64_t)g * idx_ld + prm.k_off[sc];
    const int64_t b = g / S;
    int32_t *rm = prm.rowmap[sc], *bg = prm.blockgroup[sc];
    for (int k = lane; k < rows; k += lpg) {
        const int pt = c < 1 ? -1 : src[k < real ? k : 0];             // c == 0: empty ball, the list holds nothing
        rm[off + k] = (pt >= 0 && pt < N) ? (int32_t)(b * N + pt) : -1;
        if ((k & 7) == 0) bg[(off + k) >> 3] = g;
    }
}

}  // namespace ev2h

extern "C" int ev2h_group_compact_i32(const int32_t *idx, int idx_ld, const int32_t *cnt, int B, int N, int S, int n_scales,
                                      const int32_t *nsample_host,
                                      int32_t *const *rowmap_host, int32_t *const *blockgroup_host, int32_t *n_rows_dev,
                                      ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(idx && cnt && nsample_host && rowmap_host && blockgroup_host && n_rows_dev,
                 "ev2h_group_compact_i32: null argument");
    EV2H_REQUIRE(B > 0 && N > 0 && S > 0 && n_scales >= 1 && n_scales <= 4, "ev2h_group_compact_i32: bad sizes");
    const int64_t G64 = (int64_t)B * S;
    EV2H_REQUIRE(G64 * 128 < 2147483647LL, "ev2h_group_compact_i32: too many groups for 32-bit row offsets");
    const int G = (int)G64;
    CompactScales prm;
    int off = 0;
    for (int i = 0; i < 4; ++i) {
        const bool on = i < n_scales;
        prm.K[i] = on ? nsample_host[i] : 0;
        prm.k_off[i] = off;
        prm.rowmap[i] = on ? rowmap_host[i] : nullptr;
        prm.blockgroup[i] = on ? blockgroup_host[i] : nullptr;
        if (on) {
            EV2H_REQUIRE(nsample_host[i] > 0 && nsample_host[i] % 8 == 0 && prm.rowmap[i] && prm.blockgroup[i],
                         "ev2h_group_compact_i32: scale %d: K must be a positive multiple of 8 and buffers non-null", i);
            off += nsample_host[i];
        }
    }
    EV2H_REQUIRE(off <= idx_ld, "ev2h_group_compact_i32: idx_ld smaller than the sum of K");
    cudaStream_t st = as_stream(stream);
    cudaError_t e = cudaMemsetAsync(n_rows_dev, 0, sizeof(int32_t) * n_scales, st);
    if (e != cudaSuccess) return fail(EV2H_ERR_CUDA, "ev2h_group_compact_i32: memset: %s", cudaGetErrorString(e));
    // sized for 32 lanes per group; scales with fewer lanes per group leave the tail of their grid row idle
    compact_fill_kernel<<<dim3((unsigned)((G + 7) / 8), (unsigned)n_scales), 256, 0, st>>>(idx, idx_ld, cnt, G, N, S, n_rows_dev, prm);
    return check_launch("ev2h_group_compact_i32");
}

// ---- exact-duplicate points ------------------------------------------------------------------------------
// Event windows are drawn WITH replacement from the per-pixel aggregates (reference dataset code, SURVEY.md 8d:
// ~40 % of a window's 2048 points are exact copies of an earlier point).  Two neighbours with identical records
// give identical MLP rows, which the max-pool cannot tell apart, so the compacted row list keeps only the first
// occurrence.  first[b,n] = 1 iff no point m < n of window b has the same 32-byte record.
namespace ev2h {

constexpr int kUniqSlots = 8192;          // open-addressing table per window, >= 2 x the points hashed at once (windows up to 4096 points;
                                          // longer ones take a table of the next power of two >= 2 N, up to 32768 slots = 128 KB)
constexpr int kUniqThreads = 1024;

__device__ __forceinline__ bool same_record(const uint4 *rec, int a, int b) {
    const uint4 a0 = rec[2 * a], a1 = rec[2 * a + 1], b0 = rec[2 * b], b1 = rec[2 * b + 1];
    return a0.x == b0.x && a0.y == b0.y && a0.z == b0.z && a0.w == b0.w && a1.x == b1.x && a1.y == b1.y && a1.z == b1.z && a1.w == b1.w;
}

__global__ void __launch_bounds__(kUniqThreads)
first_occurrence_kernel(const float *__restrict__ pts8, int N, uint8_t *__restrict__ first, int slots) {
    extern __shared__ int table[];            // [slots], a power of two
    const uint4 *rec = reinterpret_cast<const uint4 *>(pts8 + (int64_t)blockIdx.x * N * 8);
    uint8_t *out = first + (int64_t)blockIdx.x * N;
    for (int i = threadIdx.x; i < slots; i += kUniqThreads) table[i] = 0x7fffffff;
    __syncthreads();
    // the hash covers all eight words: records of few features keep xyz in words 4..7, and records that differ only in
    // unhashed words would all probe one chain (16384 such records: 258 ms with words 0..4 hashed, 0.14 ms with all
    // eight, on a B200)
    auto slot_of = [&](int n) {
        const uint4 a = rec[2 * n], b = rec[2 * n + 1];
        uint32_t h = a.x * 0x9E3779B1u ^ a.y * 0x85EBCA77u ^ a.z * 0xC2B2AE3Du ^ a.w * 0x27D4EB2Fu ^ b.x * 0x165667B1u ^
                     b.y * 0xD3A2646Du ^ b.z * 0xFD7046C5u ^ b.w * 0xB55A4F09u;
        h ^= h >> 15;
        return (int)(h & (slots - 1));
    };
    // phase 1: every record ends up in exactly one slot holding the smallest index that carries it
    for (int n = threadIdx.x; n < N; n += kUniqThreads) {
        int h = slot_of(n);
        for (;;) {
            const int cur = atomicCAS(&table[h], 0x7fffffff, n);
            if (cur == 0x7fffffff) break;                                 // claimed an empty slot
            if (same_record(rec, cur, n)) { atomicMin(&table[h], n); break; }
            h = (h + 1) & (slots - 1);
        }
    }
    __syncthreads();
    // phase 2: look the record up again; the slot now holds its first occurrence
    for (int n = threadIdx.x; n < N; n += kUniqThreads) {
        int h = slot_of(n);
        for (;;) {
            const int cur = table[h];
            if (same_record(rec, cur, n)) { out[n] = cur == n ? 1 : 0; break; }
            h = (h + 1) & (slots - 1);
        }
    }
}

}  // namespace ev2h

extern "C" int ev2h_first_occurrence_u8(const float *pts8, int B, int N, uint8_t *first, ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(pts8 && first, "ev2h_first_occurrence_u8: null argument");
    EV2H_REQUIRE(B > 0 && N > 0 && ((uintptr_t)pts8 & 15) == 0, "ev2h_first_occurrence_u8: bad sizes or misaligned records");
    if (N > 16384) return fail(EV2H_ERR_UNSUPPORTED, "ev2h_first_occurrence_u8: N=%d exceeds 16384 points per window", N);
    int slots = kUniqSlots;
    while (slots < 2 * N) slots *= 2;
    const size_t smem = (size_t)slots * sizeof(int);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(first_occurrence_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return fail(EV2H_ERR_CUDA, "ev2h_first_occurrence_u8: smem attribute: %s", cudaGetErrorString(e));
    }
    first_occurrence_kernel<<<(unsigned)B, kUniqThreads, smem, as_stream(stream)>>>(pts8, N, first, slots);
    return check_launch("ev2h_first_occurrence_u8");
}
