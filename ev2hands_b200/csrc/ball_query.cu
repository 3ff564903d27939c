// Multi-radius ball query: all radii of a layer in one scan over the window's points,
// 32 centres x 8 point ranges per CTA.
//
// Replaces query_ball_point + square_distance (reference
// src/Ev2Hands/model/pointnet2_utils.py:87-107, :19-40).  The reference builds a
// [B,S,N] int64 index matrix, masks it, and SORTS every row to find the first K
// in-radius indices; scanning the points in index order yields the same list
// directly, so memory is O(S*K) and nothing is sorted.
//
// Bit-exactness with the reference lives in sqdist_expanded(): same expression,
// same rounding order as aten's  -2*matmul + |q|^2 + |p|^2  (see SURVEY.md 7.1).
#include "common.cuh"
#include <string.h>
#include "geom.cuh"

namespace ev2h {

// packed fp32x2 arithmetic (sm_100): both halves are IEEE round-to-nearest operations, bit-identical to the scalar ones
__device__ __forceinline__ uint64_t pack2f(float a, float b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void unpack2f(uint64_t v, float &a, float &b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t mul2f(uint64_t a, uint64_t b) { uint64_t d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ uint64_t add2f(uint64_t a, uint64_t b) { uint64_t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ uint64_t fma2f(uint64_t a, uint64_t b, uint64_t c) { uint64_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }

constexpr int kMaxScales = 4;
constexpr int kBqCentres = 32;    // centres per CTA (one per lane)
constexpr int kBqSegs = 8;        // point ranges scanned in parallel (one per warp)
constexpr int kBqTile = 1024;     // points staged per pass (16 KB of float4: six CTAs per SM, one wave for sa1 at B = 64)

// Optional in-kernel row compaction (see compact.cu for the format): per scale the list of rows the fused kernel
// has to evaluate - every group's real (and, with first_flag, non-duplicate) neighbours rounded up to 8 rows.
struct BallCompact {
    int32_t *rowmap[kMaxScales];
    int32_t *blockgroup[kMaxScales];
    int32_t *n_rows;                  // [n_scales], zeroed before the launch; nullptr = no compaction
};

struct BallParams {
    float r2[kMaxScales];
    int K[kMaxScales];
    int k_off[kMaxScales];
    int k_total;
    float r2_max;
};

// One CTA = kBqCentres centres of one window x kBqSegs point segments.  Lanes of a warp are 32
// different centres looking at the SAME point (a broadcast shared-memory read); the warps of a CTA
// split every staged tile of points into kBqSegs consecutive index ranges.  "First K in index order"
// is kept by scanning each range twice: pass 1 counts the hits per (centre, range, radius), a prefix
// over the ranges gives every range its output offset, pass 2 re-evaluates the distances and writes the
// hits in place while the offset is below K.  Twice the arithmetic, kBqSegs times the parallelism (the
// one-thread-per-centre scan left the SMs at 7 warps each).
template <int NS>
__global__ void __launch_bounds__(kBqCentres * kBqSegs)
ball_query_kernel(const float *__restrict__ xyz, int64_t sb, int64_t sc, int64_t sn,
                  const float *__restrict__ centres, int N, int S, BallParams prm,
                  int32_t *__restrict__ out, int32_t *__restrict__ cnt_out,
                  const uint8_t *__restrict__ first_flag, int32_t *__restrict__ uniq_out, int32_t *__restrict__ ucnt_out,
                  BallCompact comp, int s_base, int s_end) {
    // Optional second list (first_flag != nullptr): the same first-K hits without exact duplicates of an earlier
    // point (first_flag[b,n] = 0), in index order, for the row compaction; ucnt_out = its length.
    // The flag travels in the sign bit of the staged |p|^2 (a sum of squares is never negative), read back with fabsf.
    // staged points, two per record pair so that the distance runs on packed fp32x2 arithmetic (two IEEE operations per
    // instruction, each half rounded exactly like the scalar instruction): ptsA[i] = (x0, x1, y0, y1), ptsB[i] =
    // (z0, z1, |p0|^2, |p1|^2) for points 2i, 2i + 1 of the tile; flagw = first-occurrence bits, one word per 32 points
    __shared__ float4 ptsA[kBqTile / 2], ptsB[kBqTile / 2];
    __shared__ uint32_t flagw[kBqTile / 32];
    __shared__ int ucnt_s[kBqSegs][NS][kBqCentres];
    __shared__ int uemit_s[NS][kBqCentres];              // unique hits written (i.e. within the first K hits), summed over ranges
    __shared__ int cnt_s[kBqSegs][NS][kBqCentres];      // hits of this tile per (range, radius, centre)
    __shared__ int first_s[kBqSegs][NS][kBqCentres];    // first hit of this tile per (range, radius, centre), N if none
    const int b = blockIdx.y;
    const int lane = threadIdx.x & 31, seg = threadIdx.x >> 5;
    // this launch covers the centres [s_base, s_end) of every window (the whole layer, or a range of it while the
    // sampling of the later centres is still running, see ev2h_ball_query_compact_range_f32)
    const int s = s_base + blockIdx.x * kBqCentres + lane;
    const bool live = s < s_end;
    const float *base = xyz + (int64_t)b * sb;

    float qx = 0.f, qy = 0.f, qz = 0.f;
    if (live) {
        const float *c = centres + ((int64_t)b * S + s) * 3;
        qx = c[0]; qy = c[1]; qz = c[2];
    }
    const float qn = sq_norm3(qx, qy, qz);
    int32_t *row = out + ((int64_t)b * S + (live ? s : 0)) * prm.k_total;
    const bool dedup = first_flag != nullptr;
    int32_t *urow = dedup ? uniq_out + ((int64_t)b * S + (live ? s : 0)) * prm.k_total : nullptr;
    int utotal[NS], emitted[NS];                         // unique hits seen so far (same in every warp) / written by this thread
#pragma unroll
    for (int k = 0; k < NS; ++k) { utotal[k] = 0; emitted[k] = 0; }
    if (threadIdx.x < NS * kBqCentres) (&uemit_s[0][0])[threadIdx.x] = 0;     // visible after the first barrier of the tile loop

    int total[NS], first[NS];                            // running over the tiles already processed (same in every warp)
#pragma unroll
    for (int k = 0; k < NS; ++k) { total[k] = 0; first[k] = N; }

    for (int t0 = 0; t0 < N; t0 += kBqTile) {
        const int n_tile = min(kBqTile, N - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < ((n_tile + 31) & ~31); i += kBqCentres * kBqSegs) {
            // past the end of the tile: a point far outside every radius.  Pass 1 still evaluates it (the last word of the
            // last range may be partly padding) and masks its bit off: for a centre with a +inf coordinate its distance is
            // -inf + inf = NaN, which the inclusive rule would take as a hit
            float x = 1e18f, y = 1e18f, z = 1e18f;
            bool fresh = false;
            if (i < n_tile) {
                const int64_t g = (int64_t)(t0 + i) * sn;
                x = base[g]; y = base[sc + g]; z = base[2 * sc + g];
                fresh = !(dedup && first_flag[(int64_t)b * N + t0 + i] == 0);
            }
            const float nn = sq_norm3(x, y, z);
            float *pa = reinterpret_cast<float *>(&ptsA[i >> 1]) + (i & 1), *pb = reinterpret_cast<float *>(&ptsB[i >> 1]) + (i & 1);
            pa[0] = x; pa[2] = y; pb[0] = z; pb[2] = nn;
            const uint32_t fw = __ballot_sync(0xffffffffu, fresh);        // i / 32 is the same for the whole warp
            if (lane == 0) flagw[i >> 5] = fw;
        }
        __syncthreads();
        // ranges are whole 32-point words (pairs never straddle a range)
        const int per = (((n_tile + kBqSegs - 1) / kBqSegs) + 31) & ~31;              // <= kBqTile / kBqSegs = 32 * WORDS points
        const int i0 = min(seg * per, n_tile), i1 = min(i0 + per, n_tile);

        // pass 1: one distance evaluation per (centre, point); the hits of this range are kept as bit masks
        // (bit j of word w = point i0 + 32 w + j), so placing them later needs no second evaluation
        constexpr int WORDS = kBqTile / kBqSegs / 32;
        uint32_t hit[NS][WORDS], fl[WORDS];
        int cnt[NS], fst[NS], ucnt[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) { cnt[k] = 0; fst[k] = N; ucnt[k] = 0; }
        const uint64_t qx2 = pack2f(qx, qx), qy2 = pack2f(qy, qy), qz2 = pack2f(qz, qz), qn2 = pack2f(qn, qn), m2 = pack2f(-2.0f, -2.0f);
#pragma unroll
        for (int w = 0; w < WORDS; ++w) {
            uint32_t m[NS];
#pragma unroll
            for (int k = 0; k < NS; ++k) m[k] = 0u;
            fl[w] = 0u;
            if (i0 + 32 * w < i1) {
                fl[w] = flagw[(i0 >> 5) + w];
                const int pbase = (i0 >> 1) + 16 * w;
                // fully unrolled and branch-free: the hit bits are immediates and every radius costs one compare and one
                // predicated OR per point (with a "skip if outside the largest radius" branch 83 % of the points took
                // the hit path with ~2 of 32 lanes active: ncu, profiles/r02_geom16k_ncu_summary.txt)
#pragma unroll
                for (int j = 0; j < 32; j += 2) {
                    const float4 a = ptsA[pbase + (j >> 1)], c = ptsB[pbase + (j >> 1)];
                    // sqdist_expanded for two points at once: x*x', two FMAs, * -2, + |q|^2, + |p|^2 (geom.cuh)
                    uint64_t t = mul2f(qx2, pack2f(a.x, a.y));
                    t = fma2f(qy2, pack2f(a.z, a.w), t);
                    t = fma2f(qz2, pack2f(c.x, c.y), t);
                    t = mul2f(m2, t);
                    t = add2f(t, qn2);
                    t = add2f(t, pack2f(c.z, c.w));
                    float d0, d1;
                    unpack2f(t, d0, d1);
#pragma unroll
                    for (int k = 0; k < NS; ++k) {
                        if (!(d0 > prm.r2[k])) m[k] |= 1u << j;              // group_idx[sqrdists > r**2] = N  (:102)
                        if (!(d1 > prm.r2[k])) m[k] |= 2u << j;
                    }
                }
                // the padding at the end of the last word is no point: clear its bits.  Inside this branch, where only
                // the word that holds padding pays for it (masking every word: 86 instead of 80 registers for three
                // radii, one CTA less per SM, the whole step 2 % slower on a B200)
                const int live_pts = i1 - (i0 + 32 * w);
                if (live_pts < 32) {
#pragma unroll
                    for (int k = 0; k < NS; ++k) m[k] &= (1u << live_pts) - 1u;
                }
            }
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                hit[k][w] = m[k];
                if (m[k] != 0u && cnt[k] == 0) fst[k] = t0 + i0 + 32 * w + __ffs(m[k]) - 1;
                cnt[k] += __popc(m[k]);
                ucnt[k] += __popc(m[k] & fl[w]);
            }
        }
#pragma unroll
        for (int k = 0; k < NS; ++k) { cnt_s[seg][k][lane] = cnt[k]; first_s[seg][k][lane] = fst[k]; ucnt_s[seg][k][lane] = ucnt[k]; }
        __syncthreads();

        // offsets of this range, and the tile's totals
        // (the unique-hit offsets ignore the K cut-off: hits are emitted in index order, so those that make
        // the cut are a prefix of the unique sequence and their positions are unaffected by the ones that do not)
        int off[NS], tile_total[NS], uoff[NS], utile[NS];
        bool any_room = false;
#pragma unroll
        for (int k = 0; k < NS; ++k) {
            int o = total[k], tt = 0, uo = utotal[k], ut = 0;
            for (int g = 0; g < kBqSegs; ++g) {
                const int c = cnt_s[g][k][lane], uc = ucnt_s[g][k][lane];
                if (g < seg) { o += c; uo += uc; }
                tt += c; ut += uc;
                if (first[k] == N && first_s[g][k][lane] != N) first[k] = first_s[g][k][lane];
            }
            off[k] = o; tile_total[k] = tt; uoff[k] = uo; utile[k] = ut;
            any_room = any_room || (cnt[k] > 0 && o < prm.K[k]);
        }

        // pass 2: walk the set bits and write the hits of this range at their final positions
        if (live && any_room) {
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                int o = off[k], uo = uoff[k];
#pragma unroll
                for (int w = 0; w < WORDS; ++w) {
                    uint32_t m = hit[k][w];
                    while (m != 0u && o < prm.K[k]) {
                        const int j = __ffs(m) - 1;
                        m &= m - 1u;
                        const int pt = t0 + i0 + 32 * w + j;
                        row[prm.k_off[k] + o] = pt;
                        if (dedup && ((fl[w] >> j) & 1u)) { urow[prm.k_off[k] + uo] = pt; ++uo; ++emitted[k]; }
                        ++o;
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < NS; ++k) { total[k] += tile_total[k]; utotal[k] += utile[k]; }
    }
    if (dedup) {
#pragma unroll
        for (int k = 0; k < NS; ++k)
            if (emitted[k]) atomicAdd(&uemit_s[k][lane], emitted[k]);
    }
    __syncthreads();
    if (comp.n_rows != nullptr) {
        // ---- row compaction in place: reserve this CTA's rows of every scale with one atomic add, then copy the
        // hit lists (written above by all the warps; visible after the barrier) into the compact row list
        __shared__ int coff_s[NS][kBqCentres], ccnt_s[NS][kBqCentres];
        if (seg == 0) {
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                const int c = dedup ? uemit_s[k][lane] : min(total[k], prm.K[k]);
                const int rows = live ? ((max(c, 1) + 7) & ~7) : 0;
                int incl = rows;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, d);
                    if (lane >= d) incl += v;
                }
                int base = 0;
                if (lane == 31 && incl > 0) base = atomicAdd(comp.n_rows + k, incl);
                base = __shfl_sync(0xffffffffu, base, 31);
                coff_s[k][lane] = base + incl - rows;
                ccnt_s[k][lane] = c;
            }
        }
        __syncthreads();
        const int32_t *lists = dedup ? uniq_out : out;
        for (int cidx = seg; cidx < kBqCentres; cidx += kBqSegs) {
            const int sc_ = s_base + blockIdx.x * kBqCentres + cidx;
            if (sc_ >= s_end) break;
            const int64_t g = (int64_t)b * S + sc_;
#pragma unroll
            for (int k = 0; k < NS; ++k) {
                const int c = ccnt_s[k][cidx], real = max(c, 1), rows = (real + 7) & ~7, off = coff_s[k][cidx];
                const int32_t *src = lists + g * prm.k_total + prm.k_off[k];
                for (int j = lane; j < rows; j += 32) {
                    const int pt = c < 1 ? -1 : src[j < real ? j : 0];        // c == 0: empty ball
                    comp.rowmap[k][off + j] = (pt >= 0 && pt < N) ? (int32_t)((int64_t)b * N + pt) : -1;
                    if ((j & 7) == 0) comp.blockgroup[k][(off + j) >> 3] = (int32_t)g;
                }
            }
        }
    }
    if (!live) return;
    if (ucnt_out != nullptr && seg == 0) {
#pragma unroll
        for (int k = 0; k < NS; ++k) ucnt_out[(int64_t)k * gridDim.y * S + (int64_t)b * S + s] = uemit_s[k][lane];
    }
    if (cnt_out != nullptr && seg == 0) {                // real (unpadded) neighbours per scale, for the row compaction
#pragma unroll
        for (int k = 0; k < NS; ++k) cnt_out[(int64_t)k * gridDim.y * S + (int64_t)b * S + s] = min(total[k], prm.K[k]);   // [scale][b*S+s]
    }
    // pad with the first hit (:104-106); the ranges share the padding slots
#pragma unroll
    for (int k = 0; k < NS; ++k)
        for (int j = total[k] + seg; j < prm.K[k]; j += kBqSegs) row[prm.k_off[k] + j] = first[k];
}

// square_distance as a standalone op (pointnet2_utils.py:19-40): out[b,s,n], bit-exact.
__global__ void __launch_bounds__(256)
square_distance_kernel(const float *__restrict__ src, const float *__restrict__ dst, int S, int N,
                       float *__restrict__ out, int64_t total) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int n = (int)(e % N);
    const int64_t bs = e / N;
    const int64_t b = bs / S;
    const float *q = src + bs * 3, *p = dst + (b * N + n) * 3;
    const float4 pp = make_float4(p[0], p[1], p[2], sq_norm3(p[0], p[1], p[2]));
    out[e] = sqdist_expanded(q[0], q[1], q[2], sq_norm3(q[0], q[1], q[2]), pp);
}

// index_points (pointnet2_utils.py:43-60): out[b,m,:] = table[b, idx[b,m], :]
__global__ void __launch_bounds__(256)
index_rows_kernel(const float *__restrict__ table, const int32_t *__restrict__ idx, int N, int Mi, int C,
                  float *__restrict__ out, int64_t total) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int c = (int)(e % C);
    const int64_t bm = e / C;
    const int64_t b = bm / Mi;
    const int p = idx[bm];
    out[e] = (p >= 0 && p < N) ? table[(b * N + p) * (int64_t)C + c] : 0.f;
}

}  // namespace ev2h

extern "C" int ev2h_square_distance_f32(const float *src_rows, const float *dst_rows, int B, int S, int N,
                                        float *out, ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(src_rows && dst_rows && out, "ev2h_square_distance_f32: null argument");
    EV2H_REQUIRE(B > 0 && S > 0 && N > 0, "ev2h_square_distance_f32: bad sizes");
    const int64_t total = (int64_t)B * S * N;
    square_distance_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(src_rows, dst_rows, S, N, out, total);
    return check_launch("ev2h_square_distance_f32");
}

extern "C" int ev2h_index_rows_f32(const float *table_rows, const int32_t *idx, int B, int N, int M, int C,
                                   float *out, ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(table_rows && idx && out, "ev2h_index_rows_f32: null argument");
    EV2H_REQUIRE(B > 0 && N > 0 && M > 0 && C > 0, "ev2h_index_rows_f32: bad sizes");
    const int64_t total = (int64_t)B * M * C;
    index_rows_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(stream)>>>(table_rows, idx, N, M, C, out, total);
    return check_launch("ev2h_index_rows_f32");
}

static int ball_query_impl(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                           const float *centres_rows, int B, int N, int S, int n_scales,
                           const float *radius_sq_host, const int32_t *nsample_host,
                           int32_t *out_idx, int32_t *out_cnt, const uint8_t *first_flag, int32_t *out_uniq, int32_t *out_ucnt,
                           int32_t *const *rowmap_host, int32_t *const *blockgroup_host, int32_t *n_rows_dev,
                           ev2h_stream_t stream, int s_begin = 0, int s_count = -1, int reset_rows = 1);

extern "C" int ev2h_ball_query_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                   const float *centres_rows, int B, int N, int S, int n_scales,
                                   const float *radius_sq_host, const int32_t *nsample_host,
                                   int32_t *out_idx, ev2h_stream_t stream) {
    return ball_query_impl(xyz, stride_b, stride_c, stride_n, centres_rows, B, N, S, n_scales, radius_sq_host, nsample_host,
                           out_idx, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, stream);
}

extern "C" int ev2h_ball_query_cnt_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                       const float *centres_rows, int B, int N, int S, int n_scales,
                                       const float *radius_sq_host, const int32_t *nsample_host,
                                       int32_t *out_idx, int32_t *out_cnt, ev2h_stream_t stream) {
    return ball_query_impl(xyz, stride_b, stride_c, stride_n, centres_rows, B, N, S, n_scales, radius_sq_host, nsample_host,
                           out_idx, out_cnt, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, stream);
}

extern "C" int ev2h_ball_query_uniq_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                        const float *centres_rows, int B, int N, int S, int n_scales,
                                        const float *radius_sq_host, const int32_t *nsample_host,
                                        int32_t *out_idx, const uint8_t *first_flag, int32_t *out_uniq, int32_t *out_ucnt,
                                        ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(first_flag && out_uniq && out_ucnt, "ev2h_ball_query_uniq_f32: null argument");
    return ball_query_impl(xyz, stride_b, stride_c, stride_n, centres_rows, B, N, S, n_scales, radius_sq_host, nsample_host,
                           out_idx, nullptr, first_flag, out_uniq, out_ucnt, nullptr, nullptr, nullptr, stream);
}

extern "C" int ev2h_ball_query_compact_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                           const float *centres_rows, int B, int N, int S, int n_scales,
                                           const float *radius_sq_host, const int32_t *nsample_host,
                                           int32_t *out_idx, const uint8_t *first_flag, int32_t *uniq_scratch,
                                           int32_t *const *rowmap_host, int32_t *const *blockgroup_host, int32_t *n_rows_dev,
                                           ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(rowmap_host && blockgroup_host && n_rows_dev, "ev2h_ball_query_compact_f32: null argument");
    EV2H_REQUIRE((first_flag == nullptr) == (uniq_scratch == nullptr), "ev2h_ball_query_compact_f32: first_flag and uniq_scratch go together");
    EV2H_REQUIRE((int64_t)B * S * 128 < 2147483647LL, "ev2h_ball_query_compact_f32: too many groups for 32-bit row offsets");
    return ball_query_impl(xyz, stride_b, stride_c, stride_n, centres_rows, B, N, S, n_scales, radius_sq_host, nsample_host,
                           out_idx, nullptr, first_flag, uniq_scratch, nullptr, rowmap_host, blockgroup_host, n_rows_dev, stream);
}

extern "C" int ev2h_ball_query_compact_range_f32(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                                                 const float *centres_rows, int B, int N, int S, int s_begin, int s_count, int reset_rows,
                                                 int n_scales, const float *radius_sq_host, const int32_t *nsample_host,
                                                 int32_t *out_idx, const uint8_t *first_flag, int32_t *uniq_scratch,
                                                 int32_t *const *rowmap_host, int32_t *const *blockgroup_host, int32_t *n_rows_dev,
                                                 ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(rowmap_host && blockgroup_host && n_rows_dev, "ev2h_ball_query_compact_range_f32: null argument");
    EV2H_REQUIRE((first_flag == nullptr) == (uniq_scratch == nullptr), "ev2h_ball_query_compact_range_f32: first_flag and uniq_scratch go together");
    EV2H_REQUIRE((int64_t)B * S * 128 < 2147483647LL, "ev2h_ball_query_compact_range_f32: too many groups for 32-bit row offsets");
    return ball_query_impl(xyz, stride_b, stride_c, stride_n, centres_rows, B, N, S, n_scales, radius_sq_host, nsample_host,
                           out_idx, nullptr, first_flag, uniq_scratch, nullptr, rowmap_host, blockgroup_host, n_rows_dev, stream,
                           s_begin, s_count, reset_rows);
}

static int ball_query_impl(const float *xyz, int64_t stride_b, int64_t stride_c, int64_t stride_n,
                           const float *centres_rows, int B, int N, int S, int n_scales,
                           const float *radius_sq_host, const int32_t *nsample_host,
                           int32_t *out_idx, int32_t *out_cnt, const uint8_t *first_flag, int32_t *out_uniq, int32_t *out_ucnt,
                           int32_t *const *rowmap_host, int32_t *const *blockgroup_host, int32_t *n_rows_dev,
                           ev2h_stream_t stream, int s_begin, int s_count, int reset_rows) {
    using namespace ev2h;
    EV2H_REQUIRE(xyz && centres_rows && out_idx && radius_sq_host && nsample_host, "ev2h_ball_query_f32: null argument");
    if (s_count < 0) s_count = S - s_begin;
    EV2H_REQUIRE(s_begin >= 0 && s_count > 0 && s_begin + s_count <= S && s_begin % kBqCentres == 0,
                 "ev2h_ball_query_f32: centre range [%d, %d) of %d (the start must be a multiple of %d)", s_begin, s_begin + s_count, S, kBqCentres);
    EV2H_REQUIRE(B > 0 && N > 0 && S > 0, "ev2h_ball_query_f32: B, N, S must be positive");
    EV2H_REQUIRE(B <= 65535, "ev2h_ball_query_f32: B=%d exceeds 65535 windows per call", B);
    if (n_scales < 1 || n_scales > kMaxScales)
        return fail(EV2H_ERR_UNSUPPORTED, "ev2h_ball_query_f32: n_scales=%d not in 1..%d", n_scales, kMaxScales);
    BallParams prm;
    int off = 0;
    prm.r2_max = radius_sq_host[0];
    for (int i = 0; i < kMaxScales; ++i) {
        const bool on = i < n_scales;
        prm.r2[i] = on ? radius_sq_host[i] : 0.f;
        prm.K[i] = on ? nsample_host[i] : 0;
        prm.k_off[i] = off;
        if (on) {
            EV2H_REQUIRE(nsample_host[i] > 0, "ev2h_ball_query_f32: nsample[%d] must be positive", i);
            off += nsample_host[i];
            // NaN-safe max: keep a NaN radius out of r2_max so the prefilter never drops a candidate
            if (radius_sq_host[i] > prm.r2_max) prm.r2_max = radius_sq_host[i];
        }
    }
    prm.k_total = off;
    BallCompact comp;
    memset(&comp, 0, sizeof(comp));
    if (n_rows_dev != nullptr) {
        for (int i = 0; i < n_scales; ++i) {
            EV2H_REQUIRE(rowmap_host[i] && blockgroup_host[i] && nsample_host[i] % 8 == 0,
                         "ev2h_ball_query_compact_f32: scale %d: K must be a multiple of 8 and buffers non-null", i);
            comp.rowmap[i] = rowmap_host[i];
            comp.blockgroup[i] = blockgroup_host[i];
        }
        comp.n_rows = n_rows_dev;
        if (reset_rows) {
            cudaError_t e = cudaMemsetAsync(n_rows_dev, 0, sizeof(int32_t) * n_scales, as_stream(stream));
            if (e != cudaSuccess) return fail(EV2H_ERR_CUDA, "ev2h_ball_query_compact_f32: memset: %s", cudaGetErrorString(e));
        }
    }
    dim3 grid((s_count + kBqCentres - 1) / kBqCentres, B);
    const int s_end = s_begin + s_count;
    constexpr int kBqThreads = kBqCentres * kBqSegs;
    cudaStream_t st = as_stream(stream);
    switch (n_scales) {
        case 1: ball_query_kernel<1><<<grid, kBqThreads, 0, st>>>(xyz, stride_b, stride_c, stride_n, centres_rows, N, S, prm, out_idx, out_cnt, first_flag, out_uniq, out_ucnt, comp, s_begin, s_end); break;
        case 2: ball_query_kernel<2><<<grid, kBqThreads, 0, st>>>(xyz, stride_b, stride_c, stride_n, centres_rows, N, S, prm, out_idx, out_cnt, first_flag, out_uniq, out_ucnt, comp, s_begin, s_end); break;
        case 3: ball_query_kernel<3><<<grid, kBqThreads, 0, st>>>(xyz, stride_b, stride_c, stride_n, centres_rows, N, S, prm, out_idx, out_cnt, first_flag, out_uniq, out_ucnt, comp, s_begin, s_end); break;
        default: ball_query_kernel<4><<<grid, kBqThreads, 0, st>>>(xyz, stride_b, stride_c, stride_n, centres_rows, N, S, prm, out_idx, out_cnt, first_flag, out_uniq, out_ucnt, comp, s_begin, s_end); break;
    }
    return check_launch("ev2h_ball_query_f32");
}
