// Shared-MLP layer on the 5th-generation tensor cores (tcgen05 / TMEM):
//     y = relu(x W' + b'), optionally max-pooled over runs of K consecutive rows.
//
// Replaces one Conv2d(1x1) + BatchNorm2d(eval) + ReLU step of the reference MLP
// (src/Ev2Hands/model/pointnet2_utils.py:253-256 / :193-197) and, when pooling, the
// torch.max over the neighbour axis (:257 / :199) - same contract as linear_ffma.cu.
//
// Two arithmetic modes over fp32 activations in HBM:
//   TF32X3  fp32-accurate: x = x_hi + x_lo, w = w_hi + w_lo (hi exactly tf32), three
//           kind::tf32 UMMAs per K step: x_lo*w_hi + x_hi*w_lo + x_hi*w_hi, fp32 accumulate.
//   BF16    one kind::f16 UMMA per K step on bf16-rounded operands, fp32 accumulate.
//
// Persistent, warp-specialised CTA (one per SM), 128-row tiles:
//   warps 5+   loaders : groups of 4 warps take K chunks (32 input channels x 128 rows) round-robin:
//                        fp32 LDG.128, split / convert, write the UMMA operand image to shared memory
//                        (K-major, no swizzle: 16-byte chunks, consecutive rows contiguous);
//                        weights arrive pre-packed in the same image by ONE bulk async copy/stage
//   warp 4     issuer  : one thread issues tcgen05.mma into one of two TMEM accumulators and
//                        commits to the stage's "empty" barrier / the accumulator's "full" barrier
//   warps 0-3  epilogue: tcgen05.ld their 32 TMEM lanes, bias + ReLU, then either store the
//                        row or reduce the max over the group with warp REDUX (+ shared memory
//                        across warps) - overlapped with the next tile's UMMAs.
#include "common.cuh"
#include "tc_common.cuh"
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace ev2h {

constexpr int TC_BLOCK_M = 128;
constexpr int TC_KC = 32;              // input channels per pipeline stage
constexpr int TC_MAX_N = 256;          // accumulator width per tile (two of them fill TMEM's 512 columns)
constexpr int TC_LOADER_GROUPS = 2;    // groups of 4 loader warps working on different stages
constexpr int TC_THREADS = 32 * (5 + 4 * TC_LOADER_GROUPS);   // 4 epilogue + 1 issuer + loader warps
constexpr int TC_MAX_STAGES = 8;

// MIXED: tf32 hi*hi + two bf16 correction products;  F16X3: fp16 hi/lo pairs, three kind::f16 products (tc::split_f16x2)
enum { TC_MODE_BF16 = 0, TC_MODE_TF32X3 = 1, TC_MODE_MIXED = 2, TC_MODE_F16X3 = 3 };

__host__ __device__ constexpr int tc_elem_bytes(int mode) { return (mode == TC_MODE_BF16 || mode == TC_MODE_F16X3) ? 2 : 4; }
// bytes of one operand image holding `rows` rows x TC_KC channels (one precision part)
__host__ __device__ constexpr int tc_part_bytes(int mode, int rows) { return rows * TC_KC * tc_elem_bytes(mode); }
__host__ __device__ constexpr int tc_parts(int mode) { return mode == TC_MODE_BF16 ? 1 : 2; }
__host__ __device__ constexpr int tc_stage_bytes(int mode, int n_blk) {
    return tc_parts(mode) * (tc_part_bytes(mode, TC_BLOCK_M) + tc_part_bytes(mode, n_blk));
}

struct TcParams {
    const float *x; int64_t M; int ld_x; int Cin;
    const uint8_t *w_packed; const float *bias;
    int n_blk;          // accumulator width (multiple of 16, <= 256)
    int n_blocks;       // ceil(Cout_pad / n_blk)
    int n_kc;           // ceil(Cin / 32)
    int Cout; int pool_rows;
    float *y; int ld_y; int y_col_off;
    int n_store_total;  // columns of y that may be written (>= Cout when zero padding exists)
    int stages;
    int debug;
    int relu;           // 0: y = x W' + b' (no activation)
    // Conv1d over the row axis (kernel size `taps`, zero padding taps / 2, rows_per_win consecutive rows = one sequence):
    // the operand row of output row r is [x[r - taps/2], ..., x[r + taps/2]] (tap_cin channels each), rows outside the
    // sequence being zero - gathered by the loaders, never materialised.  taps == 1: the plain layer.
    int taps, tap_cin, rows_per_win;
    // optional per-channel affine AFTER the activation (a BatchNorm that follows the ReLU): y = act(.) * scale + shift
    const float *post_scale, *post_shift;
    int32_t *range_flag;    // optional (F16X3): bit 0 set when an activation operand left the fp16 range or was NaN
};

// ---- weight packing: folded [Cin_pad16, ld_w] fp32 (input-channel major) -> per (n-block, stage)
// shared-memory images so a stage is one contiguous bulk copy.
template <int MODE>
__global__ void __launch_bounds__(256)
tc_pack_kernel(const float *__restrict__ wt, int ld_w, int cin_rows, int cout_cols, int n_blk, int n_blocks,
               int n_kc, int kc_len, uint8_t *__restrict__ out) {
    const int64_t total = (int64_t)n_blocks * n_kc * n_blk * kc_len;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= total) return;
    const int kk = (int)(e % kc_len);
    int64_t t = e / kc_len;
    const int n = (int)(t % n_blk);
    t /= n_blk;
    const int kc = (int)(t % n_kc);
    const int nb = (int)(t / n_kc);
    const int k = kc * kc_len + kk, col = nb * n_blk + n;
    const float w = (k < cin_rows && col < cout_cols) ? wt[(int64_t)k * ld_w + col] : 0.f;
    constexpr int EB = tc_elem_bytes(MODE);
    constexpr int CH = 16 / EB;                         // elements per 16-byte chunk
    const size_t part = (size_t)n_blk * kc_len * EB;
    uint8_t *stage = out + ((size_t)nb * n_kc + kc) * (tc_parts(MODE) * part);
    const size_t off = (size_t)(kk / CH) * ((size_t)n_blk * 16) + (size_t)n * 16 + (size_t)(kk % CH) * EB;
    if (MODE == TC_MODE_BF16) {
        *reinterpret_cast<__nv_bfloat16 *>(stage + off) = __float2bfloat16_rn(w);
    } else if (MODE == TC_MODE_F16X3) {
        // [hi as fp16 | lo as fp16], 16-byte chunks of 8 channels
        const __half hi = __float2half_rn(w);
        *reinterpret_cast<__half *>(stage + off) = hi;
        *reinterpret_cast<__half *>(stage + part + off) = __float2half_rn(w - __half2float(hi));
    } else if (MODE == TC_MODE_MIXED) {
        // [hi as tf32 | w as bf16 | lo as bf16]: the fused kernel's hi*hi runs in tf32, the two correction
        // products on the bf16 copies (16-byte chunks of 8 channels)
        float hi, lo;
        tc::split_tf32(w, hi, lo);
        *reinterpret_cast<float *>(stage + off) = hi;
        const size_t off16 = (size_t)(kk / 8) * ((size_t)n_blk * 16) + (size_t)n * 16 + (size_t)(kk % 8) * 2;
        *reinterpret_cast<__nv_bfloat16 *>(stage + part + off16) = __float2bfloat16_rn(w);
        *reinterpret_cast<__nv_bfloat16 *>(stage + part + part / 2 + off16) = __float2bfloat16_rn(lo);
    } else {
        float hi, lo;
        tc::split_tf32(w, hi, lo);
        *reinterpret_cast<float *>(stage + off) = hi;
        *reinterpret_cast<float *>(stage + part + off) = lo;
    }
}

template <int MODE>
__global__ void __launch_bounds__(TC_THREADS, 1)
linear_tc_kernel(const TcParams p) {
    extern __shared__ __align__(128) uint8_t tc_smem[];
    constexpr int EB = tc_elem_bytes(MODE);
    constexpr int PARTS = tc_parts(MODE);
    constexpr int A_PART = tc_part_bytes(MODE, TC_BLOCK_M);
    constexpr int CH = 16 / EB;                 // elements per 16-byte chunk: 4 (tf32) / 8 (bf16)
    constexpr int UMMA_K = 32 / EB;             // 8 (tf32) / 16 (bf16)
    constexpr int K_STEPS = TC_KC / UMMA_K;     // 4 / 2
    const int n_blk = p.n_blk;
    const int b_part = tc_part_bytes(MODE, n_blk);
    const int stage_bytes = PARTS * (A_PART + b_part);
    const int stages = p.stages;

    uint8_t *ring = tc_smem;
    uint8_t *tail = tc_smem + (size_t)stages * stage_bytes;
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(tail);           // [stages]
    uint64_t *empty_bar = full_bar + TC_MAX_STAGES;                    // [stages]
    uint64_t *acc_full = empty_bar + TC_MAX_STAGES;                    // [2]
    uint64_t *acc_empty = acc_full + 2;                                // [2]
    uint32_t *tmem_base_slot = reinterpret_cast<uint32_t *>(acc_empty + 2);
    float *bias_s = reinterpret_cast<float *>(tmem_base_slot + 4);     // [n_blocks * n_blk]
    float *post_a = bias_s + p.n_blocks * n_blk;                       // [n_blocks * n_blk] each (scale 1 / shift 0 when absent)
    float *post_b = post_a + p.n_blocks * n_blk;
    float *red = post_b + p.n_blocks * n_blk;                          // [2][4][n_blk]

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t m_tiles = (p.M + TC_BLOCK_M - 1) / TC_BLOCK_M;
    const int64_t n_tiles = m_tiles * p.n_blocks;

    if (tid == 0) {
        for (int s = 0; s < stages; ++s) {
            tc::mbar_init(full_bar + s, 128 + 1);     // 128 loader arrivals + the weight copy's expect_tx arrival
            tc::mbar_init(empty_bar + s, 1);          // one tcgen05.commit
        }
        for (int a = 0; a < 2; ++a) {
            tc::mbar_init(acc_full + a, 1);
            tc::mbar_init(acc_empty + a, 128);
        }
        tc::fence_mbar_init();
    }
    for (int i = tid; i < p.n_blocks * n_blk; i += TC_THREADS) {
        bias_s[i] = p.bias[i];
        post_a[i] = (p.post_scale && i < p.Cout) ? p.post_scale[i] : 1.f;
        post_b[i] = (p.post_shift && i < p.Cout) ? p.post_shift[i] : 0.f;
    }
    const bool post = p.post_scale != nullptr || p.post_shift != nullptr;
    if (warp == 4) tc::tmem_alloc(tmem_base_slot, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_base_slot;

    if (warp >= 5) {
        // ================================ loaders ================================
        // TC_LOADER_GROUPS groups of 4 warps take the K chunks round-robin, so several stages are
        // being fetched at once.  Inside a group, warp wq owns rows [32 wq, 32 wq + 32) of the tile.
        // Lane mapping: 8 consecutive lanes = 8 consecutive rows of ONE 16-byte operand chunk (a
        // conflict-free 128-byte shared-memory store), the 4 lane octets = 4 adjacent chunks, so a
        // warp-wide load covers 8 rows x 64 contiguous bytes (full 32-byte sectors).
        const int lw = warp - 5, grp = lw >> 2, wq = lw & 3;
        const int l8 = lane & 7, oct = lane >> 3;
        // Channels [tap_cin, ld_x) of a row are padding: never part of the product, whatever they hold.  A float4 that
        // starts below tap_cin lies inside the row (ld_x is a multiple of 4); its components from tap_cin on are zeroed
        // when the chunk is converted (not at the load: the loads of the next chunk must stay in flight).  With taps > 1,
        // tap_cin is a multiple of 32 and a chunk never crosses it.
        const int k_lim = p.tap_cin;
        auto mask_tail = [&](float4 &t, int k) {
            if (k + 1 >= k_lim) t.y = 0.f;
            if (k + 2 >= k_lim) t.z = 0.f;
            if (k + 3 >= k_lim) t.w = 0.f;
        };
        uint32_t hmax = 0;      // F16X3: running maximum of |fp16 hi word| pairs this thread wrote (range check)
        // The group's NEXT chunk is loaded into registers before the current one is converted and stored, so
        // the global-load latency of a stage overlaps the previous stage's wait / store / arrive.
        const uint32_t my_tiles = (uint32_t)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
        const uint32_t total = my_tiles * (uint32_t)p.n_kc;                 // chunks this CTA walks
        auto issue_loads = [&](uint32_t n, float4 (&v)[8]) {
            const int64_t tile = blockIdx.x + (int64_t)(n / (uint32_t)p.n_kc) * gridDim.x;
            const int kc = (int)(n % (uint32_t)p.n_kc);
            const int64_t m0 = (tile / p.n_blocks) * TC_BLOCK_M;
            // Conv1d taps: a 32-channel chunk lies inside one tap (tap_cin is a multiple of 32); its source row is shifted
            // by tap - taps / 2 and must stay inside the output row's sequence
            const int tap = p.taps > 1 ? (kc * TC_KC) / p.tap_cin : 0;
            const int k_base = kc * TC_KC - tap * p.tap_cin;
            const int shift = tap - (p.taps >> 1);
            auto src_row = [&](int64_t out_row, bool &ok) {
                ok = out_row < p.M;
                if (p.taps == 1) return out_row;
                const int64_t sr = out_row + shift;
                ok = ok && sr >= 0 && sr < p.M && (sr / p.rows_per_win) == (out_row / p.rows_per_win);
                return sr;
            };
            if (MODE == TC_MODE_TF32X3) {                     // (MIXED uses the 8-channels-per-lane mapping below)
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int row = 32 * wq + (i >> 1) * 8 + l8;
                    const int k = k_base + 4 * (oct + 4 * (i & 1));
                    bool ok;
                    const int64_t sr = src_row(m0 + row, ok);
                    v[i] = (ok && k < k_lim)
                               ? __ldg(reinterpret_cast<const float4 *>(p.x + sr * (int64_t)p.ld_x + k))
                               : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            } else {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int row = 32 * wq + i * 8 + l8;
                    const int k = k_base + 8 * oct;
                    bool ok;
                    const int64_t sr = src_row(m0 + row, ok);
                    const float *src = p.x + sr * (int64_t)p.ld_x + k;
                    v[2 * i] = (ok && k < k_lim) ? __ldg(reinterpret_cast<const float4 *>(src)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    v[2 * i + 1] = (ok && k + 4 < k_lim) ? __ldg(reinterpret_cast<const float4 *>(src + 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
        };
        // Stage ownership: the number of stages is a multiple of TC_LOADER_GROUPS (host), so stage n % stages is always
        // filled by group n % TC_LOADER_GROUPS and a group waits on the "empty" barriers of its OWN stages only.  Its
        // wait for the phase that frees chunk n then can never be more than one phase behind the barrier (the next
        // completion needs this very group's fill).  Round 1 let every group walk all stages and wait on the other
        // group's barriers too; an observer that reached its try_wait after the stage had been filled, consumed AND
        // released again saw the parity flipped back and blocked for good - one CTA in ~10^5 tiles, found when the
        // training path ran the kernel over 2 M rows (the time-bounded wait trapped instead of hanging the GPU).
        float4 v[8];
        if ((uint32_t)grp < total) issue_loads((uint32_t)grp, v);
        for (uint32_t n = (uint32_t)grp; n < total; n += TC_LOADER_GROUPS) {
            {
                const int stage = (int)(n % (uint32_t)stages);
                const uint32_t phase = (n / (uint32_t)stages) & 1u;
                {
                    const int64_t tile = blockIdx.x + (int64_t)(n / (uint32_t)p.n_kc) * gridDim.x;
                    const int kc = (int)(n % (uint32_t)p.n_kc);
                    const int nb = (int)(tile % p.n_blocks);
                    float4 vn[8];
                    const bool has_next = n + TC_LOADER_GROUPS < total;
                    if (has_next) issue_loads(n + TC_LOADER_GROUPS, vn);
                    if (p.taps == 1 && (kc + 1) * TC_KC > k_lim) {      // the chunk that ends mid-way: warp-uniform branch
                        if (MODE == TC_MODE_TF32X3) {
#pragma unroll
                            for (int i = 0; i < 8; ++i) mask_tail(v[i], kc * TC_KC + 4 * (oct + 4 * (i & 1)));
                        } else {
#pragma unroll
                            for (int i = 0; i < 8; ++i) mask_tail(v[i], kc * TC_KC + 8 * oct + 4 * (i & 1));
                        }
                    }
                    tc::mbar_wait(empty_bar + stage, phase ^ 1);
                    uint8_t *st = ring + (size_t)stage * stage_bytes;
                    if (wq == 0 && lane == 0) {
                        const uint32_t wbytes = (uint32_t)(PARTS * b_part);
                        tc::mbar_arrive_expect_tx(full_bar + stage, wbytes);
                        tc::bulk_g2s(st + PARTS * A_PART, p.w_packed + ((size_t)nb * p.n_kc + kc) * wbytes, wbytes,
                                     full_bar + stage);
                    }
                    if (MODE == TC_MODE_TF32X3) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            const int row = 32 * wq + (i >> 1) * 8 + l8;
                            const int c = oct + 4 * (i & 1);
                            float4 hi, lo;
                            tc::split_tf32(v[i].x, hi.x, lo.x); tc::split_tf32(v[i].y, hi.y, lo.y);
                            tc::split_tf32(v[i].z, hi.z, lo.z); tc::split_tf32(v[i].w, hi.w, lo.w);
                            *reinterpret_cast<float4 *>(st + c * (TC_BLOCK_M * 16) + row * 16) = hi;
                            *reinterpret_cast<float4 *>(st + A_PART + c * (TC_BLOCK_M * 16) + row * 16) = lo;
                        }
                    } else if (MODE == TC_MODE_F16X3) {
                        // [x_hi as fp16 | x_lo as fp16]: 8 channels of a row = one 16-byte chunk of each part
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int row = 32 * wq + i * 8 + l8;
                            uint4 hb, lb;
                            tc::split_f16x2(v[2 * i].x, v[2 * i].y, hb.x, lb.x); tc::split_f16x2(v[2 * i].z, v[2 * i].w, hb.y, lb.y);
                            tc::split_f16x2(v[2 * i + 1].x, v[2 * i + 1].y, hb.z, lb.z); tc::split_f16x2(v[2 * i + 1].z, v[2 * i + 1].w, hb.w, lb.w);
                            // inputs may be negative here (unlike the fused kernel's post-ReLU operands): sign bits off
                            hmax = tc::max_u16x2(tc::max_u16x2(hmax, tc::max_u16x2(hb.x & 0x7fff7fffu, hb.y & 0x7fff7fffu)),
                                                 tc::max_u16x2(hb.z & 0x7fff7fffu, hb.w & 0x7fff7fffu));
                            *reinterpret_cast<uint4 *>(st + oct * (TC_BLOCK_M * 16) + row * 16) = hb;
                            *reinterpret_cast<uint4 *>(st + A_PART + oct * (TC_BLOCK_M * 16) + row * 16) = lb;
                        }
                    } else if (MODE == TC_MODE_MIXED) {
                        // [x_hi as tf32 | x as bf16 | x_lo as bf16] (the layout of tc_pack_kernel<MIXED> and of
                        // sa_fused_tc.cu): 8 channels of a row = two tf32 chunks and one chunk of each bf16 copy
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int row = 32 * wq + i * 8 + l8;
                            float4 h0, l0, h1, l1;
                            tc::split_tf32(v[2 * i].x, h0.x, l0.x); tc::split_tf32(v[2 * i].y, h0.y, l0.y);
                            tc::split_tf32(v[2 * i].z, h0.z, l0.z); tc::split_tf32(v[2 * i].w, h0.w, l0.w);
                            tc::split_tf32(v[2 * i + 1].x, h1.x, l1.x); tc::split_tf32(v[2 * i + 1].y, h1.y, l1.y);
                            tc::split_tf32(v[2 * i + 1].z, h1.z, l1.z); tc::split_tf32(v[2 * i + 1].w, h1.w, l1.w);
                            *reinterpret_cast<float4 *>(st + (2 * oct) * (TC_BLOCK_M * 16) + row * 16) = h0;
                            *reinterpret_cast<float4 *>(st + (2 * oct + 1) * (TC_BLOCK_M * 16) + row * 16) = h1;
                            uint4 xb, lb;
                            xb.x = tc::bf16x2(v[2 * i].x, v[2 * i].y); xb.y = tc::bf16x2(v[2 * i].z, v[2 * i].w);
                            xb.z = tc::bf16x2(v[2 * i + 1].x, v[2 * i + 1].y); xb.w = tc::bf16x2(v[2 * i + 1].z, v[2 * i + 1].w);
                            lb.x = tc::bf16x2(l0.x, l0.y); lb.y = tc::bf16x2(l0.z, l0.w);
                            lb.z = tc::bf16x2(l1.x, l1.y); lb.w = tc::bf16x2(l1.z, l1.w);
                            *reinterpret_cast<uint4 *>(st + A_PART + oct * (TC_BLOCK_M * 16) + row * 16) = xb;
                            *reinterpret_cast<uint4 *>(st + A_PART + A_PART / 2 + oct * (TC_BLOCK_M * 16) + row * 16) = lb;
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int row = 32 * wq + i * 8 + l8;
                            __nv_bfloat162 q0 = __floats2bfloat162_rn(v[2 * i].x, v[2 * i].y);
                            __nv_bfloat162 q1 = __floats2bfloat162_rn(v[2 * i].z, v[2 * i].w);
                            __nv_bfloat162 q2 = __floats2bfloat162_rn(v[2 * i + 1].x, v[2 * i + 1].y);
                            __nv_bfloat162 q3 = __floats2bfloat162_rn(v[2 * i + 1].z, v[2 * i + 1].w);
                            uint4 pk;
                            pk.x = *reinterpret_cast<uint32_t *>(&q0); pk.y = *reinterpret_cast<uint32_t *>(&q1);
                            pk.z = *reinterpret_cast<uint32_t *>(&q2); pk.w = *reinterpret_cast<uint32_t *>(&q3);
                            *reinterpret_cast<uint4 *>(st + oct * (TC_BLOCK_M * 16) + row * 16) = pk;
                        }
                    }
                    tc::fence_proxy_async();
                    tc::mbar_arrive(full_bar + stage);
                    if (has_next) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) v[i] = vn[i];
                    }
                }
            }
        }
        if (MODE == TC_MODE_F16X3 && p.range_flag != nullptr && tc::f16x2_overflowed(hmax)) atomicOr(p.range_flag, 1);
    } else if (warp == 4) {
        // ================================ UMMA issuer ================================
        // the whole warp walks the stages, one ELECTED lane issues: descriptors stay in uniform registers (under
        // `if (lane == 0)` every UTCHMMA is wrapped in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop, see sa_fused_tc.cu)
        {
            const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_base_slot, 0);
            const uint32_t idesc = tc::instr_desc(MODE == TC_MODE_BF16 ? tc::FMT_BF16 : MODE == TC_MODE_F16X3 ? tc::FMT_F16 : tc::FMT_TF32,
                                                  TC_BLOCK_M, (uint32_t)n_blk);
            const uint32_t idesc16 = tc::instr_desc(tc::FMT_BF16, TC_BLOCK_M, (uint32_t)n_blk);      // MIXED: the correction products
            const uint32_t a_lbo = TC_BLOCK_M * 16, b_lbo = (uint32_t)n_blk * 16, sbo = 128;
            const bool swap = p.debug & 1;       // debug: exchange the roles of the two descriptor offsets
            auto desc = [&](uint32_t addr, uint32_t lbo) {
                return swap ? tc::smem_desc_kmajor(addr, sbo, lbo) : tc::smem_desc_kmajor(addr, lbo, sbo);
            };
            int stage = 0;
            uint32_t phase = 0, it = 0;
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
                const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
                tc::mbar_wait(acc_empty + acc, acc_phase ^ 1);
                tc::tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * TC_MAX_N;
                for (int kc = 0; kc < p.n_kc; ++kc) {
                    tc::mbar_wait(full_bar + stage, phase);
                    tc::tc_fence_after();
                    const uint32_t a0 = tc::smem_u32(ring + (size_t)stage * stage_bytes);
                    const uint32_t b0 = a0 + PARTS * A_PART;
                    if (tc::elect_one()) {
#pragma unroll
                    for (int j = 0; j < K_STEPS; ++j) {
                        const uint32_t a_off = (uint32_t)j * 2 * a_lbo, b_off = (uint32_t)j * 2 * b_lbo;
                        const uint32_t first = (kc > 0 || j > 0) ? 1u : 0u;
                        if (MODE == TC_MODE_TF32X3) {
                            const uint64_t a_hi = desc(a0 + a_off, a_lbo);
                            const uint64_t a_lo = desc(a0 + A_PART + a_off, a_lbo);
                            const uint64_t b_hi = desc(b0 + b_off, b_lbo);
                            const uint64_t b_lo = desc(b0 + b_part + b_off, b_lbo);
                            tc::umma_tf32(d_tmem, a_lo, b_hi, idesc, first);     // small terms first
                            tc::umma_tf32(d_tmem, a_hi, b_lo, idesc, 1u);
                            tc::umma_tf32(d_tmem, a_hi, b_hi, idesc, 1u);
                        } else if (MODE == TC_MODE_F16X3) {
                            const uint64_t a_hi = desc(a0 + a_off, a_lbo);
                            const uint64_t a_lo = desc(a0 + A_PART + a_off, a_lbo);
                            const uint64_t b_hi = desc(b0 + b_off, b_lbo);
                            const uint64_t b_lo = desc(b0 + b_part + b_off, b_lbo);
                            tc::umma_f16(d_tmem, a_lo, b_hi, idesc, first);      // small terms first
                            tc::umma_f16(d_tmem, a_hi, b_lo, idesc, 1u);
                            tc::umma_f16(d_tmem, a_hi, b_hi, idesc, 1u);
                        } else if (MODE == TC_MODE_MIXED) {
                            tc::umma_tf32(d_tmem, desc(a0 + a_off, a_lbo), desc(b0 + b_off, b_lbo), idesc, first);      // x_hi * w_hi
                        } else {
                            tc::umma_f16(d_tmem, desc(a0 + a_off, a_lbo), desc(b0 + b_off, b_lbo), idesc, first);
                        }
                    }
                    if (MODE == TC_MODE_MIXED) {
                        // the two correction products on the bf16 copies, 16 channels per UMMA: x_lo * w + x * w_lo
                        const uint32_t ax = a0 + A_PART, al = ax + A_PART / 2, bw = b0 + b_part, bl = bw + b_part / 2;
#pragma unroll
                        for (int j = 0; j < K_STEPS / 2; ++j) {
                            const uint32_t a_off = (uint32_t)j * 2 * a_lbo, b_off = (uint32_t)j * 2 * b_lbo;
                            tc::umma_f16(d_tmem, desc(al + a_off, a_lbo), desc(bw + b_off, b_lbo), idesc16, 1u);
                            tc::umma_f16(d_tmem, desc(ax + a_off, a_lbo), desc(bl + b_off, b_lbo), idesc16, 1u);
                        }
                    }
                    tc::umma_commit(empty_bar + stage);             // stage reusable once these UMMAs retire
                    }
                    __syncwarp();
                    if (++stage == stages) { stage = 0; phase ^= 1; }
                }
                if (tc::elect_one()) tc::umma_commit(acc_full + acc);                    // accumulator complete
                __syncwarp();
            }
        }
        __syncwarp();
    } else {
        // ================================ epilogue ================================
        const int q = warp;                            // TMEM lane quadrant of this warp
        const int r = q * 32 + lane;                   // row of the tile
        const int K = p.pool_rows;
        uint32_t it = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++it) {
            const uint32_t acc = it & 1, acc_phase = (it >> 1) & 1;
            const int64_t m0 = (tile / p.n_blocks) * TC_BLOCK_M;
            const int nb = (int)(tile % p.n_blocks);
            const int col0 = nb * n_blk;
            const int n_store = min(n_blk, p.n_store_total - col0);      // may be <= 0 for an all-padding block
            const bool row_ok = (m0 + r) < p.M;
            tc::mbar_wait(acc_full + acc, acc_phase);
            tc::tc_fence_after();
            const uint32_t t_addr = tmem_base + acc * TC_MAX_N + ((uint32_t)(q * 32) << 16);
            float *red_w = red + ((size_t)acc * 4 + q) * n_blk;
            for (int c0 = 0; c0 < n_blk; c0 += 32) {
                uint32_t raw[32];
                tc::tmem_ld32(t_addr + c0, raw);
                tc::tmem_ld_wait();
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float t = __uint_as_float(raw[j]) + bias_s[col0 + c0 + j];
                    v[j] = p.relu ? fmaxf(t, 0.f) : t;
                    if (post) v[j] = __fmaf_rn(v[j], post_a[col0 + c0 + j], post_b[col0 + c0 + j]);
                }
                if (K == 0) {
                    if (row_ok) {
                        float *yr = p.y + (m0 + r) * (int64_t)p.ld_y + p.y_col_off + col0 + c0;
                        const bool vec = (((p.ld_y | p.y_col_off) & 3) == 0) && ((uintptr_t)p.y & 15) == 0;
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            if (vec && c0 + j + 3 < n_store) {
                                *reinterpret_cast<float4 *>(yr + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
                            } else {
#pragma unroll
                                for (int u = 0; u < 4; ++u)
                                    if (c0 + j + u < n_store) yr[j + u] = v[j + u];
                            }
                        }
                    }
                } else {
                    // max over the 32 rows of this warp, column j ends up in lane j
                    float mine = 0.f;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const unsigned m = __reduce_max_sync(0xffffffffu, row_ok ? __float_as_uint(v[j]) : 0u);
                        if (lane == j) mine = __uint_as_float(m);
                    }
                    if (K == 32) {
                        const int64_t g = (m0 + q * 32) / 32;
                        if ((m0 + q * 32) < p.M && c0 + lane < n_store)
                            p.y[g * (int64_t)p.ld_y + p.y_col_off + col0 + c0 + lane] = mine;
                    } else {
                        if (c0 + lane < n_blk) red_w[c0 + lane] = mine;
                    }
                }
            }
            // accumulator drained: hand it back to the issuer
            tc::tc_fence_before();
            tc::mbar_arrive(acc_empty + acc);
            if (K > 32) {
                asm volatile("bar.sync 1, 128;" ::: "memory");            // the 4 epilogue warps only
                const float *ra = red + (size_t)acc * 4 * n_blk;
                if (K == 64) {
                    for (int i = tid; i < 2 * n_blk; i += 128) {
                        const int g = i / n_blk, c = i % n_blk;
                        const int64_t row0 = m0 + g * 64;
                        if (row0 < p.M && c < n_store)
                            p.y[(row0 / 64) * (int64_t)p.ld_y + p.y_col_off + col0 + c] =
                                fmaxf(ra[(2 * g) * n_blk + c], ra[(2 * g + 1) * n_blk + c]);
                    }
                } else {   // K is a multiple of 128: one group per tile (or a group spanning several tiles)
                    for (int c = tid; c < n_blk; c += 128) {
                        if (c >= n_store) continue;
                        const float m = fmaxf(fmaxf(ra[c], ra[n_blk + c]), fmaxf(ra[2 * n_blk + c], ra[3 * n_blk + c]));
                        float *dst = p.y + (m0 / K) * (int64_t)p.ld_y + p.y_col_off + col0 + c;
                        if (K == 128) *dst = m;
                        else atomicMax(reinterpret_cast<int *>(dst), __float_as_int(m));   // values are >= 0
                    }
                }
            }
        }
    }

    tc::tc_fence_before();
    __syncthreads();
    if (warp == 4) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
}

static int tc_n_blk(int Cout) { return Cout >= TC_MAX_N ? TC_MAX_N : round_up(Cout, 16); }
static int tc_n_blocks(int Cout) { return (Cout + tc_n_blk(Cout) - 1) / tc_n_blk(Cout); }
static int tc_n_kc(int Cin) { return (Cin + TC_KC - 1) / TC_KC; }

static int g_tc_debug = 0;
static bool tc_pool_supported(int K) { return K == 0 || K == 32 || K == 64 || (K % 128 == 0); }

}  // namespace ev2h

extern "C" int ev2h_tc_set_debug(int flags) { ev2h::g_tc_debug = flags; return 0; }

static int tc_n_blk_aligned(int Cout, int row_align) {
    const int n = ev2h::round_up(Cout, row_align);
    return n >= ev2h::TC_MAX_N ? ev2h::TC_MAX_N : n;
}

extern "C" int64_t ev2h_tc_packed_bytes_kc(int Cin, int Cout, int mode, int kc, int row_align) {
    using namespace ev2h;
    if (Cin <= 0 || Cout <= 0 || (mode < TC_MODE_BF16 || mode > TC_MODE_F16X3) || (kc != 16 && kc != 32) ||
        (row_align != 16 && row_align != 128)) return -1;
    const int n_blk = tc_n_blk_aligned(Cout, row_align);
    return (int64_t)((Cout + n_blk - 1) / n_blk) * ((Cin + kc - 1) / kc) * tc_parts(mode) * n_blk * kc * tc_elem_bytes(mode);
}
extern "C" int64_t ev2h_tc_packed_bytes(int Cin, int Cout, int mode) { return ev2h_tc_packed_bytes_kc(Cin, Cout, mode, ev2h::TC_KC, 16); }

extern "C" int ev2h_tc_pack_weights_kc(const float *wt, int ld_w, int Cin, int Cout, int mode, int kc, int row_align,
                                       void *packed, ev2h_stream_t stream);
extern "C" int ev2h_tc_pack_weights(const float *wt, int ld_w, int Cin, int Cout, int mode, void *packed,
                                    ev2h_stream_t stream) {
    return ev2h_tc_pack_weights_kc(wt, ld_w, Cin, Cout, mode, ev2h::TC_KC, 16, packed, stream);
}

extern "C" int ev2h_tc_pack_weights_kc(const float *wt, int ld_w, int Cin, int Cout, int mode, int kc, int row_align,
                                       void *packed, ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(kc == 16 || kc == 32, "ev2h_tc_pack_weights: K chunk must be 16 or 32");
    EV2H_REQUIRE(row_align == 16 || row_align == 128, "ev2h_tc_pack_weights: row_align must be 16 or 128");
    EV2H_REQUIRE(wt && packed, "ev2h_tc_pack_weights: null argument");
    EV2H_REQUIRE(Cin > 0 && Cout > 0 && ld_w >= Cout, "ev2h_tc_pack_weights: bad sizes");
    EV2H_REQUIRE(mode >= TC_MODE_BF16 && mode <= TC_MODE_F16X3, "ev2h_tc_pack_weights: unknown mode %d", mode);
    const int n_blk = tc_n_blk_aligned(Cout, row_align), n_blocks = (Cout + n_blk - 1) / n_blk, n_kc = (Cin + kc - 1) / kc;
    const int64_t total = (int64_t)n_blocks * n_kc * n_blk * kc;
    const unsigned grid = (unsigned)((total + 255) / 256);
    // wt comes from ev2h_fold_conv_bn_f32: round_up(Cin,16) rows of ld_w columns, zero padded
    const int cin_rows = round_up(Cin, 16);
    const int cout_cols = ld_w;
    if (mode == TC_MODE_BF16)
        tc_pack_kernel<TC_MODE_BF16><<<grid, 256, 0, as_stream(stream)>>>(wt, ld_w, cin_rows, cout_cols, n_blk, n_blocks, n_kc, kc, (uint8_t *)packed);
    else if (mode == TC_MODE_MIXED)
        tc_pack_kernel<TC_MODE_MIXED><<<grid, 256, 0, as_stream(stream)>>>(wt, ld_w, cin_rows, cout_cols, n_blk, n_blocks, n_kc, kc, (uint8_t *)packed);
    else if (mode == TC_MODE_F16X3)
        tc_pack_kernel<TC_MODE_F16X3><<<grid, 256, 0, as_stream(stream)>>>(wt, ld_w, cin_rows, cout_cols, n_blk, n_blocks, n_kc, kc, (uint8_t *)packed);
    else
        tc_pack_kernel<TC_MODE_TF32X3><<<grid, 256, 0, as_stream(stream)>>>(wt, ld_w, cin_rows, cout_cols, n_blk, n_blocks, n_kc, kc, (uint8_t *)packed);
    return check_launch("ev2h_tc_pack_weights");
}

static int linear_tc_impl(const float *x, int64_t M, int ld_x, int Cin, const void *w_packed, const float *bias, int Cout,
                          int pool_rows, float *y, int ld_y, int y_col_off, int mode, int relu, int32_t *range_flag,
                          ev2h_stream_t stream, int taps = 1, int rows_per_win = 0, const float *post_scale = nullptr,
                          const float *post_shift = nullptr);

extern "C" int ev2h_linear_relu_tc(const float *x, int64_t M, int ld_x, int Cin, const void *w_packed,
                                   const float *bias, int Cout, int pool_rows, float *y, int ld_y, int y_col_off,
                                   int mode, int32_t *range_flag, ev2h_stream_t stream) {
    return linear_tc_impl(x, M, ld_x, Cin, w_packed, bias, Cout, pool_rows, y, ld_y, y_col_off, mode, 1, range_flag, stream);
}

extern "C" int ev2h_linear_tc(const float *x, int64_t M, int ld_x, int Cin, const void *w_packed, const float *bias,
                              int Cout, float *y, int ld_y, int y_col_off, int mode, int32_t *range_flag, ev2h_stream_t stream) {
    return linear_tc_impl(x, M, ld_x, Cin, w_packed, bias, Cout, 0, y, ld_y, y_col_off, mode, 0, range_flag, stream);
}

extern "C" int ev2h_conv1d_tc(const float *x_rows, int64_t M, int ld_x, int Cin, int taps, int rows_per_seq, const void *w_packed,
                              const float *bias, int Cout, int relu, const float *post_scale, const float *post_shift,
                              float *y, int ld_y, int y_col_off, int mode, int32_t *range_flag, ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(taps == 1 || taps == 3 || taps == 5, "ev2h_conv1d_tc: kernel size %d (supported: 1, 3, 5)", taps);
    EV2H_REQUIRE(Cin > 0 && (taps == 1 || Cin % TC_KC == 0), "ev2h_conv1d_tc: Cin=%d must be a multiple of %d for kernel sizes > 1", Cin, TC_KC);
    EV2H_REQUIRE(rows_per_seq > 0 && M % rows_per_seq == 0, "ev2h_conv1d_tc: M must be a whole number of sequences");
    return linear_tc_impl(x_rows, M, ld_x, Cin * taps, w_packed, bias, Cout, 0, y, ld_y, y_col_off, mode, relu, range_flag, stream,
                          taps, rows_per_seq, post_scale, post_shift);
}

static int linear_tc_impl(const float *x, int64_t M, int ld_x, int Cin, const void *w_packed, const float *bias, int Cout,
                          int pool_rows, float *y, int ld_y, int y_col_off, int mode, int relu, int32_t *range_flag,
                          ev2h_stream_t stream, int taps, int rows_per_win, const float *post_scale, const float *post_shift) {
    using namespace ev2h;
    EV2H_REQUIRE(x && w_packed && bias && y, "ev2h_linear_relu_tc: null argument");
    EV2H_REQUIRE(M > 0 && Cin > 0 && Cout > 0, "ev2h_linear_relu_tc: bad sizes");
    EV2H_REQUIRE(mode >= TC_MODE_BF16 && mode <= TC_MODE_F16X3, "ev2h_linear_relu_tc: unknown mode %d", mode);
    EV2H_REQUIRE(ld_x % 4 == 0 && ld_x >= Cin / taps, "ev2h_linear_relu_tc: ld_x=%d must be a multiple of 4 and >= Cin=%d", ld_x, Cin / taps);
    EV2H_REQUIRE(((uintptr_t)x & 15) == 0 && ((uintptr_t)w_packed & 15) == 0, "ev2h_linear_relu_tc: x and w_packed must be 16-byte aligned");
    EV2H_REQUIRE(pool_rows >= 0 && (pool_rows == 0 || M % pool_rows == 0), "ev2h_linear_relu_tc: M must be a multiple of pool_rows");
    EV2H_REQUIRE(y_col_off >= 0 && ld_y >= y_col_off + Cout, "ev2h_linear_relu_tc: ld_y too small");
    if (!tc_pool_supported(pool_rows))
        return fail(EV2H_ERR_UNSUPPORTED, "ev2h_linear_relu_tc: pool_rows=%d (supported: 0, 32, 64, multiples of 128)", pool_rows);

    TcParams p;
    p.x = x; p.M = M; p.ld_x = ld_x; p.Cin = Cin;
    p.w_packed = (const uint8_t *)w_packed; p.bias = bias;
    p.n_blk = tc_n_blk(Cout); p.n_blocks = tc_n_blocks(Cout); p.n_kc = tc_n_kc(Cin);
    p.Cout = Cout; p.pool_rows = pool_rows; p.y = y; p.ld_y = ld_y; p.y_col_off = y_col_off;
    // bias comes from ev2h_fold_conv_bn_f32 (round_up(Cout,128) entries, zero padded) and must cover n_blocks*n_blk
    if (p.n_blocks * p.n_blk > round_up(Cout, 128))
        return fail(EV2H_ERR_UNSUPPORTED, "ev2h_linear_relu_tc: Cout=%d needs bias padding beyond round_up(Cout,128)", Cout);
    p.n_store_total = Cout;
    if (pool_rows == 0) {
        const int room = ld_y - y_col_off, padded = p.n_blocks * p.n_blk;
        p.n_store_total = room < padded ? room : padded;     // also write the exact-zero padding columns
    }
    const int stage_bytes = tc_stage_bytes(mode, p.n_blk);
    const int tail_bytes = (2 * TC_MAX_STAGES + 4) * 8 + 16 + (3 * p.n_blocks * p.n_blk + 2 * 4 * p.n_blk) * 4;
    int stages = (227 * 1024 - tail_bytes - 1024) / stage_bytes;
    if (stages > TC_MAX_STAGES) stages = TC_MAX_STAGES;
    stages -= stages % TC_LOADER_GROUPS;                     // a stage always belongs to the same loader group (see the loaders)
    if (stages < 2) return fail(EV2H_ERR_UNSUPPORTED, "ev2h_linear_relu_tc: stage of %d bytes does not fit twice", stage_bytes);
    p.stages = stages;
    p.debug = g_tc_debug;
    p.relu = relu;
    p.taps = taps; p.tap_cin = Cin / taps; p.rows_per_win = rows_per_win > 0 ? rows_per_win : 1;
    p.post_scale = post_scale; p.post_shift = post_shift;
    p.range_flag = mode == TC_MODE_F16X3 ? range_flag : nullptr;
    const size_t smem = (size_t)stages * stage_bytes + tail_bytes;

    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t n_tiles = ((M + TC_BLOCK_M - 1) / TC_BLOCK_M) * p.n_blocks;
    const unsigned grid = (unsigned)(n_tiles < sms ? n_tiles : sms);
    cudaError_t e;
    if (mode == TC_MODE_BF16) {
        e = cudaFuncSetAttribute(linear_tc_kernel<TC_MODE_BF16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) linear_tc_kernel<TC_MODE_BF16><<<grid, TC_THREADS, smem, as_stream(stream)>>>(p);
    } else if (mode == TC_MODE_MIXED) {
        e = cudaFuncSetAttribute(linear_tc_kernel<TC_MODE_MIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) linear_tc_kernel<TC_MODE_MIXED><<<grid, TC_THREADS, smem, as_stream(stream)>>>(p);
    } else if (mode == TC_MODE_F16X3) {
        e = cudaFuncSetAttribute(linear_tc_kernel<TC_MODE_F16X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) linear_tc_kernel<TC_MODE_F16X3><<<grid, TC_THREADS, smem, as_stream(stream)>>>(p);
    } else {
        e = cudaFuncSetAttribute(linear_tc_kernel<TC_MODE_TF32X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) linear_tc_kernel<TC_MODE_TF32X3><<<grid, TC_THREADS, smem, as_stream(stream)>>>(p);
    }
    if (e != cudaSuccess) return fail(EV2H_ERR_CUDA, "ev2h_linear_relu_tc: smem attribute (%zu bytes): %s", smem, cudaGetErrorString(e));
    return check_launch("ev2h_linear_relu_tc");
}
