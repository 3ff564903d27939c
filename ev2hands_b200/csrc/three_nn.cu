// Feature propagation, geometric half: three nearest sources with inverse-distance weights, and the
// weighted interpolation of their features.
//
// Replaces, in PointNetFeaturePropagation.forward (reference
// src/Ev2Hands/model/pointnet2_utils.py:294-301), square_distance + a FULL sort of every [S] row +
// index_points + the weighted sum.  One thread per query point keeps the three smallest distances while
// scanning the sources in index order (ties keep the lower index, like the reference's sort on these
// inputs), so the [B,N,S] distance matrix and the sort never exist.
#include "common.cuh"
#include "geom.cuh"

namespace ev2h {

constexpr int kNnThreads = 128;
constexpr int kNnTile = 1024;     // sources staged per pass (16 KB of float4)

__global__ void __launch_bounds__(kNnThreads)
three_nn_kernel(const float *__restrict__ q, int64_t qb, int64_t qc, int64_t qn_,
                const float *__restrict__ src, int64_t sb, int64_t sc, int64_t sn,
                int N, int S, int32_t *__restrict__ idx, float *__restrict__ weight) {
    __shared__ float4 pts[kNnTile];
    const int b = blockIdx.y;
    const int n = blockIdx.x * kNnThreads + threadIdx.x;
    const bool live = n < N;
    float qx = 0.f, qy = 0.f, qz = 0.f;
    if (live) {
        const float *p = q + (int64_t)b * qb + (int64_t)n * qn_;
        qx = p[0]; qy = p[qc]; qz = p[2 * qc];
    }
    const float qq = sq_norm3(qx, qy, qz);
    float d0 = INFINITY, d1 = INFINITY, d2 = INFINITY;
    int i0 = 0, i1 = 0, i2 = 0;
    const float *sbase = src + (int64_t)b * sb;
    for (int t0 = 0; t0 < S; t0 += kNnTile) {
        const int cnt = min(kNnTile, S - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < cnt; i += kNnThreads) {
            const float *p = sbase + (int64_t)(t0 + i) * sn;
            const float x = p[0], y = p[sc], z = p[2 * sc];
            pts[i] = make_float4(x, y, z, sq_norm3(x, y, z));
        }
        __syncthreads();
        if (!live) continue;
        for (int i = 0; i < cnt; ++i) {
            const float d = sqdist_expanded(qx, qy, qz, qq, pts[i]);
            if (d < d2) {                       // strict: an equal distance later in index order stays behind
                const int j = t0 + i;
                if (d < d1) {
                    d2 = d1; i2 = i1;
                    if (d < d0) { d1 = d0; i1 = i0; d0 = d; i0 = j; }
                    else { d1 = d; i1 = j; }
                } else { d2 = d; i2 = j; }
            }
        }
    }
    if (!live) return;
    // dist_recip = 1 / (d + 1e-8); norm = sum over the three; weight = dist_recip / norm   (:298-300)
    const float r0 = __fdiv_rn(1.0f, __fadd_rn(d0, 1e-8f)), r1 = __fdiv_rn(1.0f, __fadd_rn(d1, 1e-8f)),
                r2 = __fdiv_rn(1.0f, __fadd_rn(d2, 1e-8f));
    const float norm = __fadd_rn(__fadd_rn(r0, r1), r2);
    const int64_t o = ((int64_t)b * N + n) * 3;
    idx[o] = i0; idx[o + 1] = i1; idx[o + 2] = i2;
    weight[o] = __fdiv_rn(r0, norm); weight[o + 1] = __fdiv_rn(r1, norm); weight[o + 2] = __fdiv_rn(r2, norm);
}

// out[b, n, col + c] = (f[i0] * w0 + f[i1] * w1) + f[i2] * w2, products and sums rounded separately like the
// reference's  torch.sum(index_points(points2, idx) * weight, dim=2)  (:301).  One thread per 4 channels.
__global__ void __launch_bounds__(256)
three_interp_kernel(const float *__restrict__ feats, int ld_f, const int32_t *__restrict__ idx, const float *__restrict__ weight,
                    int64_t rows, int N, int S, int D, float *__restrict__ out, int ld_out, int col) {
    const int quads = (D + 3) / 4;
    const int64_t total = rows * quads;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / quads;
        const int c = (int)(e - r * quads) * 4;
        const int64_t b = r / N;
        const int32_t *id = idx + r * 3;
        const float *w = weight + r * 3;
        const float w0 = w[0], w1 = w[1], w2 = w[2];
        const float *f0 = feats + (b * S + id[0]) * (int64_t)ld_f + c, *f1 = feats + (b * S + id[1]) * (int64_t)ld_f + c,
                    *f2 = feats + (b * S + id[2]) * (int64_t)ld_f + c;
        float *o = out + r * (int64_t)ld_out + col + c;
        if (c + 3 < D && (ld_f & 3) == 0 && ((ld_out | col) & 3) == 0 && (((uintptr_t)feats | (uintptr_t)out) & 15) == 0) {
            const float4 a = *reinterpret_cast<const float4 *>(f0), bb = *reinterpret_cast<const float4 *>(f1),
                         cc = *reinterpret_cast<const float4 *>(f2);
            float4 v;
            v.x = __fadd_rn(__fadd_rn(__fmul_rn(a.x, w0), __fmul_rn(bb.x, w1)), __fmul_rn(cc.x, w2));
            v.y = __fadd_rn(__fadd_rn(__fmul_rn(a.y, w0), __fmul_rn(bb.y, w1)), __fmul_rn(cc.y, w2));
            v.z = __fadd_rn(__fadd_rn(__fmul_rn(a.z, w0), __fmul_rn(bb.z, w1)), __fmul_rn(cc.z, w2));
            v.w = __fadd_rn(__fadd_rn(__fmul_rn(a.w, w0), __fmul_rn(bb.w, w1)), __fmul_rn(cc.w, w2));
            *reinterpret_cast<float4 *>(o) = v;
        } else {
            for (int k = 0; k < 4 && c + k < D; ++k)
                o[k] = __fadd_rn(__fadd_rn(__fmul_rn(f0[k], w0), __fmul_rn(f1[k], w1)), __fmul_rn(f2[k], w2));
        }
    }
}

}  // namespace ev2h

extern "C" int ev2h_three_nn_f32(const float *xyz1, int64_t q_stride_b, int64_t q_stride_c, int64_t q_stride_n,
                                 const float *xyz2, int64_t s_stride_b, int64_t s_stride_c, int64_t s_stride_n,
                                 int B, int N, int S, int32_t *idx, float *weight, ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(xyz1 && xyz2 && idx && weight, "ev2h_three_nn_f32: null argument");
    EV2H_REQUIRE(B > 0 && N > 0, "ev2h_three_nn_f32: bad sizes");
    if (S < 3) return fail(EV2H_ERR_UNSUPPORTED, "ev2h_three_nn_f32: needs at least 3 source points, got %d", S);
    dim3 grid((unsigned)((N + kNnThreads - 1) / kNnThreads), (unsigned)B);
    three_nn_kernel<<<grid, kNnThreads, 0, as_stream(stream)>>>(xyz1, q_stride_b, q_stride_c, q_stride_n, xyz2, s_stride_b,
                                                                s_stride_c, s_stride_n, N, S, idx, weight);
    return check_launch("ev2h_three_nn_f32");
}

extern "C" int ev2h_three_interp_f32(const float *feats_rows, int ld_f, const int32_t *idx, const float *weight,
                                     int B, int N, int S, int D, float *out_rows, int ld_out, int col,
                                     ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(feats_rows && idx && weight && out_rows, "ev2h_three_interp_f32: null argument");
    EV2H_REQUIRE(B > 0 && N > 0 && S > 0 && D > 0 && ld_f >= D && col >= 0 && ld_out >= col + D, "ev2h_three_interp_f32: bad sizes");
    const int64_t rows = (int64_t)B * N, total = rows * ((D + 3) / 4);
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int64_t want = (total + 255) / 256, cap = (int64_t)sms * 16;
    three_interp_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, as_stream(stream)>>>(feats_rows, ld_f, idx, weight, rows, N, S, D,
                                                                                             out_rows, ld_out, col);
    return check_launch("ev2h_three_interp_f32");
}
