// Shared-MLP layer on the CUDA cores in exact fp32 (FFMA): y = relu(x W' + b'),
// optionally max-pooled over runs of K consecutive rows.
//
// Replaces one Conv2d(1x1) + BatchNorm2d(eval) + ReLU step of the reference MLP
// (src/Ev2Hands/model/pointnet2_utils.py:253-256 / :193-197) and, when pooling,
// the torch.max over the neighbour axis (:257 / :199).
//
// This is the fp32-exact path: it is the parity anchor for the tensor-core
// kernels and the fallback for layer shapes they do not cover.  Classic
// 128x128x16 register-tiled SGEMM, 256 threads, 8x8 outputs per thread,
// shared-memory double buffering with register prefetch.  x tiles are stored
// k-major in shared memory so both operands are read as conflict-free LDS.128.
#include "common.cuh"

namespace ev2h {

constexpr int BM = 128, BN = 128, BK = 16, LIN_THREADS = 256;

__device__ __forceinline__ void atomic_max_nonneg(float *addr, float v) {
    // valid for v >= 0 and *addr >= 0: the int ordering of the bit patterns is the float ordering
    atomicMax(reinterpret_cast<int *>(addr), __float_as_int(v));
}

// x[k .. k+3] with the channels from Cin on zeroed: columns Cin .. ld_x - 1 are padding and must not enter the product
// (a NaN or Inf there would survive the zero weight rows), whatever they hold
__device__ __forceinline__ float4 tail_masked(float4 v, int k, int Cin) {
    if (k + 4 > Cin) {
        if (k + 1 >= Cin) v.y = 0.f;
        if (k + 2 >= Cin) v.z = 0.f;
        if (k + 3 >= Cin) v.w = 0.f;
    }
    return v;
}

__global__ void __launch_bounds__(LIN_THREADS, 2)
linear_relu_kernel(const float *__restrict__ x, int64_t M, int ld_x, int Cin,
                   const float *__restrict__ wt, int ld_w, const float *__restrict__ bias,
                   int n_store, int pool_rows, float *__restrict__ y, int ld_y, int y_col_off,
                   int n_col_blocks, int relu) {
    __shared__ __align__(16) float Xs[2][BK][BM];
    __shared__ __align__(16) float Ws[2][BK][BN];

    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    // column blocks of one row tile are neighbours in launch order, so the x tile they share
    // is still in L2 when the second one asks for it
    const int n0 = (int)(blockIdx.x % n_col_blocks) * BN;
    const int64_t m0 = (int64_t)(blockIdx.x / n_col_blocks) * BM;

    // global -> register staging assignments
    const int xr = tid & 127, xq = tid >> 7;            // x: row xr, float4 #xq and #xq+2 of the 16-wide k slab
    const int wk = tid >> 5, wc = (tid & 31) * 4;       // w: rows wk and wk+8, 4 columns at wc
    const bool x_row_ok = (m0 + xr) < M;
    const float *x_row = x + (m0 + xr) * (int64_t)ld_x;

    float4 xa, xb, wa, wb;
    auto load_tiles = [&](int k0) {
        xa = xb = make_float4(0.f, 0.f, 0.f, 0.f);
        const int ka = k0 + 4 * xq, kb = k0 + 4 * (xq + 2);
        if (x_row_ok && ka < Cin) xa = tail_masked(*reinterpret_cast<const float4 *>(x_row + ka), ka, Cin);
        if (x_row_ok && kb < Cin) xb = tail_masked(*reinterpret_cast<const float4 *>(x_row + kb), kb, Cin);
        wa = *reinterpret_cast<const float4 *>(wt + (int64_t)(k0 + wk) * ld_w + n0 + wc);
        wb = *reinterpret_cast<const float4 *>(wt + (int64_t)(k0 + wk + 8) * ld_w + n0 + wc);
    };
    auto store_tiles = [&](int buf) {
        Xs[buf][4 * xq + 0][xr] = xa.x; Xs[buf][4 * xq + 1][xr] = xa.y;
        Xs[buf][4 * xq + 2][xr] = xa.z; Xs[buf][4 * xq + 3][xr] = xa.w;
        Xs[buf][4 * xq + 8][xr] = xb.x; Xs[buf][4 * xq + 9][xr] = xb.y;
        Xs[buf][4 * xq + 10][xr] = xb.z; Xs[buf][4 * xq + 11][xr] = xb.w;
        *reinterpret_cast<float4 *>(&Ws[buf][wk][wc]) = wa;
        *reinterpret_cast<float4 *>(&Ws[buf][wk + 8][wc]) = wb;
    };

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    const int n_k = (Cin + BK - 1) / BK;     // wt is zero padded to a multiple of 16 rows
    load_tiles(0);
    store_tiles(0);
    __syncthreads();
    for (int kt = 0; kt < n_k; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < n_k) load_tiles((kt + 1) * BK);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&Xs[buf][k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&Xs[buf][k][64 + ty * 4]);
            const float4 b0 = *reinterpret_cast<const float4 *>(&Ws[buf][k][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4 *>(&Ws[buf][k][64 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        if (kt + 1 < n_k) {
            store_tiles(buf ^ 1);
            __syncthreads();
        }
    }

    // epilogue: + b', ReLU
    float bj[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) bj[j] = bias[n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4))];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = relu ? fmaxf(acc[i][j] + bj[j], 0.f) : acc[i][j] + bj[j];

    if (pool_rows == 0) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int64_t m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
            if (m >= M) continue;
            float *yr = y + m * (int64_t)ld_y + y_col_off;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int n = n0 + h * 64 + tx * 4;
                if (n + 3 < n_store && ((ld_y | y_col_off) & 3) == 0 && ((uintptr_t)y & 15) == 0) {
                    *reinterpret_cast<float4 *>(yr + n) =
                        make_float4(acc[i][4 * h], acc[i][4 * h + 1], acc[i][4 * h + 2], acc[i][4 * h + 3]);
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (n + j < n_store) yr[n + j] = acc[i][4 * h + j];
                }
            }
        }
        return;
    }

    // pooled epilogue: max over runs of pool_rows consecutive rows.
    const int K = pool_rows;
    const bool aligned = (K % 4 == 0) && ((BM % K == 0) || (K % BM == 0));
    if (aligned) {
        // rows of one 4-row bundle share a group; reduce bundles through shared memory first
        __syncthreads();
        float *red = &Xs[0][0][0];                      // [groups_in_tile <= 32][BN] floats, 16 KB available
        const int groups = K >= BM ? 1 : BM / K;
        for (int i = tid; i < groups * BN; i += LIN_THREADS) red[i] = 0.f;
        __syncthreads();
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int r = h * 64 + ty * 4;              // first row of the bundle inside the tile
            const int g = K >= BM ? 0 : r / K;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                float m = 0.f;
#pragma unroll
                for (int i = 0; i < 4; ++i)
                    if (m0 + r + i < M) m = fmaxf(m, acc[4 * h + i][j]);
                const int n = j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4);
                atomic_max_nonneg(&red[g * BN + n], m);
            }
        }
        __syncthreads();
        for (int i = tid; i < groups * BN; i += LIN_THREADS) {
            const int g = i / BN, n = n0 + (i % BN);
            const int64_t first_row = m0 + (int64_t)g * (K >= BM ? BM : K);
            if (n >= n_store || first_row >= M) continue;
            float *dst = y + (first_row / K) * (int64_t)ld_y + y_col_off + n;
            if (K > BM) atomic_max_nonneg(dst, red[i]);   // group spans several tiles
            else *dst = red[i];
        }
        return;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (m >= M) continue;
        float *yr = y + (m / K) * (int64_t)ld_y + y_col_off;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
            if (n < n_store) atomic_max_nonneg(yr + n, acc[i][j]);
        }
    }
}

}  // namespace ev2h

static int linear_f32_impl(const float *x, int64_t M, int ld_x, int Cin, const float *wt, const float *bias, int Cout,
                           int pool_rows, float *y, int ld_y, int y_col_off, int relu, ev2h_stream_t stream);

extern "C" int ev2h_linear_relu_f32(const float *x, int64_t M, int ld_x, int Cin, const float *wt,
                                    const float *bias, int Cout, int pool_rows, float *y, int ld_y,
                                    int y_col_off, ev2h_stream_t stream) {
    return linear_f32_impl(x, M, ld_x, Cin, wt, bias, Cout, pool_rows, y, ld_y, y_col_off, 1, stream);
}

extern "C" int ev2h_linear_f32(const float *x, int64_t M, int ld_x, int Cin, const float *wt, const float *bias,
                               int Cout, float *y, int ld_y, int y_col_off, ev2h_stream_t stream) {
    return linear_f32_impl(x, M, ld_x, Cin, wt, bias, Cout, 0, y, ld_y, y_col_off, 0, stream);
}

static int linear_f32_impl(const float *x, int64_t M, int ld_x, int Cin, const float *wt, const float *bias, int Cout,
                           int pool_rows, float *y, int ld_y, int y_col_off, int relu, ev2h_stream_t stream) {
    using namespace ev2h;
    EV2H_REQUIRE(x && wt && bias && y, "ev2h_linear_relu_f32: null argument");
    EV2H_REQUIRE(M > 0 && Cin > 0 && Cout > 0, "ev2h_linear_relu_f32: bad sizes");
    EV2H_REQUIRE(ld_x % 4 == 0 && ld_x >= Cin, "ev2h_linear_relu_f32: ld_x=%d must be a multiple of 4 and >= Cin=%d", ld_x, Cin);
    EV2H_REQUIRE(((uintptr_t)x & 15) == 0 && ((uintptr_t)wt & 15) == 0, "ev2h_linear_relu_f32: x and wt must be 16-byte aligned");
    EV2H_REQUIRE(pool_rows >= 0 && (pool_rows == 0 || M % pool_rows == 0), "ev2h_linear_relu_f32: M must be a multiple of pool_rows");
    EV2H_REQUIRE(y_col_off >= 0 && ld_y >= y_col_off + Cout, "ev2h_linear_relu_f32: ld_y too small");
    const int cout_pad = round_up(Cout, BN);
    // Without pooling, columns [Cout, min(Cout_pad, ld_y - off)) are written too: they are exact zeros
    // (zero weights, zero bias) and keep the padding of the next layer's input finite.
    int n_store = Cout;
    if (pool_rows == 0) n_store = (ld_y - y_col_off) < cout_pad ? (ld_y - y_col_off) : cout_pad;
    const int64_t tiles_m = (M + BM - 1) / BM;
    const int n_col_blocks = cout_pad / BN;
    if (tiles_m * n_col_blocks > 0x7fffffffLL)
        return fail(EV2H_ERR_UNSUPPORTED, "ev2h_linear_relu_f32: M=%lld is too large for one launch; split the call", (long long)M);
    dim3 grid((unsigned)(tiles_m * n_col_blocks));
    linear_relu_kernel<<<grid, LIN_THREADS, 0, as_stream(stream)>>>(x, M, ld_x, Cin, wt, cout_pad, bias, n_store,
                                                                    pool_rows, y, ld_y, y_col_off, n_col_blocks, relu);
    return check_launch("ev2h_linear_relu_f32");
}
