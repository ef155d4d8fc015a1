// residual.cu — DeepCrossing: gather + concat + N residual units, forward and backward.
//   residual_unit: relu(x + W2 relu(W1 x + b1) + b2)   (DeepCrossing/deepcrossing.py:25-42,157-159)
// W1/W2 are nn.Linear layers created inside every call and never registered
// (DeepCrossing/deepcrossing.py:37,39), so only d(out)/d(x) is observable.
//
// One CTA owns a tile of samples (64, or 32 for wide hidden layers); activations stay in shared
// memory, feature-major, across all units; each unit's two GEMMs run on tile_gemm.cuh with the
// unit's weights staged in shared memory.  The forward keeps the units' inputs/outputs
// (nets[0..N], [B,d] each) for the backward, which recomputes the hidden layer instead of
// storing it.  Packed per-unit weights (rk_resunit_pack_floats), Hp = roundup(H,8), dp = roundup(d,4):
//   [W1^T d x Hp][b1 Hp][W2^T Hp x dp][b2 dp][W2 d x Hp][W1 Hp x dp]      (zero padded)
// Every block must fit the 227 KiB of shared memory a block may have; that, not d, H <= 256 alone,
// bounds the widths.  The backward takes every (d, H) the forward takes: it stages W1 over W1^T | b1
// once the hidden layer has been recomputed, and halves its tile height where the block would not fit.
#include <string.h>
#include "common.cuh"
#include "tile_gemm.cuh"

namespace rk {

constexpr int kResThreads = 256;

struct ResLayout {
    int d, H, dp, Hp, w1t, b1, w2t, b2, w2, w1, total;
    __host__ __device__ ResLayout(int d_, int H_) : d(d_), H(H_) {
        dp = (d + 3) / 4 * 4;
        Hp = (H + 7) / 8 * 8;
        w1t = 0;
        b1  = w1t + d * Hp;
        w2t = b1 + Hp;
        b2  = w2t + Hp * dp;
        w2  = b2 + dp;
        w1  = w2 + d * Hp;
        total = w1 + Hp * dp;
    }
};

struct ResParams {
    FieldSet     fs;
    const float* dense;
    const float* units;      // n_units packed blocks
    int32_t      n_dense, d, H, n_units, rows;   // rows = samples per tile
    int64_t      B;
};

__device__ __forceinline__ void res_copy(float* dst, const float* __restrict__ src, int n) {
    for (int i = threadIdx.x; i < n; i += kResThreads) dst[i] = __ldg(src + i);
}

__global__ void __launch_bounds__(kResThreads)
resunits_fwd_kernel(const __grid_constant__ ResParams p, float* __restrict__ nets, int32_t* err_flag) {
    extern __shared__ __align__(16) float smem_raw[];
    const ResLayout L(p.d, p.H);
    const int R = p.rows, ld = R + 4, d = p.d;
    float* W  = smem_raw;                       // w1t | b1 | w2t | b2 of the current unit
    float* X  = W + (L.w2);                     // [dp][ld]
    float* Hs = X + L.dp * ld;                  // [Hp][ld]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b0 = (int64_t)blockIdx.x * R;
    const int ns = (int)((p.B - b0) < R ? (p.B - b0) : R);

    // gather + concat: one warp per sample, lanes over the columns
    for (int i = tid; i < L.dp * ld; i += kResThreads) X[i] = 0.f;
    __syncthreads();
    for (int s = warp; s < ns; s += kResThreads / 32) {
        const int64_t b = b0 + s;
        for (int c = lane; c < d; c += 32) {
            float v = 0.f;
            if (c < p.n_dense) {
                v = __ldg(p.dense + b * p.n_dense + c);
            } else {
                for (int f = 0; f < p.fs.F; ++f)
                    if (c >= p.fs.off[f] && c < p.fs.off[f] + p.fs.dim[f]) {
                        const int64_t row = checked_row(__ldg(p.fs.idx[f] + b), p.fs.rows[f], err_flag);
                        v = __ldg(p.fs.weight[f] + row * p.fs.dim[f] + c - p.fs.off[f]);
                    }
            }
            X[c * ld + s] = v;
            nets[b * d + c] = v;
        }
    }
    __syncthreads();
    for (int u = 0; u < p.n_units; ++u) {
        res_copy(W, p.units + (int64_t)u * L.total, L.w2);
        __syncthreads();
        const float* b1 = W + L.b1;
        const float* b2 = W + L.b2;
        tile_gemm<8, kResThreads>(X, ld, W + L.w1t, L.Hp, d, L.Hp, R, [&](int m0, int n0, float (&acc)[4][8]) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i][j] = fmaxf(acc[i][j] + b1[n0 + j], 0.f);
            store_tile_kmajor<8>(Hs, ld, m0, n0, acc);
        });
        __syncthreads();
        tile_gemm<4, kResThreads>(Hs, ld, W + L.w2t, L.dp, L.Hp, L.dp, R, [&](int m0, int n0, float (&acc)[4][4]) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 x = *reinterpret_cast<const float4*>(X + (n0 + j) * ld + m0);
                const float bb = b2[n0 + j];
                acc[0][j] = fmaxf(x.x + acc[0][j] + bb, 0.f);
                acc[1][j] = fmaxf(x.y + acc[1][j] + bb, 0.f);
                acc[2][j] = fmaxf(x.z + acc[2][j] + bb, 0.f);
                acc[3][j] = fmaxf(x.w + acc[3][j] + bb, 0.f);
            }
            store_tile_kmajor<4>(X, ld, m0, n0, acc);
        });
        __syncthreads();
        float* out = nets + (int64_t)(u + 1) * p.B * d;
        for (int item = tid; item < ns * d; item += kResThreads) {
            const int s = item / d, c = item - s * d;
            out[(b0 + s) * d + c] = X[c * ld + s];
        }
        __syncthreads();
    }
}

// Backward weights: W1^T | b1, later W1 in the same space, then W2.
__host__ __device__ inline int res_bwd_w1_floats(const ResLayout& L) {
    return L.d * L.Hp + L.Hp > L.Hp * L.dp ? L.d * L.Hp + L.Hp : L.Hp * L.dp;
}

__global__ void __launch_bounds__(kResThreads)
resunits_bwd_kernel(const float* __restrict__ nets, const float* __restrict__ units, int n_units, int H, int d,
                    int rows, int64_t B, const float* __restrict__ g_out, float* __restrict__ g_x0) {
    extern __shared__ __align__(16) float smem_raw[];
    const ResLayout L(d, H);
    const int R = rows, ld = R + 4;
    float* W1t = smem_raw;                    // [d][Hp]
    float* b1  = W1t + d * L.Hp;              // [Hp]
    float* W1  = smem_raw;                    // [Hp][dp] (as registered: B operand of gh x W1), over W1t | b1
    float* W2  = smem_raw + res_bwd_w1_floats(L);   // [d][Hp]  (as registered: B operand of gz x W2)
    float* X   = W2 + d * L.Hp;               // [dp][ld]
    float* G   = X + L.dp * ld;               // [dp][ld]
    float* Hs  = G + L.dp * ld;               // [Hp][ld]
    const int tid = threadIdx.x;
    const int64_t b0 = (int64_t)blockIdx.x * R;
    const int ns = (int)((B - b0) < R ? (B - b0) : R);

    for (int i = tid; i < L.dp * ld; i += kResThreads) { X[i] = 0.f; G[i] = 0.f; }
    __syncthreads();
    for (int item = tid; item < ns * d; item += kResThreads) {
        const int s = item / d, c = item - s * d;
        G[c * ld + s] = g_out[(b0 + s) * d + c];
    }
    for (int u = n_units - 1; u >= 0; --u) {
        const float* pack = units + (int64_t)u * L.total;
        res_copy(W1t, pack + L.w1t, d * L.Hp);
        res_copy(b1, pack + L.b1, L.Hp);
        res_copy(W2, pack + L.w2, d * L.Hp);
        __syncthreads();   // also orders the previous unit's G writes before the reads below
        const float* xin  = nets + (int64_t)u * B * d;
        const float* xout = nets + (int64_t)(u + 1) * B * d;
        for (int item = tid; item < ns * d; item += kResThreads) {
            const int s = item / d, c = item - s * d;
            X[c * ld + s] = xin[(b0 + s) * d + c];
            if (!(xout[(b0 + s) * d + c] > 0.f)) G[c * ld + s] = 0.f;      // outer ReLU
        }
        __syncthreads();
        tile_gemm<8, kResThreads>(X, ld, W1t, L.Hp, d, L.Hp, R, [&](int m0, int n0, float (&acc)[4][8]) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[i][j] = fmaxf(acc[i][j] + b1[n0 + j], 0.f);
            store_tile_kmajor<8>(Hs, ld, m0, n0, acc);
        });
        __syncthreads();
        res_copy(W1, pack + L.w1, L.Hp * L.dp);   // W1^T and b1 are dead from here on
        // gh = (gz x W2) masked by the hidden ReLU, in place over Hs
        tile_gemm<8, kResThreads>(G, ld, W2, L.Hp, d, L.Hp, R, [&](int m0, int n0, float (&acc)[4][8]) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float4 h = *reinterpret_cast<const float4*>(Hs + (n0 + j) * ld + m0);
                acc[0][j] = h.x > 0.f ? acc[0][j] : 0.f;
                acc[1][j] = h.y > 0.f ? acc[1][j] : 0.f;
                acc[2][j] = h.z > 0.f ? acc[2][j] : 0.f;
                acc[3][j] = h.w > 0.f ? acc[3][j] : 0.f;
            }
            store_tile_kmajor<8>(Hs, ld, m0, n0, acc);
        });
        __syncthreads();
        // g_x = gz + gh x W1, in place over G
        tile_gemm<4, kResThreads>(Hs, ld, W1, L.dp, L.Hp, L.dp, R, [&](int m0, int n0, float (&acc)[4][4]) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float4 g = *reinterpret_cast<const float4*>(G + (n0 + j) * ld + m0);
                acc[0][j] += g.x; acc[1][j] += g.y; acc[2][j] += g.z; acc[3][j] += g.w;
            }
            store_tile_kmajor<4>(G, ld, m0, n0, acc);
        });
        __syncthreads();
    }
    for (int item = tid; item < ns * d; item += kResThreads) {
        const int s = item / d, c = item - s * d;
        g_x0[(b0 + s) * d + c] = G[c * ld + s];
    }
}

constexpr size_t kResSmemMax = 227 * 1024;   // dynamic shared memory a block may have

static int res_rows(int H) { return H > 128 ? 32 : 64; }

static size_t res_fwd_smem(const ResLayout& L, int rows) {
    return sizeof(float) * ((size_t)L.w2 + (size_t)(L.dp + L.Hp) * (rows + 4));
}

static size_t res_bwd_smem(const ResLayout& L, int rows) {
    return sizeof(float) * ((size_t)res_bwd_w1_floats(L) + (size_t)L.d * L.Hp + (size_t)(2 * L.dp + L.Hp) * (rows + 4));
}

}  // namespace rk

extern "C" {

int rk_resunit_pack_floats(int d, int H) { return rk::ResLayout(d, H).total; }

int rk_resunits_fwd(const rk_field_t* fields, int F, const float* dense, int n_dense, const float* units,
                    int n_units, int H, int64_t B, float* nets, int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    ResParams p;
    memset(&p, 0, sizeof(p));
    if (int rc = pack_fields(fields, F, &p.fs)) return rc;
    RK_CHECK_ARG(n_dense >= 0 && (n_dense == 0 || dense), "resunits: dense is NULL");
    int d = n_dense;
    for (int f = 0; f < F; ++f) {
        RK_CHECK_ARG(fields[f].out_off >= n_dense, "resunits: field %d overlaps the dense block", f);
        if (fields[f].out_off + fields[f].dim > d) d = fields[f].out_off + fields[f].dim;
    }
    int covered = n_dense;
    for (int f = 0; f < F; ++f) covered += fields[f].dim;
    RK_CHECK_ARG(covered == d, "resunits: the fields do not tile the %d-wide row", d);
    RK_CHECK_ARG(d >= 1 && d <= 256 && H >= 1 && H <= 256 && n_units >= 0,
                 "resunits: d=%d H=%d units=%d (d and H must lie in [1, 256], units >= 0)", d, H, n_units);
    RK_CHECK_ARG(nets && (n_units == 0 || units), "resunits: NULL pointer");
    if (B == 0) return 0;
    p.dense = dense; p.units = units; p.n_dense = n_dense; p.d = d; p.H = H; p.n_units = n_units;
    p.rows = res_rows(H); p.B = B;
    const ResLayout L(d, H);
    const size_t smem = res_fwd_smem(L, p.rows);
    RK_CHECK_ARG(smem <= kResSmemMax, "resunits_fwd: d=%d H=%d needs %zu bytes of shared memory, a block may have %zu",
                 d, H, smem, kResSmemMax);
    RK_CUDA(cudaFuncSetAttribute(resunits_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    resunits_fwd_kernel<<<(int)ceil_div(B, p.rows), kResThreads, smem, (cudaStream_t)stream_>>>(p, nets, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}

int rk_resunits_bwd(const float* nets, const float* units, int n_units, int H, int d, int64_t B,
                    const float* g_out, float* g_x0, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(nets && g_out && g_x0 && (n_units == 0 || units), "resunits_bwd: NULL pointer");
    RK_CHECK_ARG(d >= 1 && d <= 256 && H >= 1 && H <= 256 && n_units >= 0,
                 "resunits_bwd: d=%d H=%d units=%d (d and H must lie in [1, 256], units >= 0)", d, H, n_units);
    if (B == 0) return 0;
    const ResLayout L(d, H);
    int rows = res_rows(H);
    while (rows > 4 && res_bwd_smem(L, rows) > kResSmemMax) rows >>= 1;
    const size_t smem = res_bwd_smem(L, rows);
    RK_CHECK_ARG(smem <= kResSmemMax, "resunits_bwd: d=%d H=%d needs %zu bytes of shared memory, a block may have %zu",
                 d, H, smem, kResSmemMax);
    RK_CUDA(cudaFuncSetAttribute(resunits_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    resunits_bwd_kernel<<<(int)ceil_div(B, rows), kResThreads, smem, (cudaStream_t)stream_>>>(
        nets, units, n_units, H, d, rows, B, g_out, g_x0);
    RK_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
