// linear.cu — weight and bias gradients of the towers' nn.Linear layers.
//
//   dW[N, K] = G^T X = sum_b G[b, :]^T X[b, :]        db[N] = sum_b G[b, :]
//
// Both are one reduction over the batch, and both operands are row-major [B, *], so every batch row
// contributes a contiguous piece of a G row and of an X row.  The grid is (K tiles) x (N tiles) x
// (S batch slabs): a CTA owns a 64 x 64 tile of dW and the rows of one slab, and S is chosen from the
// shape so that the grid fills the GPU even where there are only a handful of output tiles (cuBLAS runs
// these shapes as 72-576 CTAs of split-K).  Each step stages 32 rows of the G and X column tiles into
// shared memory with cp.async, double-buffered; every thread keeps a 4 x 4 register tile of fp32 FMA
// accumulators.  The CTAs of the first K tile also sum their G column tile for db (in double: a Linear
// followed by a batch norm has a bias gradient that is zero up to cancellation).
//
// With S > 1 every CTA writes its tile to partials[S][N*K] (db to partials[S*N*K + s*N + n]) and a second
// launch adds the S partials per element in slab order.  No atomics: results are bit-identical from run
// to run and from graph replay to replay.
#include "common.cuh"

namespace rk {

constexpr int kLinTile = 64;                 // dW tile: 64 outputs (n) x 64 inputs (k)
constexpr int kLinRows = 32;                 // batch rows staged per step
constexpr int kLinThreads = 256;             // 16 x 16 threads, 4 x 4 outputs each
constexpr int kLinTargetCtas = 148 * 4;      // B200: 148 SMs, 4 CTAs of this kernel resident on each

// Batch slabs for a (B, K, N) problem: enough to put about kLinTargetCtas CTAs in the grid, with every
// slab a whole number of staged steps.  The same function sizes the grid and the scratch.
static void linear_plan(int64_t B, int K, int N, int* slabs, int64_t* slab_rows) {
    const int64_t tiles = ceil_div(K, kLinTile) * ceil_div(N, kLinTile);
    const int64_t want = ceil_div(kLinTargetCtas, tiles);
    int64_t rows = ceil_div(ceil_div(B, want), kLinRows) * kLinRows;
    *slab_rows = rows;
    *slabs = (int)ceil_div(B, rows);
}

template <int V>
__device__ __forceinline__ void cp_async(float* dst, const float* src, bool valid) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2, %3;\n" ::"r"(d), "l"(src), "n"(V * 4),
                 "r"(valid ? V * 4 : 0));
}

// Stages rows [row0, row0 + kLinRows) ∩ [.., row_end) and columns [col0, col0 + 64) ∩ [.., cols) of a
// row-major matrix; whatever falls outside is zero-filled.  V floats per copy: V divides cols and ld.
template <int V>
__device__ __forceinline__ void stage(float (*dst)[kLinTile], const float* __restrict__ src, int64_t ld,
                                      int cols, int64_t row0, int64_t row_end, int col0) {
    constexpr int kPerRow = kLinTile / V;
#pragma unroll
    for (int e = threadIdx.x; e < kLinRows * kPerRow; e += kLinThreads) {
        const int r = e / kPerRow, c = (e % kPerRow) * V;
        const int64_t row = row0 + r;
        const bool valid = row < row_end && col0 + c < cols;
        cp_async<V>(&dst[r][c], valid ? src + row * ld + col0 + c : src, valid);
    }
}

template <int V>
__global__ void __launch_bounds__(kLinThreads, 4)
linear_wgrad_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ g, int64_t ldg,
                    int64_t B, int K, int N, int64_t slab_rows, float* __restrict__ dW, float* __restrict__ db,
                    float* __restrict__ partials) {
    __shared__ __align__(16) float sG[2][kLinRows][kLinTile];
    __shared__ __align__(16) float sX[2][kLinRows][kLinTile];
    __shared__ double sDb[kLinThreads / kLinTile][kLinTile];

    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int k0 = blockIdx.x * kLinTile, n0 = blockIdx.y * kLinTile, slab = blockIdx.z;
    const int64_t row0 = (int64_t)slab * slab_rows;
    const int64_t row_end = min(B, row0 + slab_rows);
    const int steps = (int)((row_end - row0 + kLinRows - 1) / kLinRows);
    const bool with_db = db != nullptr && blockIdx.x == 0;

    float acc[4][4] = {};
    double dbacc = 0.0;                          // column n0 + (tid & 63), rows tid >> 6 + 4i of every step

    stage<V>(sG[0], g, ldg, N, row0, row_end, n0);
    stage<V>(sX[0], x, ldx, K, row0, row_end, k0);
    asm volatile("cp.async.commit_group;\n" ::);
    for (int st = 0; st < steps; ++st) {
        const int buf = st & 1;
        if (st + 1 < steps) {
            const int64_t r = row0 + (int64_t)(st + 1) * kLinRows;
            stage<V>(sG[buf ^ 1], g, ldg, N, r, row_end, n0);
            stage<V>(sX[buf ^ 1], x, ldx, K, r, row_end, k0);
            asm volatile("cp.async.commit_group;\n" ::);
            asm volatile("cp.async.wait_group 1;\n" ::);
        } else {
            asm volatile("cp.async.wait_group 0;\n" ::);
        }
        __syncthreads();
#pragma unroll 8
        for (int r = 0; r < kLinRows; ++r) {
            const float4 a = *reinterpret_cast<const float4*>(&sG[buf][r][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&sX[buf][r][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (with_db) {
#pragma unroll
            for (int r = tid >> 6; r < kLinRows; r += kLinThreads / kLinTile)
                dbacc += (double)sG[buf][r][tid & 63];
        }
        __syncthreads();                         // the buffer is restaged by the next step
    }

    const int64_t NK = (int64_t)N * K;
    float* out = partials ? partials + (int64_t)slab * NK : dW;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= N) break;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + tx * 4 + j;
            if (k < K) out[(int64_t)n * K + k] = acc[i][j];
        }
    }
    if (with_db) {
        sDb[tid >> 6][tid & 63] = dbacc;
        __syncthreads();
        const int n = n0 + tid;
        if (tid < kLinTile && n < N) {
            double s = 0.0;
#pragma unroll
            for (int q = 0; q < kLinThreads / kLinTile; ++q) s += sDb[q][tid];
            if (partials) partials[(int64_t)gridDim.z * NK + (int64_t)slab * N + n] = (float)s;
            else db[n] = (float)s;
        }
    }
}

// dW[i] = sum over s of partials[s * NK + i], db[n] likewise from the db block; slab order, in double.
__global__ void linear_wgrad_reduce_kernel(const float* __restrict__ partials, int S, int64_t NK, int N,
                                           float* __restrict__ dW, float* __restrict__ db) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const float* p;
    int64_t stride;
    float* out;
    if (i < NK) {
        p = partials + i, stride = NK, out = dW + i;
    } else if (db != nullptr && i < NK + N) {
        p = partials + (int64_t)S * NK + (i - NK), stride = N, out = db + (i - NK);
    } else {
        return;
    }
    double s = 0.0;
#pragma unroll 4
    for (int c = 0; c < S; ++c) s += (double)p[(int64_t)c * stride];
    *out = (float)s;
}

template <int V>
static int launch_linear_wgrad(const float* x, int64_t ldx, const float* g, int64_t ldg, int64_t B, int K, int N,
                               int S, int64_t slab_rows, float* dW, float* db, float* partials, cudaStream_t s) {
    const dim3 grid((unsigned)ceil_div(K, kLinTile), (unsigned)ceil_div(N, kLinTile), (unsigned)S);
    linear_wgrad_kernel<V><<<grid, kLinThreads, 0, s>>>(x, ldx, g, ldg, B, K, N, slab_rows, dW, db,
                                                        S > 1 ? partials : nullptr);
    RK_LAUNCH_CHECK();
    return 0;
}

}  // namespace rk

using namespace rk;

extern "C" {

int64_t rk_linear_wgrad_scratch_floats(int64_t B, int K, int N) {
    if (B < 1 || K < 1 || N < 1) return -1;
    int S;
    int64_t rows;
    linear_plan(B, K, N, &S, &rows);
    return S > 1 ? (int64_t)S * ((int64_t)N * K + N) : 0;
}

int rk_linear_wgrad(const float* x, int64_t ldx, const float* g, int64_t ldg, int64_t B, int K, int N,
                    float* dW, float* db, float* partials, rk_stream_t stream) {
    RK_CHECK_ARG(x && g && dW, "linear_wgrad: null x, g or dW");
    RK_CHECK_ARG(B >= 1 && K >= 1 && N >= 1, "linear_wgrad: bad shape B=%lld K=%d N=%d", (long long)B, K, N);
    RK_CHECK_ARG(ldx >= K && ldg >= N, "linear_wgrad: row pitch ldx=%lld < K=%d or ldg=%lld < N=%d",
                 (long long)ldx, K, (long long)ldg, N);
    RK_CHECK_ARG(ceil_div(N, kLinTile) <= 65535, "linear_wgrad: N=%d above %d", N, 65535 * kLinTile);
    int S;
    int64_t slab_rows;
    linear_plan(B, K, N, &S, &slab_rows);
    RK_CHECK_ARG(S == 1 || partials, "linear_wgrad: %d batch slabs need rk_linear_wgrad_scratch_floats floats "
                 "of partials", S);
    cudaStream_t s = (cudaStream_t)stream;
    // Widest copy that every row piece allows: V floats divide the width, the pitch and the base address.
    auto fits = [&](int v) {
        return K % v == 0 && N % v == 0 && ldx % v == 0 && ldg % v == 0 &&
               (uintptr_t)x % (4 * v) == 0 && (uintptr_t)g % (4 * v) == 0;
    };
    int rc;
    if (fits(4)) rc = launch_linear_wgrad<4>(x, ldx, g, ldg, B, K, N, S, slab_rows, dW, db, partials, s);
    else if (fits(2)) rc = launch_linear_wgrad<2>(x, ldx, g, ldg, B, K, N, S, slab_rows, dW, db, partials, s);
    else rc = launch_linear_wgrad<1>(x, ldx, g, ldg, B, K, N, S, slab_rows, dW, db, partials, s);
    if (rc || S == 1) return rc;
    const int64_t count = (int64_t)N * K + (db ? N : 0);
    linear_wgrad_reduce_kernel<<<(unsigned)ceil_div(count, 256), 256, 0, s>>>(partials, S, (int64_t)N * K, N, dW, db);
    RK_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
