// linear.cu — weight and bias gradients of the towers' nn.Linear layers, on the tensor core (tcgen05, 3xTF32).
//
//   dW[N, K] = G^T X = sum_b G[b, :]^T X[b, :]        db[N] = sum_b G[b, :]
//
// Both are one reduction over the batch, and both operands are row-major [B, *], so every batch row
// contributes a contiguous piece of a G row and of an X row.  The grid is (K tiles) x (N tiles) x
// (S batch slabs): a CTA owns a 128 x (up to 128) tile of dW and the rows of one slab, and S comes from
// linear_plan, which sizes the scratch too, so that the grid fills the GPU even where there are only a
// handful of output tiles.
//
// Where that grid would hold fewer than kTcMinCtas CTAs (half the SMs: a small batch, such as DeepFM's
// 256 -> 128 at B = 1024 with 64 CTAs of 32 rows), the same product runs instead as the fp32 SIMT kernel
// linear_wgrad_kernel over 64 x 64 tiles, four times as many CTAs: there the tensor-core CTAs spend most of
// their time outside the MMAs (TMEM allocation, the 128 x 128 epilogue), and scripts/bench_mm.py measured the
// SIMT kernel faster at that shape (10.2 against 12.3 us with L2 flushed; DESIGN section 3).
//
// The product is one tcgen05.mma per 8 batch rows: M = 128 outputs n (one TMEM lane each), N = the CTA's
// inputs k rounded up to 32 (K = 82 is one N = 96 tile), K = 8 batch rows.  Both operands are MN-major: a
// staged batch row of G or X is, in its natural row-major order, one 128-byte line per 32 columns, in the
// only layout MN-major tf32 takes (SWIZZLE_128B_BASE32B: 4 lines form a 512-byte atom whose 32-byte granules
// are XORed with line % 4; one MMA's K is two atoms, +1024 bytes), and the 32-column blocks of a stage are
// kTcBlock bytes apart (the leading byte offset).  So no transpose is needed.  Threads load the rows (16, 8
// or 4 bytes per load, whatever pitch and base allow; outside [0, B) x [0, N) x [0, K) is zero), split each
// value into hi = tf32(x) and lo = x - hi in registers and store both into hi / lo tiles; per 8 rows one
// thread issues G_hi.X_hi, G_lo.X_hi, G_hi.X_lo into the fp32 accumulator in TMEM.  That keeps about 22 bits of every
// operand (split bf16 would keep about 16, which is the whole fp32 error bar for DIN).  kTcStages stages
// of 16 rows are in flight: each has an mbarrier that tcgen05.commit signals when the MMAs reading it are
// done, and only then is it restaged; the next stage's rows are already loading into registers meanwhile.
// The CTAs of the first K tile also sum G for db in double, per thread over the columns it stages, the
// per-thread sums combined in a fixed order (a Linear followed by a batch norm has a bias gradient that is
// zero up to cancellation).
//
// With S > 1 every CTA writes its tile to partials[S][N*K] (db to partials[S*N*K + s*N + n]) and a second
// launch adds the S partials per element in slab order.  No atomics: results are bit-identical from run
// to run and from graph replay to replay, and do not depend on the load width.
#include "common.cuh"
#include "umma.cuh"

namespace rk {

using namespace tc;

constexpr int kLinTile = 64;                 // the plan's unit of dW tiles, and the SIMT kernel's (64 x 64)
constexpr int kLinRows = 32;                 // slab rows are a multiple of this: the SIMT kernel's step
constexpr int kLinTargetCtas = 148 * 4;      // B200: 148 SMs; CTAs of 64 x 64 tiles the plan aims for
constexpr int kLinThreads = 256;             // SIMT kernel: 16 x 16 threads, 4 x 4 outputs each

// Batch slabs for a (B, K, N) problem: enough to put about kLinTargetCtas 64 x 64 tiles in the grid, with
// every slab a whole number of kLinRows rows.  The same function sizes the grid and the scratch.  With the
// kernel's 128 x 128 tiles that is 148-152 CTAs for DIN's three layers at B = 8192.
static void linear_plan(int64_t B, int K, int N, int* slabs, int64_t* slab_rows) {
    const int64_t tiles = ceil_div(K, kLinTile) * ceil_div(N, kLinTile);
    const int64_t want = ceil_div(kLinTargetCtas, tiles);
    int64_t rows = ceil_div(ceil_div(B, want), kLinRows) * kLinRows;
    *slab_rows = rows;
    *slabs = (int)ceil_div(B, rows);
}

constexpr int kTcN = 128;                    // outputs n per CTA: the MMA's M
constexpr int kTcK = 128;                    // inputs k per CTA at most: the MMA's N
constexpr int kTcMinCtas = 148 / 2;          // smaller grids run the SIMT kernel (half the B200's SMs)
constexpr int kTcThreads = 256;
constexpr int kTcRows = 16;                  // batch rows per stage: two MMAs' K
constexpr int kTcStages = 3;
constexpr int kTcLine = 128;                 // one staged row of 32 fp32 columns
constexpr int kTcBlock = kTcRows * kTcLine;  // 2048: one 32-column block of a stage (the leading byte offset)
constexpr int kTcTile = 4 * kTcBlock;        // 8 KB: 128 columns x 16 rows
constexpr int kTcStageBytes = 4 * kTcTile;   // G hi, G lo, X hi, X lo: 32 KB
constexpr int kTcOutLd = kTcK + 1;           // epilogue transpose tile [128][129] floats, then db sums [8][128] doubles
// Shared memory: 1024 bytes of alignment slack + 3 stages x 32 KB + barriers = 97 KB, so 2 CTAs are resident
// per SM (the 256-thread CTA is also capped at 128 registers for that), and 2 x kTcTmemCols = 256 <= 512 TMEM
// columns: tcgen05.alloc never waits for another CTA of this kernel.
constexpr int kTcTmemCols = 128;
constexpr size_t kTcSmemBytes = 1024 + (size_t)kTcStages * kTcStageBytes + 64;
static_assert(kTcN * kTcOutLd * 4 + 8 * kTcN * 8 <= kTcStages * kTcStageBytes, "epilogue tiles fit the stages");
static_assert(kTcRows * (kTcN / 4) == 2 * kTcThreads && kTcRows * (kTcK / 4) == 2 * kTcThreads,
              "two 16-byte chunks of G and at most two of X per thread and stage");

// ---- tensor-core kernel ----

// Byte offset, within an operand tile, of the 16-byte chunk holding columns 4c..4c+3 of stage row r: block
// c / 8, line r, 32-byte granule (c % 8) / 2 XOR r % 4 (the 128B-base-32B swizzle), half c % 2 of it.
__device__ __forceinline__ uint32_t tc_chunk_offset(int r, int c) {
    return (uint32_t)((c >> 3) * kTcBlock + r * kTcLine + ((((c & 7) >> 1) ^ (r & 3)) << 5) + ((c & 1) << 4));
}

// Columns col..col+3 of one row, zero outside the row range or beyond `cols`: V floats per load (V divides
// cols, the pitch and the base address, so a V-wide piece is wholly inside or wholly outside).
template <int V>
__device__ __forceinline__ float4 load_chunk(const float* __restrict__ src, int64_t ld, int cols, bool row_ok,
                                             int64_t row, int col) {
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    const float* p = src + row * ld + col;
#pragma unroll
    for (int j = 0; j < 4; j += V) {
        if (!row_ok || col + j >= cols) continue;
        if constexpr (V == 4) {
            const float4 q = __ldg(reinterpret_cast<const float4*>(p));
            v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
        } else if constexpr (V == 2) {
            const float2 q = __ldg(reinterpret_cast<const float2*>(p + j));
            v[j] = q.x, v[j + 1] = q.y;
        } else {
            v[j] = __ldg(p + j);
        }
    }
    return make_float4(v[0], v[1], v[2], v[3]);
}

__device__ __forceinline__ void store_chunk_tf32(uint8_t* hi_tile, uint8_t* lo_tile, uint32_t off, float4 v) {
    float4 h, l;
    split_tf32(v.x, h.x, l.x);
    split_tf32(v.y, h.y, l.y);
    split_tf32(v.z, h.z, l.z);
    split_tf32(v.w, h.w, l.w);
    *reinterpret_cast<float4*>(hi_tile + off) = h;
    *reinterpret_cast<float4*>(lo_tile + off) = l;
}

template <int V>
__global__ void __launch_bounds__(kTcThreads, 2)
linear_wgrad_tc_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ g, int64_t ldg,
                       int64_t B, int K, int N, int64_t slab_rows, float* __restrict__ dW, float* __restrict__ db,
                       float* __restrict__ partials) {
    extern __shared__ uint8_t smem_raw_lin[];
    uint8_t* stages = smem_raw_lin + ((1024u - (smem_u32(smem_raw_lin) & 1023u)) & 1023u);
    uint64_t* bar = reinterpret_cast<uint64_t*>(stages + kTcStages * kTcStageBytes);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bar + kTcStages);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int k0 = blockIdx.x * kTcK, n0 = blockIdx.y * kTcN, slab = blockIdx.z;
    const int nk = min(kTcK, (K - k0 + 31) & ~31);            // the MMA's N
    const int xc = nk / 4;                                     // 16-byte X chunks per staged row
    const int64_t row0 = (int64_t)slab * slab_rows;
    const int64_t row_end = min(B, row0 + slab_rows);
    const int steps = (int)((row_end - row0 + kTcRows - 1) / kTcRows);
    const bool with_db = db != nullptr && blockIdx.x == 0;

    if (tid == 0)
        for (int i = 0; i < kTcStages; ++i) mbar_init(&bar[i], 1);
    if (warp == 0) tmem_alloc(tmem_slot, kTcTmemCols);         // the same warp deallocates
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t idesc = umma_idesc_tf32(nk) | kUmmaAMn | kUmmaBMn;

    // This thread's chunks of every stage: G rows (tid / 32) + 8i, columns 4 (tid % 32); X chunk tid + 256i.
    const int gcol = 4 * lane;
    int grow[2], xrow[2], xcol[2];
    uint32_t goff[2], xoff[2];
    bool xon[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        grow[i] = warp + 8 * i;
        goff[i] = tc_chunk_offset(grow[i], lane);
        const int e = tid + kTcThreads * i;
        xon[i] = e < kTcRows * xc;
        xrow[i] = xon[i] ? e / xc : 0;
        xcol[i] = xon[i] ? 4 * (e - xrow[i] * xc) : 0;
        xoff[i] = tc_chunk_offset(xrow[i], xcol[i] / 4);
    }
    auto load_step = [&](int st, float4 (&gv)[2], float4 (&xv)[2]) {
        const int64_t r0 = row0 + (int64_t)st * kTcRows;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            gv[i] = load_chunk<V>(g, ldg, N, r0 + grow[i] < row_end, r0 + grow[i], n0 + gcol);
            xv[i] = load_chunk<V>(x, ldx, K, xon[i] && r0 + xrow[i] < row_end, r0 + xrow[i], k0 + xcol[i]);
        }
    };

    double dbacc[4] = {0.0, 0.0, 0.0, 0.0};                    // columns n0 + gcol + j
    float4 gc[2], xv[2];
    load_step(0, gc, xv);
    for (int st = 0; st < steps; ++st) {
        const int buf = st % kTcStages;
        float4 gn[2], xn[2];
        load_step(st + 1, gn, xn);                             // zeros past the slab; in flight while this step is stored
        if (st >= kTcStages) mbar_wait(&bar[buf], ((st - kTcStages) / kTcStages) & 1);   // its MMAs have read buf
        uint8_t* s = stages + buf * kTcStageBytes;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            store_chunk_tf32(s, s + kTcTile, goff[i], gc[i]);
            if (xon[i]) store_chunk_tf32(s + 2 * kTcTile, s + 3 * kTcTile, xoff[i], xv[i]);
            if (with_db) {
                dbacc[0] += (double)gc[i].x, dbacc[1] += (double)gc[i].y;
                dbacc[2] += (double)gc[i].z, dbacc[3] += (double)gc[i].w;
            }
        }
        fence_async_smem();                                    // generic-proxy stores -> the MMAs' async proxy
        __syncthreads();
        if (tid == 0) {
            fence_after();
            const int64_t left = row_end - (row0 + (int64_t)st * kTcRows);
            const int kmma = left >= kTcRows ? kTcRows / 8 : (int)((left + 7) / 8);
            const uint32_t a = smem_u32(s);
            for (int kk = 0; kk < kmma; ++kk) {
                const uint32_t o = 1024u * kk;
                const uint64_t g_hi = umma_desc_mn_tf32(a + o, kTcBlock);
                const uint64_t g_lo = umma_desc_mn_tf32(a + kTcTile + o, kTcBlock);
                const uint64_t x_hi = umma_desc_mn_tf32(a + 2 * kTcTile + o, kTcBlock);
                const uint64_t x_lo = umma_desc_mn_tf32(a + 3 * kTcTile + o, kTcBlock);
                umma_tf32(tmem, g_hi, x_hi, idesc, (st > 0 || kk > 0) ? 1u : 0u);
                umma_tf32(tmem, g_lo, x_hi, idesc, 1u);
                umma_tf32(tmem, g_hi, x_lo, idesc, 1u);
            }
            umma_commit(&bar[buf]);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) gc[i] = gn[i], xv[i] = xn[i];
    }
    const int last = steps - 1;
    mbar_wait(&bar[last % kTcStages], (last / kTcStages) & 1);  // every MMA of the CTA is done
    fence_after();

    // Accumulator -> shared memory (the stages are free now) -> coalesced rows of dW or partials[slab].
    float* sOut = reinterpret_cast<float*>(stages);
    double* sDb = reinterpret_cast<double*>(stages + kTcN * kTcOutLd * 4);
    const int quarter = warp & 3;                              // a warp reads TMEM lanes 32 (warp % 4) ..
    for (int j = warp >> 2; j < nk / 32; j += 2) {
        float v[32];
        tmem_ld32(tmem + ((uint32_t)(quarter * 32) << 16) + 32 * j, v);
        float* row = sOut + (quarter * 32 + lane) * kTcOutLd + 32 * j;
#pragma unroll
        for (int i = 0; i < 32; ++i) row[i] = v[i];
    }
    if (with_db) {
#pragma unroll
        for (int j = 0; j < 4; ++j) sDb[warp * kTcN + gcol + j] = dbacc[j];
    }
    fence_before();
    __syncthreads();
    if (warp == 0) {
        fence_after();
        tmem_dealloc(tmem, kTcTmemCols);
    }

    const int64_t NK = (int64_t)N * K;
    float* out = partials ? partials + (int64_t)slab * NK : dW;
    const int kc = min(kTcK, K - k0);
    for (int r = warp; r < kTcN && n0 + r < N; r += kTcThreads / 32) {
        float* orow = out + (int64_t)(n0 + r) * K + k0;
        for (int c = lane; c < kc; c += 32) orow[c] = sOut[r * kTcOutLd + c];
    }
    if (with_db && tid < kTcN && n0 + tid < N) {
        double sum = 0.0;
#pragma unroll
        for (int q = 0; q < kTcThreads / 32; ++q) sum += sDb[q * kTcN + tid];
        if (partials) partials[(int64_t)gridDim.z * NK + (int64_t)slab * N + n0 + tid] = (float)sum;
        else db[n0 + tid] = (float)sum;
    }
}

// ---- fp32 SIMT kernel for small grids: 64 x 64 tiles, 32 rows per step staged by cp.async ----

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
    const dim3 grid((unsigned)ceil_div(K, kTcK), (unsigned)ceil_div(N, kTcN), (unsigned)S);
    float* part = S > 1 ? partials : nullptr;
    if ((int64_t)grid.x * grid.y * grid.z < kTcMinCtas) {
        const dim3 simt((unsigned)ceil_div(K, kLinTile), (unsigned)ceil_div(N, kLinTile), (unsigned)S);
        linear_wgrad_kernel<V><<<simt, kLinThreads, 0, s>>>(x, ldx, g, ldg, B, K, N, slab_rows, dW, db, part);
    } else {
        RK_CUDA(cudaFuncSetAttribute(linear_wgrad_tc_kernel<V>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)kTcSmemBytes));
        linear_wgrad_tc_kernel<V><<<grid, kTcThreads, kTcSmemBytes, s>>>(x, ldx, g, ldg, B, K, N, slab_rows, dW, db,
                                                                        part);
    }
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
