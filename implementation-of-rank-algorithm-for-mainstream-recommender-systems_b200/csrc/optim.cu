// optim.cu — row-wise (lazy) Adam on the touched rows of an embedding table (SURVEY 8(f) item 3).
//
// The reference trains with optim.Adam over DENSE [V, D] gradients: every step zero-fills and sweeps
// whole tables although a batch touches a few thousand rows (38 % of the DeepFM CPU step).  Given the
// compact gradient the occurrence plan already produces — the unique touched rows and one summed
// gradient row each — this kernel updates only those rows of weight / exp_avg / exp_avg_sq.  The
// arithmetic is torch.optim.SparseAdam's (moments of untouched rows are not decayed, the bias
// correction uses the global step), which is a different optimizer from dense Adam: opt-in.
// rk_adam_step (below) is dense Adam itself.
#include <string.h>
#include "common.cuh"

namespace rk {

template <int VEC>
__global__ void __launch_bounds__(256)
rowwise_adam_kernel(float* __restrict__ weight, float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq,
                    const int64_t* __restrict__ rows, const float* __restrict__ grads, int64_t n,
                    const int64_t* __restrict__ n_dev, int D, int64_t V,
                    float beta1, float beta2, float eps, float step_size, int32_t* err_flag) {
    const int units = D / VEC;
    const int64_t gid = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    const int64_t i = gid / units;
    const int u = (int)(gid - i * units);
    if (n_dev) {                                      // the live count sits on the device (no host sync upstream)
        const int64_t live = __ldg(n_dev);
        if (live < n) n = live;
    }
    if (i >= n) return;
    const int64_t raw = __ldg(rows + i);
    if ((uint64_t)raw >= (uint64_t)V) {               // never write outside the table
        if (err_flag) atomicOr(err_flag, 1);
        return;
    }
    const int64_t off = raw * D + u * VEC;
    Vec<VEC> g, m, v, w;
    g.load(grads + i * D + u * VEC);
    m.load_plain(exp_avg + off);
    v.load_plain(exp_avg_sq + off);
    w.load_plain(weight + off);
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
        // torch.optim.SparseAdam: m += (g - m)(1 - b1); v += (g^2 - v)(1 - b2); w -= step_size * m / (sqrt(v) + eps)
        m.v[k] = m.v[k] + (g.v[k] - m.v[k]) * (1.0f - beta1);
        v.v[k] = v.v[k] + (g.v[k] * g.v[k] - v.v[k]) * (1.0f - beta2);
        w.v[k] = w.v[k] - step_size * (m.v[k] / (sqrtf(v.v[k]) + eps));
    }
    m.store(exp_avg + off);
    v.store(exp_avg_sq + off);
    w.store(weight + off);
}

}  // namespace rk

static int rowwise_adam_launch(float* weight, float* exp_avg, float* exp_avg_sq, const int64_t* rows, const float* grads,
                               int64_t n, const int64_t* n_dev, int D, int64_t V, float lr, float beta1, float beta2,
                               float eps, int64_t step, int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(weight && exp_avg && exp_avg_sq && (n == 0 || (rows && grads)), "rowwise_adam: NULL pointer");
    RK_CHECK_ARG(n >= 0 && D >= 1 && V >= 1 && step >= 1, "rowwise_adam: n=%lld D=%d V=%lld step=%lld", (long long)n, D,
                 (long long)V, (long long)step);
    if (n == 0) return 0;
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    const float step_size = (float)((double)lr * sqrt(bc2) / bc1);
    int vec = D % 4 == 0 ? 4 : (D % 2 == 0 ? 2 : 1);
    auto mis = [&](const void* p) { return ((uintptr_t)p % (4 * vec)) != 0; };
    while (vec > 1 && (mis(weight) || mis(exp_avg) || mis(exp_avg_sq) || mis(grads))) vec >>= 1;
    const int64_t threads = n * (D / vec);
    const int grid = (int)ceil_div(threads, 256);
    cudaStream_t s = (cudaStream_t)stream_;
    if (vec == 4) rowwise_adam_kernel<4><<<grid, 256, 0, s>>>(weight, exp_avg, exp_avg_sq, rows, grads, n, n_dev, D, V, beta1, beta2, eps, step_size, err_flag);
    else if (vec == 2) rowwise_adam_kernel<2><<<grid, 256, 0, s>>>(weight, exp_avg, exp_avg_sq, rows, grads, n, n_dev, D, V, beta1, beta2, eps, step_size, err_flag);
    else rowwise_adam_kernel<1><<<grid, 256, 0, s>>>(weight, exp_avg, exp_avg_sq, rows, grads, n, n_dev, D, V, beta1, beta2, eps, step_size, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}

extern "C" int rk_rowwise_adam(float* weight, float* exp_avg, float* exp_avg_sq, const int64_t* rows,
                               const float* grads, int64_t n, int D, int64_t V, float lr, float beta1, float beta2,
                               float eps, int64_t step, int32_t* err_flag, rk_stream_t stream_) {
    return rowwise_adam_launch(weight, exp_avg, exp_avg_sq, rows, grads, n, nullptr, D, V, lr, beta1, beta2, eps, step,
                               err_flag, stream_);
}

extern "C" int rk_rowwise_adam_touched(float* weight, float* exp_avg, float* exp_avg_sq, const int64_t* rows,
                                       const float* grads, const int64_t* count, int64_t capacity, int D, int64_t V,
                                       float lr, float beta1, float beta2, float eps, int64_t step, int32_t* err_flag,
                                       rk_stream_t stream_) {
    RK_CHECK_ARG(count, "rowwise_adam_touched: count is NULL");
    return rowwise_adam_launch(weight, exp_avg, exp_avg_sq, rows, grads, capacity, count, D, V, lr, beta1, beta2, eps,
                               step, err_flag, stream_);
}

// ---- dense Adam, bit-identical to torch.optim.Adam(fused=True), in one launch over every tensor ----------------
// The reference's optimizer (optim.Adam(model.parameters(), lr), e.g. DCN/dcn.py:246) decays the moments of every
// row every step.  An untouched row's gradient is exactly zero, so the update needs no dense gradient: a tensor
// with a touched-rows gradient (distinct ascending rows, summed values, count on the device) is swept row by row
// and takes g = 0 where no slot names the row.  Dense .grad tensors (towers; tables in the default mode) are a
// plain sweep.  Arithmetic: ATen's fused_adam_utils.cuh adam_math, ADAM_MODE::ORIGINAL, no weight decay /
// amsgrad / maximize / grad scale, with the step read from its float32 tensor (incremented before the launch).
//
// Work split: every CTA owns one chunk of one tensor — kAdamChunk elements of a dense tensor, or the rows
// [r0, r1) of a touched one (at most kAdamChunk elements).  A touched CTA finds its first slot with a 256-ary
// search of rows[0:count] (three rounds for 10^7 slots), maps the rows of its range to their slots in shared
// memory, then does the same vectorised pass as a dense CTA.  Memory-bound: p, m, v read and written (24 B per
// element) plus the gradient (4 B per element dense, the touched rows only otherwise).
namespace rk {

constexpr int kAdamThreads = 256;
constexpr int kAdamChunk   = 4096;       // elements per CTA (16 KB of each of p, m, v)

struct AdamJob {
    float*         p;
    float*         m;
    float*         v;
    const float*   step;
    const float*   g;         // dense gradient, or the touched values [capacity, dim]
    const int64_t* trows;     // NULL: dense
    const int64_t* tcount;
    int64_t        capacity;
    int64_t        rows;      // dense: numel (dim 1)
    int32_t        dim;
    int32_t        rows_per_chunk;
    int32_t        chunk_start;
    int32_t        vec;       // 4, 2 or 1 floats per access of p, m, v (and g when gvec)
    int32_t        gvec;      // touched values can be read with the same vector width
    float          lr, beta1, beta2, eps;
};
struct AdamParams {
    AdamJob job[RK_ADAM_MAX_TENSORS];
    int32_t n;
};
static_assert(sizeof(AdamParams) <= 32764, "kernel parameter limit");

__device__ __forceinline__ void adam_elem(float& p, float& m, float& v, float g, const AdamJob& j, float step_size,
                                          float bc2_sqrt) {
    m = fmaf(j.beta1, m, fmaf(-j.beta1, g, g));
    const float gg = g * g;
    v = fmaf(j.beta2, v, fmaf(-j.beta2, gg, gg));
    const float denom = sqrtf(v) / bc2_sqrt + j.eps;
    p -= step_size * m / denom;
}

// gradient of element `le` (counted from the chunk's first element) of a touched tensor
__device__ __forceinline__ float touched_grad_at(const AdamJob& j, const int32_t* slot_of, int64_t first, int64_t le) {
    const int64_t r = le / j.dim;
    const int32_t s = slot_of[r];
    return s < 0 ? 0.f : __ldg(j.g + (first + s) * j.dim + (le - r * j.dim));
}

template <int VEC, bool GVEC>
__device__ __forceinline__ void adam_sweep(const AdamJob& j, int64_t r0, int64_t r1, const int32_t* slot_of,
                                           int64_t first, float step_size, float bc2_sqrt) {
    const int64_t e0 = r0 * j.dim, n = (r1 - r0) * j.dim;
    const int64_t nvec = n / VEC;
    for (int64_t i = threadIdx.x; i < nvec; i += kAdamThreads) {
        const int64_t le = i * VEC;
        Vec<VEC> p, m, v, g;
        p.load_plain(j.p + e0 + le);
        m.load_plain(j.m + e0 + le);
        v.load_plain(j.v + e0 + le);
        if (!j.trows) {
            g.load(j.g + e0 + le);
        } else if (GVEC) {                       // dim % VEC == 0: the vector lies inside one row
            const int64_t r = le / j.dim;
            const int32_t s = slot_of[r];
            if (s < 0) vec_zero(g);
            else g.load(j.g + (first + s) * j.dim + (le - r * j.dim));
        } else {
#pragma unroll
            for (int k = 0; k < VEC; ++k) g.v[k] = touched_grad_at(j, slot_of, first, le + k);
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) adam_elem(p.v[k], m.v[k], v.v[k], g.v[k], j, step_size, bc2_sqrt);
        p.store(j.p + e0 + le);
        m.store(j.m + e0 + le);
        v.store(j.v + e0 + le);
    }
    for (int64_t le = nvec * VEC + threadIdx.x; le < n; le += kAdamThreads) {     // tail of an odd-sized tensor
        float p = j.p[e0 + le], m = j.m[e0 + le], v = j.v[e0 + le];
        const float g = j.trows ? touched_grad_at(j, slot_of, first, le) : __ldg(j.g + e0 + le);
        adam_elem(p, m, v, g, j, step_size, bc2_sqrt);
        j.p[e0 + le] = p;
        j.m[e0 + le] = m;
        j.v[e0 + le] = v;
    }
}

__global__ void __launch_bounds__(kAdamThreads)
adam_kernel(const __grid_constant__ AdamParams P, int32_t* err_flag) {
    __shared__ int32_t slot_of[kAdamChunk];     // local row -> touched slot - first, or -1
    int lo = 0, hi = P.n - 1;                   // the last job whose chunks start at or before this CTA
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (P.job[mid].chunk_start <= (int)blockIdx.x) lo = mid;
        else hi = mid - 1;
    }
    const AdamJob& j = P.job[lo];
    const int64_t r0 = (int64_t)(blockIdx.x - j.chunk_start) * j.rows_per_chunk;
    const int64_t r1 = min(r0 + j.rows_per_chunk, j.rows);

    // torch's fused functor: bias corrections in fp32 from the fp32 step
    const float step = __ldg(j.step);
    const float bc1 = 1.f - powf(j.beta1, step);
    const float bc2_sqrt = sqrtf(1.f - powf(j.beta2, step));
    const float step_size = j.lr / bc1;

    int64_t first = 0;
    if (j.trows) {
        for (int i = threadIdx.x; i < r1 - r0; i += kAdamThreads) slot_of[i] = -1;
        int64_t count = j.capacity > 0 ? __ldg(j.tcount) : 0;
        count = count < 0 ? 0 : (count > j.capacity ? j.capacity : count);
        // first slot whose row is >= r0: every round probes 256 evenly spaced slots of [lo, hi)
        int64_t slo = 0, shi = count;
        while (slo < shi) {
            const int64_t stride = (shi - slo + kAdamThreads - 1) / kAdamThreads;
            const int64_t probe = slo + threadIdx.x * stride;
            const int below = __syncthreads_count(probe < shi && __ldg(j.trows + probe) < r0);
            if (below == 0) break;
            const int64_t next_lo = slo + (below - 1) * stride + 1;
            shi = min(shi, slo + below * stride);
            slo = next_lo;
        }
        first = slo;
        __syncthreads();                                  // the -1 fill is complete
        for (int64_t s = first + threadIdx.x; s < count && s < first + (r1 - r0); s += kAdamThreads) {
            const int64_t row = __ldg(j.trows + s);
            if (row >= r0 && row < r1) slot_of[row - r0] = (int32_t)(s - first);
        }
        if (threadIdx.x == 0 && err_flag) {               // rows outside [0, V) are skipped and flagged
            if (r0 == 0 && first > 0) atomicOr(err_flag, 1);
            if (r1 == j.rows && count > 0 && __ldg(j.trows + count - 1) >= j.rows) atomicOr(err_flag, 1);
        }
        __syncthreads();
    }
    if (j.vec == 4) {
        if (j.gvec) adam_sweep<4, true>(j, r0, r1, slot_of, first, step_size, bc2_sqrt);
        else adam_sweep<4, false>(j, r0, r1, slot_of, first, step_size, bc2_sqrt);
    } else if (j.vec == 2) {
        if (j.gvec) adam_sweep<2, true>(j, r0, r1, slot_of, first, step_size, bc2_sqrt);
        else adam_sweep<2, false>(j, r0, r1, slot_of, first, step_size, bc2_sqrt);
    } else {
        adam_sweep<1, true>(j, r0, r1, slot_of, first, step_size, bc2_sqrt);
    }
}

}  // namespace rk

static_assert(sizeof(rk_adam_tensor_t) == 104, "rk_adam_tensor_t layout (mirrored by _lib.RkAdamTensor)");

extern "C" int rk_adam_step(const rk_adam_tensor_t* tensors, int n, int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(n >= 0 && n <= RK_ADAM_MAX_TENSORS && (n == 0 || tensors), "adam_step: n=%d (max %d)", n,
                 RK_ADAM_MAX_TENSORS);
    AdamParams P;
    memset(&P, 0, sizeof(P));
    int64_t chunks = 0;
    auto aligned = [](const void* q, int bytes) { return ((uintptr_t)q % bytes) == 0; };
    for (int i = 0; i < n; ++i) {
        const rk_adam_tensor_t& t = tensors[i];
        const bool touched = t.touched_count != nullptr;
        RK_CHECK_ARG(t.param && t.exp_avg && t.exp_avg_sq && t.step, "adam_step: tensor %d: NULL pointer", i);
        RK_CHECK_ARG(touched != (t.grad != nullptr), "adam_step: tensor %d needs exactly one of grad / touched_count", i);
        RK_CHECK_ARG(t.rows >= 0 && t.dim >= 1, "adam_step: tensor %d: rows=%lld dim=%d", i, (long long)t.rows, t.dim);
        RK_CHECK_ARG(!touched || (t.capacity >= 0 && (t.capacity == 0 || (t.touched_rows && t.touched_values))),
                     "adam_step: tensor %d: touched capacity=%lld with NULL rows / values", i, (long long)t.capacity);
        if (t.rows == 0) continue;
        AdamJob& j = P.job[P.n];
        j.p = t.param;
        j.m = t.exp_avg;
        j.v = t.exp_avg_sq;
        j.step = t.step;
        j.g = touched ? t.touched_values : t.grad;
        j.trows = touched ? t.touched_rows : nullptr;
        j.tcount = touched ? t.touched_count : nullptr;
        j.capacity = t.capacity;
        j.lr = t.lr;
        j.beta1 = t.beta1;
        j.beta2 = t.beta2;
        j.eps = t.eps;
        if (touched) {                 // a chunk is whole rows; chunk starts stay 16-byte aligned where dim allows
            j.rows = t.rows;
            j.dim = t.dim;
            const int rpc = (kAdamChunk / t.dim) & ~3;
            j.rows_per_chunk = rpc > 0 ? rpc : 1;
        } else {                       // dense: flat over all elements
            RK_CHECK_ARG(t.rows <= INT64_MAX / t.dim, "adam_step: tensor %d too large", i);
            j.rows = t.rows * t.dim;
            j.dim = 1;
            j.rows_per_chunk = kAdamChunk;
        }
        int vec = 4;
        while (vec > 1 && !(aligned(j.p, 4 * vec) && aligned(j.m, 4 * vec) && aligned(j.v, 4 * vec) &&
                            ((int64_t)j.rows_per_chunk * j.dim) % vec == 0 && (touched || aligned(j.g, 4 * vec))))
            vec >>= 1;
        j.vec = vec;
        j.gvec = !touched || (j.dim % vec == 0 && aligned(j.g, 4 * vec));
        j.chunk_start = (int32_t)chunks;
        chunks += ceil_div(j.rows, j.rows_per_chunk);
        RK_CHECK_ARG(chunks < INT32_MAX, "adam_step: %lld chunks in one launch", (long long)chunks);
        ++P.n;
    }
    if (P.n == 0) return 0;
    adam_kernel<<<(unsigned)chunks, kAdamThreads, 0, (cudaStream_t)stream_>>>(P, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}
