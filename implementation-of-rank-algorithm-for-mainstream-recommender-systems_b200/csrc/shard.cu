// shard.cu — device side of the row-sharded embedding table (BASELINE config 5 "scaled": the
// feedid table of BST grown to 1e8 rows, block-partitioned by row over the ranks, SURVEY §8e).
// The reference has no distributed code; these kernels are the index bookkeeping around the two
// NCCL all-to-alls (indices out, rows back; mirrored for gradients):
//   rk_shard_owner   : owner[i] = idx[i] / rows_per_rank                     (bounds-checked)
//   rk_shard_route   : from the stable owner-sorted order (rk_plan_build on owner[]) produce the
//                      send buffer of owner-local row ids, the inverse permutation and the
//                      per-owner counts
// Integer, latency-bound work on a few hundred thousand elements per step.
#include "common.cuh"

namespace rk {

__global__ void __launch_bounds__(256)
shard_owner_kernel(const int64_t* __restrict__ idx, int64_t n, int64_t rows_total, int64_t rows_per_rank,
                   int64_t* __restrict__ owner, int32_t* err_flag) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        owner[i] = checked_row(idx[i], rows_total, err_flag) / rows_per_rank;
}

// sorted_owner / perm: output of rk_plan_build over owner[] (perm = original position, stable).
__global__ void __launch_bounds__(256)
shard_route_kernel(const int64_t* __restrict__ idx, const uint32_t* __restrict__ sorted_owner,
                   const uint32_t* __restrict__ perm, int64_t n, int64_t rows_total, int64_t rows_per_rank, int W,
                   int64_t* __restrict__ send_local, int64_t* __restrict__ inv, int64_t* __restrict__ counts) {
    __shared__ unsigned int hist[64];
    for (int i = threadIdx.x; i < 64; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t w = sorted_owner[i];
        const uint32_t src = perm[i];
        int64_t row = idx[src];
        if ((uint64_t)row >= (uint64_t)rows_total) row = 0;      // flagged by shard_owner_kernel
        send_local[i] = row - (int64_t)w * rows_per_rank;
        inv[src] = i;
        atomicAdd(&hist[w], 1u);
    }
    __syncthreads();
    for (int w = threadIdx.x; w < W; w += blockDim.x)
        if (hist[w]) atomicAdd(reinterpret_cast<unsigned long long*>(counts + w), (unsigned long long)hist[w]);
}

// One CTA, chunked scan: rank[i] = number of distinct keys before position i (keys sorted);
// uniq[rank] = key - key_base for every head; *n_uniq = number of distinct live keys.  Keys equal
// to dead_key (padding sentinel, sorted last) are left out.
struct CompactField {
    int64_t  start, n;            // slice of the sorted keys
    uint32_t key_base, dead_key;  // of the incoming keys
    uint32_t out_base, out_dead;  // of the rank keys written out
};
struct CompactFields {
    CompactField f[RK_MAX_FIELDS];
};

__global__ void __launch_bounds__(1024)
plan_compact_kernel(const uint32_t* __restrict__ keys_all, const __grid_constant__ CompactFields fields,
                    uint32_t* __restrict__ rank_all, int64_t* __restrict__ uniq_all, int64_t* __restrict__ n_uniq_all) {
    __shared__ uint32_t warp_tot[32];
    __shared__ uint32_t carry_s;
    const CompactField& fd = fields.f[blockIdx.x];
    const uint32_t* keys = keys_all + fd.start;
    uint32_t* rank_keys = rank_all + fd.start;
    int64_t* uniq = uniq_all + fd.start;
    int64_t* n_uniq = n_uniq_all + blockIdx.x;
    const int64_t n = fd.n;
    const uint32_t key_base = fd.key_base, dead_key = fd.dead_key;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) carry_s = 0;
    __syncthreads();
    for (int64_t base = 0; base < n; base += 1024) {
        const int64_t i = base + t;
        uint32_t k = 0, head = 0;
        if (i < n) {
            k = keys[i];
            head = (k != dead_key) && (i == 0 || keys[i - 1] != k) ? 1u : 0u;
        }
        uint32_t inc = head;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(kFull, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) warp_tot[w] = inc;
        __syncthreads();
        uint32_t before = carry_s;
        for (int ww = 0; ww < w; ++ww) before += warp_tot[ww];
        const uint32_t incl = before + inc;          // heads up to and including i
        if (i < n) {
            // rank of i's segment = heads before or at i, minus one; dead keys keep a sentinel rank
            rank_keys[i] = (k == dead_key) ? fd.out_dead : fd.out_base + incl - 1;
            if (head) uniq[incl - 1] = (int64_t)(k - key_base);
        }
        __syncthreads();
        if (t == 1023) carry_s = incl;
        __syncthreads();
    }
    if (t == 0) *n_uniq = carry_s;
}

}  // namespace rk

extern "C" {

int rk_shard_owner(const int64_t* idx, int64_t n, int64_t rows_total, int64_t rows_per_rank, int64_t* owner,
                   int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(n >= 0 && rows_total > 0 && rows_per_rank > 0, "shard_owner: bad sizes");
    if (n == 0) return 0;
    RK_CHECK_ARG(idx && owner, "shard_owner: NULL pointer");
    int64_t grid = ceil_div(n, 256);
    if (grid > (int64_t)sm_count() * 8) grid = (int64_t)sm_count() * 8;
    shard_owner_kernel<<<(int)grid, 256, 0, (cudaStream_t)stream_>>>(idx, n, rows_total, rows_per_rank, owner, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}

int rk_shard_route(const int64_t* idx, const uint32_t* sorted_owner, const uint32_t* perm, int64_t n,
                   int64_t rows_total, int64_t rows_per_rank, int W, int64_t* send_local, int64_t* inv,
                   int64_t* counts, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(W >= 1 && W <= 64, "shard_route: world size %d outside [1,64]", W);
    RK_CHECK_ARG(n >= 0 && rows_total > 0 && rows_per_rank > 0, "shard_route: bad sizes");
    RK_CHECK_ARG(counts, "shard_route: counts is NULL");
    cudaStream_t s = (cudaStream_t)stream_;
    RK_CUDA(cudaMemsetAsync(counts, 0, sizeof(int64_t) * W, s));
    if (n == 0) return 0;
    RK_CHECK_ARG(idx && sorted_owner && perm && send_local && inv, "shard_route: NULL pointer");
    int64_t grid = ceil_div(n, 256);
    if (grid > (int64_t)sm_count() * 4) grid = (int64_t)sm_count() * 4;
    shard_route_kernel<<<(int)grid, 256, 0, s>>>(idx, sorted_owner, perm, n, rows_total, rows_per_rank, W,
                                                 send_local, inv, counts);
    RK_LAUNCH_CHECK();
    return 0;
}

int rk_plan_compact_fields(const uint32_t* sorted_keys, const int64_t* n, const int64_t* rows, const int64_t* cap,
                           int F, uint32_t* rank_keys, int64_t* uniq_rows, int64_t* n_uniq, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(F >= 1 && F <= RK_MAX_FIELDS && n && rows && cap && n_uniq, "plan_compact_fields: bad argument");
    cudaStream_t s = (cudaStream_t)stream_;
    CompactFields cf;
    int64_t start = 0, in_base = 0, out_base = 0;
    for (int f = 0; f < F; ++f) {
        RK_CHECK_ARG(n[f] >= 0 && rows[f] > 0 && cap[f] > 0, "plan_compact_fields: field %d: n=%lld rows=%lld cap=%lld", f,
                     (long long)n[f], (long long)rows[f], (long long)cap[f]);
        // the key layout of rk_plan_build / rk_embgrad_segment_reduce: field f owns rows[f] + 1 keys
        cf.f[f] = CompactField{start, n[f], (uint32_t)in_base, (uint32_t)(in_base + rows[f]), (uint32_t)out_base,
                               (uint32_t)(out_base + cap[f])};
        start += n[f];
        in_base += rows[f] + 1;
        out_base += cap[f] + 1;
    }
    RK_CHECK_ARG(in_base < (1ll << 32) && out_base < (1ll << 32), "plan_compact_fields: key space overflow");
    if (start == 0) {
        RK_CUDA(cudaMemsetAsync(n_uniq, 0, sizeof(int64_t) * F, s));
        return 0;
    }
    RK_CHECK_ARG(sorted_keys && rank_keys && uniq_rows, "plan_compact_fields: NULL pointer");
    plan_compact_kernel<<<F, 1024, 0, s>>>(sorted_keys, cf, rank_keys, uniq_rows, n_uniq);
    RK_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
