// metrics.cu — evaluation metrics on the device: exact ROC AUC, per-group AUC (uAUC), log loss and
// accuracy.  Replaces the per-step loss.item()/label.cpu()/prob.cpu() syncs and the per-epoch sklearn
// roc_auc_score / accuracy_score over host lists (DeepFM/deepfm.py:173-180, :184-208).
//
// AUC as integers.  Sort the samples by (group, score) — an order-preserving uint32 key of the score,
// the LSD radix sort of plan_sort.cu, then a stable pass over the group id — and cut the order into
// runs of equal (group, key).  A run r with pos_r positives and neg_r negatives, neg_before_r
// negatives below it in its group, adds pos_r * (2 neg_before_r + neg_r) to 2U, the doubled
// Mann-Whitney numerator with ties counted one half; AUC = 2U / (2 P N) is sklearn's tie-averaged
// roc_auc_score.  Every quantity is an integer, so the result is exact whatever the input order and
// the tiling; the per-group sums use integer atomics, which are order-independent.  Floating point
// appears only in the per-group divisions and the uAUC / log-loss sums, both in a fixed order.
//
// The run pass works per element, so a run may span any number of tiles.  For the sample at sorted
// position j with NC = negatives before j, RS = the start of its run, NRS = negatives before RS and
// NGS = negatives before its group's start:
//   positive: 2 (NRS - NGS) + (NC - NRS)    (negatives below the run, twice; the run's negatives before j)
//   negative: (j - RS) - (NC - NRS)         (the run's positives before j)
// summed over a run this is pos_r (2 neg_before_r) + pos_r neg_r: every (positive, negative) pair of
// the run is counted once, by whichever comes later.  NC is a prefix sum and RS / NRS / NGS are
// "last start" values, i.e. prefix maxima: a tile pass of aggregates, one CTA that scans them, and a
// tile pass that finishes the scan and adds each group's in-tile segment to that group's counters.
//
// Data-parallel ranks: rk_metrics_merge concatenates the all-gathered buffers of every rank (each rank's
// filled prefix, rank-major) and ORs their statuses, so rk_metrics_compute sees the whole evaluation set.
#include <string.h>
#include "common.cuh"
#include "radix_sort.cuh"

namespace rk {

constexpr int kAppendThreads = 256;
constexpr int kAppendMaxCtas = 1024;
constexpr int kMetricTile    = 2048;                        // positions per CTA of every pass
constexpr int kKeyThreads    = 256;
constexpr int kKeyRounds     = kMetricTile / kKeyThreads;
constexpr int kRunThreads    = 512;
constexpr int kRunWarps      = kRunThreads / 32;
constexpr int kPer           = kMetricTile / kRunThreads;   // consecutive positions per thread
constexpr int kCarryThreads  = 1024;
constexpr int kFinalThreads  = 1024;

// Order-preserving map of a finite fp32 to uint32: negatives get all bits flipped, positives only the
// sign bit.  -0.0 is mapped to +0.0 first: they compare equal, so they must tie (as sklearn ties them).
__device__ __forceinline__ uint32_t score_key(float s) {
    uint32_t u = __float_as_uint(s);
    if (u == 0x80000000u) u = 0u;
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// ---------------------------------------------------------------------------------------- append
__global__ void __launch_bounds__(kAppendThreads)
metrics_append_kernel(const float* __restrict__ score, const float* __restrict__ label,
                      const int64_t* __restrict__ group, int64_t B, float* __restrict__ score_buf,
                      float* __restrict__ label_buf, int64_t* __restrict__ group_buf, int64_t capacity,
                      int64_t num_groups, int64_t* count, uint32_t* status) {
    __shared__ uint32_t bits_s;
    if (threadIdx.x == 0) bits_s = 0;
    // Every CTA reads the offset before it arrives below, and only the last CTA to arrive advances
    // it, so all CTAs of the launch see the same offset.
    const int64_t base = *(volatile const int64_t*)count;
    __syncthreads();
    uint32_t bits = 0;
    for (int64_t i = blockIdx.x * (int64_t)kAppendThreads + threadIdx.x; i < B;
         i += (int64_t)gridDim.x * kAppendThreads) {
        const float s = score[i], y = label[i];
        if (!isfinite(s)) bits |= RK_METRICS_NONFINITE;
        if (!(s >= 0.f && s <= 1.f)) bits |= RK_METRICS_NOT_PROB;
        if (!(y == 0.f || y == 1.f)) bits |= RK_METRICS_BAD_LABEL;
        int64_t g = 0;
        if (group) {
            g = group[i];
            if ((uint64_t)g >= (uint64_t)num_groups) bits |= RK_METRICS_BAD_GROUP;
        }
        const int64_t o = base + i;
        if (o >= capacity) {
            bits |= RK_METRICS_OVERFLOW;
            continue;
        }
        score_buf[o] = s;
        label_buf[o] = y;
        if (group) group_buf[o] = g;
    }
    bits = __reduce_or_sync(kFull, bits);
    if ((threadIdx.x & 31) == 0 && bits) atomicOr(&bits_s, bits);
    __syncthreads();
    if (threadIdx.x == 0) {
        if (bits_s) atomicOr(status, bits_s);
        __threadfence();
        const unsigned long long arrived = atomicAdd((unsigned long long*)(count + 1), 1ull);
        if (arrived == gridDim.x - 1) {
            count[0] = min(base + B, capacity);
            count[1] = 0;
        }
    }
}

// ---------------------------------------------------------------------------------------- compute
// Keys in storage order, plus per-CTA partials of the log loss (double) and of the correct count.
__global__ void __launch_bounds__(kKeyThreads)
metrics_key_kernel(const float* __restrict__ score, const float* __restrict__ label, int64_t n,
                   uint32_t* __restrict__ keys, uint32_t* __restrict__ vals, double* __restrict__ ll_part,
                   unsigned long long* __restrict__ acc_part) {
    __shared__ double ll_w[kKeyThreads / 32];
    __shared__ unsigned acc_w[kKeyThreads / 32];
    const int64_t base = (int64_t)blockIdx.x * kMetricTile;
    double ll = 0.0;
    unsigned acc = 0;
#pragma unroll
    for (int r = 0; r < kKeyRounds; ++r) {
        const int64_t i = base + r * kKeyThreads + threadIdx.x;
        if (i < n) {
            const float s = score[i], y = label[i];
            keys[i] = score_key(s);
            vals[i] = (uint32_t)i;
            const double p = (double)s, yd = (double)y;
            // F.binary_cross_entropy: each log clamped at -100 (so p = 0 or 1 gives a finite loss)
            ll -= yd * fmax(log(p), -100.0) + (1.0 - yd) * fmax(log1p(-p), -100.0);
            acc += (s > 0.5f) == (y > 0.5f);
        }
    }
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        ll += __shfl_xor_sync(kFull, ll, o);
        acc += __shfl_xor_sync(kFull, acc, o);
    }
    if (lane == 0) { ll_w[w] = ll; acc_w[w] = acc; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double l = 0.0;
        unsigned long long a = 0;
        for (int k = 0; k < kKeyThreads / 32; ++k) { l += ll_w[k]; a += acc_w[k]; }
        ll_part[blockIdx.x] = l;
        acc_part[blockIdx.x] = a;
    }
}

// Group keys of the score-sorted order, for the stable pass that groups it.
__global__ void __launch_bounds__(256)
group_key_kernel(const int64_t* __restrict__ group, const uint32_t* __restrict__ perm, int64_t n,
                 int64_t num_groups, uint32_t* __restrict__ keys, uint32_t* __restrict__ vals) {
    const int64_t j = blockIdx.x * 256ll + threadIdx.x;
    if (j >= n) return;
    const uint32_t i = perm[j];
    int64_t g = group[i];
    if ((uint64_t)g >= (uint64_t)num_groups) g = 0;   // flagged by rk_metrics_append; keeps the counters in bounds
    keys[j] = (uint32_t)g;
    vals[j] = i;
}

// Sorted position j -> its score key and (group << 1 | is_positive), read coalesced by the run passes.
__global__ void __launch_bounds__(256)
gather_sorted_kernel(const float* __restrict__ score, const float* __restrict__ label,
                     const uint32_t* __restrict__ perm, const uint32_t* __restrict__ group_sorted, int64_t n,
                     uint32_t* __restrict__ key, uint32_t* __restrict__ gl) {
    const int64_t j = blockIdx.x * 256ll + threadIdx.x;
    if (j >= n) return;
    const uint32_t i = perm[j];
    key[j] = score_key(score[i]);
    gl[j]  = ((group_sorted ? group_sorted[j] : 0u) << 1) | (label[i] > 0.5f ? 1u : 0u);
}

// Negatives (sum), last run start and last group start (max of positions, -1 = none).
struct Tri {
    int32_t neg, rs, gs;
};
__device__ __forceinline__ Tri tri_op(Tri a, Tri b) { return {a.neg + b.neg, max(a.rs, b.rs), max(a.gs, b.gs)}; }
__device__ __forceinline__ Tri tri_shfl_up(Tri v, int o) {
    return {__shfl_up_sync(kFull, v.neg, o), __shfl_up_sync(kFull, v.rs, o), __shfl_up_sync(kFull, v.gs, o)};
}
constexpr Tri kTriZero = {0, -1, -1};

// Exclusive block scan of one Tri per thread; *total gets the whole block's.  wsum: shared [kWarps].
template <int kWarps>
__device__ __forceinline__ Tri block_scan_tri(Tri v, Tri* wsum, Tri* total) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    Tri inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const Tri u = tri_shfl_up(inc, o);
        if (lane >= o) inc = tri_op(u, inc);
    }
    Tri prev = tri_shfl_up(inc, 1);
    if (lane == 0) prev = kTriZero;
    if (lane == 31) wsum[w] = inc;
    __syncthreads();
    Tri before = kTriZero, all = kTriZero;
    for (int k = 0; k < kWarps; ++k) {
        if (k < w) before = tri_op(before, wsum[k]);
        all = tri_op(all, wsum[k]);
    }
    *total = all;
    __syncthreads();
    return tri_op(before, prev);
}

struct TileAgg {     // per tile: negatives; global position of its last run / group start (-1: none)
    int32_t neg, rs, rs_neg, gs, gs_neg;   // *_neg: the tile's negatives before that start
};
struct TileCarry {   // per tile, over every earlier position: NC, RS, NRS, GS, NGS
    int32_t nc, rs, nrs, gs, ngs;
};

// kFinal = false: write the tile's aggregate.  kFinal = true: with the tile's carry, compute every
// position's contribution and add each group segment of the tile to u2 / pos / neg [group].
template <bool kFinal>
__global__ void __launch_bounds__(kRunThreads)
auc_tile_kernel(const uint32_t* __restrict__ key, const uint32_t* __restrict__ gl, int64_t n,
                TileAgg* __restrict__ agg, const TileCarry* __restrict__ carry,
                unsigned long long* u2, unsigned long long* pos, unsigned long long* neg) {
    __shared__ uint32_t sh_nc[kMetricTile];                       // the tile's negatives before each position
    __shared__ unsigned long long sh_c[kFinal ? kMetricTile : 1];   // inclusive prefix of the contributions
    __shared__ Tri wsum[kRunWarps];
    __shared__ unsigned long long wsum_c[kRunWarps];
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    const int64_t base = (int64_t)blockIdx.x * kMetricTile;
    const int64_t j0 = base + (int64_t)kPer * t;

    uint32_t k[kPer + 2], g[kPer + 2];   // positions j0-1 .. j0+kPer: the neighbours decide the boundaries
#pragma unroll
    for (int e = 0; e < kPer + 2; ++e) {
        const int64_t j = j0 - 1 + e;
        const bool in = j >= 0 && j < n;
        k[e] = in ? key[j] : 0u;
        g[e] = in ? gl[j] : 0u;
    }
    bool is_neg[kPer], is_rs[kPer], is_gs[kPer];
    Tri mine = kTriZero;
#pragma unroll
    for (int e = 0; e < kPer; ++e) {
        const int64_t j = j0 + e;
        const bool valid = j < n;
        is_gs[e]  = valid && (j == 0 || (g[e + 1] >> 1) != (g[e] >> 1));
        is_rs[e]  = valid && (is_gs[e] || k[e + 1] != k[e]);
        is_neg[e] = valid && !(g[e + 1] & 1u);
        mine.neg += is_neg[e];
        if (is_rs[e]) mine.rs = (int32_t)j;
        if (is_gs[e]) mine.gs = (int32_t)j;
    }
    Tri total;
    const Tri ex = block_scan_tri<kRunWarps>(mine, wsum, &total);
    int32_t nc[kPer], rs[kPer], gs[kPer];   // in-tile: negatives before, last run / group start (-1: before the tile)
    {
        Tri run = ex;
#pragma unroll
        for (int e = 0; e < kPer; ++e) {
            nc[e] = run.neg;
            sh_nc[kPer * t + e] = (uint32_t)run.neg;
            if (is_rs[e]) run.rs = (int32_t)(j0 + e);
            if (is_gs[e]) run.gs = (int32_t)(j0 + e);
            rs[e] = run.rs;
            gs[e] = run.gs;
            run.neg += is_neg[e];
        }
    }
    __syncthreads();
    if (!kFinal) {
        if (t == 0) {
            TileAgg a;
            a.neg    = total.neg;
            a.rs     = total.rs;
            a.rs_neg = total.rs >= 0 ? (int32_t)sh_nc[total.rs - base] : 0;
            a.gs     = total.gs;
            a.gs_neg = total.gs >= 0 ? (int32_t)sh_nc[total.gs - base] : 0;
            agg[blockIdx.x] = a;
        }
        return;
    }

    const TileCarry cin = carry[blockIdx.x];
    uint32_t c[kPer];
    int32_t  NC[kPer], RS[kPer], NGS[kPer], GS[kPer];
    unsigned long long csum = 0;
#pragma unroll
    for (int e = 0; e < kPer; ++e) {
        const int32_t j = (int32_t)(j0 + e);
        NC[e]  = cin.nc + nc[e];
        RS[e]  = rs[e] >= 0 ? rs[e] : cin.rs;
        const int32_t NRS = rs[e] >= 0 ? cin.nc + (int32_t)sh_nc[rs[e] - base] : cin.nrs;
        GS[e]  = gs[e] >= 0 ? gs[e] : cin.gs;
        NGS[e] = gs[e] >= 0 ? cin.nc + (int32_t)sh_nc[gs[e] - base] : cin.ngs;
        const bool p = j < n && !is_neg[e];
        c[e] = j >= n ? 0u
             : p ? 2u * (uint32_t)(NRS - NGS[e]) + (uint32_t)(NC[e] - NRS)
                 : (uint32_t)(j - RS[e]) - (uint32_t)(NC[e] - NRS);
        csum += c[e];
    }
    {   // inclusive prefix of the contributions inside the tile
        unsigned long long inc = csum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long u = __shfl_up_sync(kFull, inc, o);
            if (lane >= o) inc += u;
        }
        if (lane == 31) wsum_c[w] = inc;
        __syncthreads();
        unsigned long long run = inc - csum;
        for (int ww = 0; ww < w; ++ww) run += wsum_c[ww];
#pragma unroll
        for (int e = 0; e < kPer; ++e) {
            run += c[e];
            sh_c[kPer * t + e] = run;
        }
    }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < kPer; ++e) {
        const int64_t j = j0 + e;
        if (j >= n) break;
        const bool seg_end = j == n - 1 || kPer * t + e == kMetricTile - 1 || (g[e + 2] >> 1) != (g[e + 1] >> 1);
        if (!seg_end) continue;
        // the segment: positions s .. j of one group inside this tile
        const int64_t s = GS[e] >= base ? GS[e] : base;
        const unsigned long long seg_c = sh_c[j - base] - (s > base ? sh_c[s - 1 - base] : 0ull);
        const int32_t seg_neg = NC[e] + (int32_t)is_neg[e] - (GS[e] >= base ? NGS[e] : cin.nc);
        const int32_t seg_pos = (int32_t)(j - s + 1) - seg_neg;
        const uint32_t grp = g[e + 1] >> 1;
        atomicAdd(u2 + grp, seg_c);
        atomicAdd(pos + grp, (unsigned long long)seg_pos);
        atomicAdd(neg + grp, (unsigned long long)seg_neg);
    }
}

// One CTA: exclusive scan of the tile aggregates into the tiles' carries.
__global__ void __launch_bounds__(kCarryThreads)
auc_carry_kernel(const TileAgg* __restrict__ agg, int tiles, TileCarry* carry) {
    __shared__ Tri wsum[kCarryThreads / 32];
    __shared__ Tri run_s;
    const int t = threadIdx.x;
    if (t == 0) run_s = kTriZero;
    __syncthreads();
    for (int b0 = 0; b0 < tiles; b0 += kCarryThreads) {
        const int i = b0 + t;
        Tri v = kTriZero;
        if (i < tiles) {
            const TileAgg a = agg[i];
            v = {a.neg, a.rs, a.gs};
        }
        Tri total;
        const Tri ex = tri_op(run_s, block_scan_tri<kCarryThreads / 32>(v, wsum, &total));
        if (i < tiles) carry[i] = {ex.neg, ex.rs, 0, ex.gs, 0};
        __syncthreads();
        if (t == 0) run_s = tri_op(run_s, total);
        __syncthreads();
    }
    // NRS / NGS: the negatives before that start = its tile's carry + the tile's negatives before it.
    // Global writes of this CTA are visible to it after the barrier above.
    for (int i = t; i < tiles; i += kCarryThreads) {
        const int32_t rs = carry[i].rs, gs = carry[i].gs;
        if (rs >= 0) carry[i].nrs = carry[rs / kMetricTile].nc + agg[rs / kMetricTile].rs_neg;
        if (gs >= 0) carry[i].ngs = carry[gs / kMetricTile].nc + agg[gs / kMetricTile].gs_neg;
    }
}

// One CTA: the ordered sums (log loss, correct count, uAUC over the valid groups) and the result.
__global__ void __launch_bounds__(kFinalThreads)
metrics_final_kernel(const double* __restrict__ ll_part, const unsigned long long* __restrict__ acc_part,
                     int n_parts, const unsigned long long* __restrict__ all, int64_t num_groups,
                     const unsigned long long* __restrict__ gu2, const unsigned long long* __restrict__ gpos,
                     const unsigned long long* __restrict__ gneg, rk_metrics_result_t* out) {
    __shared__ double sd[2][kFinalThreads];
    __shared__ unsigned long long su[2][kFinalThreads];
    const int t = threadIdx.x;
    double ll = 0.0, us = 0.0;
    unsigned long long acc = 0, valid = 0;
    for (int c = t; c < n_parts; c += kFinalThreads) {
        ll += ll_part[c];
        acc += acc_part[c];
    }
    // every thread sums a contiguous range of group ids in id order; the ranges are then added in a
    // fixed tree: the order depends on num_groups only
    const int64_t per = (num_groups + kFinalThreads - 1) / kFinalThreads;
    const int64_t g1  = min(num_groups, (t + 1) * per);
    for (int64_t g = t * per; g < g1; ++g) {
        const unsigned long long p = gpos[g], q = gneg[g];
        if (p > 0 && q > 0) {
            us += (double)gu2[g] / (2.0 * (double)p * (double)q);
            ++valid;
        }
    }
    sd[0][t] = ll; sd[1][t] = us; su[0][t] = acc; su[1][t] = valid;
    __syncthreads();
    for (int h = kFinalThreads / 2; h > 0; h >>= 1) {
        if (t < h) {
            sd[0][t] += sd[0][t + h]; sd[1][t] += sd[1][t + h];
            su[0][t] += su[0][t + h]; su[1][t] += su[1][t + h];
        }
        __syncthreads();
    }
    if (t == 0) {
        out->u2 = all[0];
        out->pos = all[1];
        out->neg = all[2];
        out->correct = su[0][0];
        out->logloss_sum = sd[0][0];
        out->valid_groups = su[1][0];
        out->uauc_sum = sd[1][0];
    }
}

// ---------------------------------------------------------------------------------------- merge
// Every CTA copies part of one rank's segment: rank r = blockIdx.x / ctas_per_rank.  It recomputes the
// segment's offset (the clamped counts of the ranks before r) from the world*3 state words, so the
// launch needs no scan of its own and no host value of any count.
constexpr int kMergeThreads = 256;
constexpr int kMergeMaxCtasPerRank = 1024;

__device__ __forceinline__ int64_t merge_count(const int64_t* state_g, int64_t r, int64_t cap) {
    const int64_t c = state_g[3 * r];
    return c < 0 ? 0 : (c > cap ? cap : c);
}

__global__ void __launch_bounds__(kMergeThreads)
metrics_merge_kernel(const float* __restrict__ score_g, const float* __restrict__ label_g,
                     const int64_t* __restrict__ group_g, const int64_t* __restrict__ state_g, int64_t world,
                     int64_t cap, int64_t ctas_per_rank, float* __restrict__ score_out,
                     float* __restrict__ label_out, int64_t* __restrict__ group_out, int64_t* __restrict__ state_out) {
    __shared__ int64_t off_w[kMergeThreads / 32];
    __shared__ uint32_t bits_w[kMergeThreads / 32];
    const int64_t r = blockIdx.x / ctas_per_rank, c = blockIdx.x % ctas_per_rank;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    // block 0 sums every rank (the merged count) and ORs every status; the others only the ranks before r
    const int64_t upto = blockIdx.x == 0 ? world : r;
    int64_t off = 0;
    uint32_t bits = 0;
    for (int64_t q = threadIdx.x; q < upto; q += kMergeThreads) {
        off += merge_count(state_g, q, cap);
        bits |= (uint32_t)state_g[3 * q + 2];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) off += __shfl_xor_sync(kFull, off, o);
    bits = __reduce_or_sync(kFull, bits);
    if (lane == 0) { off_w[w] = off; bits_w[w] = bits; }
    __syncthreads();
    off = 0;
    bits = 0;
#pragma unroll
    for (int k = 0; k < kMergeThreads / 32; ++k) { off += off_w[k]; bits |= bits_w[k]; }
    if (blockIdx.x == 0) {
        if (threadIdx.x == 0) {
            state_out[0] = off;
            state_out[1] = 0;
            state_out[2] = (int64_t)bits;
        }
        off = 0;   // rank 0's segment starts at 0
    }
    const int64_t n_r = merge_count(state_g, r, cap);
    const int64_t src = r * cap;
    for (int64_t i = c * kMergeThreads + threadIdx.x; i < n_r; i += ctas_per_rank * kMergeThreads) {
        score_out[off + i] = score_g[src + i];
        label_out[off + i] = label_g[src + i];
        if (group_g) group_out[off + i] = group_g[src + i];
    }
}

static size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

struct MetricsWs {
    uint32_t *k, *v, *sk, *sp;
    void* sort_ws;
    TileAgg* agg;
    TileCarry* carry;
    double* ll_part;
    unsigned long long *acc_part, *counters;
    size_t bytes;
};

static MetricsWs metrics_layout(char* base, int64_t n, int64_t num_groups) {
    const size_t arr = al256((size_t)n * 4);
    const size_t tiles = (size_t)ceil_div(n > 0 ? n : 1, kMetricTile);
    MetricsWs w;
    size_t o = 0;
    w.k = (uint32_t*)(base + o);  o += arr;
    w.v = (uint32_t*)(base + o);  o += arr;
    w.sk = (uint32_t*)(base + o); o += arr;
    w.sp = (uint32_t*)(base + o); o += arr;
    w.sort_ws = base + o;                         o += al256(radix_sort_ws_bytes(n));
    w.agg = (TileAgg*)(base + o);                 o += al256(tiles * sizeof(TileAgg));
    w.carry = (TileCarry*)(base + o);             o += al256(tiles * sizeof(TileCarry));
    w.ll_part = (double*)(base + o);              o += al256(tiles * 8);
    w.acc_part = (unsigned long long*)(base + o); o += al256(tiles * 8);
    w.counters = (unsigned long long*)(base + o); o += al256((size_t)(3 + 3 * num_groups) * 8);
    w.bytes = o;
    return w;
}

// Sorted order perm (and sorted group ids, or NULL) -> 2U, P, N of every group into u2/pos/neg.
static int auc_pass(const MetricsWs& w, const float* score, const float* label, const uint32_t* perm,
                    const uint32_t* group_sorted, int64_t n, unsigned long long* u2, unsigned long long* pos,
                    unsigned long long* neg, cudaStream_t s) {
    const int tiles = (int)ceil_div(n, kMetricTile);
    gather_sorted_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(score, label, perm, group_sorted, n, w.k, w.v);
    RK_LAUNCH_CHECK();
    auc_tile_kernel<false><<<tiles, kRunThreads, 0, s>>>(w.k, w.v, n, w.agg, nullptr, nullptr, nullptr, nullptr);
    RK_LAUNCH_CHECK();
    auc_carry_kernel<<<1, kCarryThreads, 0, s>>>(w.agg, tiles, w.carry);
    RK_LAUNCH_CHECK();
    auc_tile_kernel<true><<<tiles, kRunThreads, 0, s>>>(w.k, w.v, n, nullptr, w.carry, u2, pos, neg);
    RK_LAUNCH_CHECK();
    return 0;
}

}  // namespace rk

extern "C" {

int rk_metrics_append(const float* score, const float* label, const int64_t* group, int64_t B,
                      float* score_buf, float* label_buf, int64_t* group_buf, int64_t capacity,
                      int64_t num_groups, int64_t* count, uint32_t* status, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(B >= 0 && capacity >= 0 && capacity < (1ll << 31),
                 "rk_metrics_append: B=%lld capacity=%lld", (long long)B, (long long)capacity);
    RK_CHECK_ARG(count && status && score_buf && label_buf, "rk_metrics_append: NULL buffer");
    RK_CHECK_ARG(!group || (group_buf && num_groups >= 1), "rk_metrics_append: groups need group_buf and num_groups >= 1");
    if (B == 0) return 0;
    RK_CHECK_ARG(score && label, "rk_metrics_append: NULL score or label");
    const int grid = (int)(ceil_div(B, kAppendThreads) < kAppendMaxCtas ? ceil_div(B, kAppendThreads) : kAppendMaxCtas);
    metrics_append_kernel<<<grid, kAppendThreads, 0, (cudaStream_t)stream_>>>(
        score, label, group, B, score_buf, label_buf, group_buf, capacity, num_groups, count, status);
    RK_LAUNCH_CHECK();
    return 0;
}

size_t rk_metrics_workspace_bytes(int64_t n, int64_t num_groups) {
    return rk::metrics_layout(nullptr, n > 0 ? n : 0, num_groups > 0 ? num_groups : 0).bytes;
}

int rk_metrics_compute(const float* score, const float* label, const int64_t* group, int64_t n,
                       int64_t num_groups, void* ws, size_t ws_bytes, rk_metrics_result_t* result,
                       rk_stream_t stream_) {
    using namespace rk;
    cudaStream_t s = (cudaStream_t)stream_;
    RK_CHECK_ARG(n >= 0 && n < (1ll << 31), "rk_metrics_compute: n=%lld outside [0, 2^31)", (long long)n);
    RK_CHECK_ARG(!group || (num_groups >= 1 && num_groups < (1ll << 31)),
                 "rk_metrics_compute: num_groups=%lld outside [1, 2^31)", (long long)num_groups);
    RK_CHECK_ARG(result, "rk_metrics_compute: NULL result");
    const int64_t G = group ? num_groups : 0;
    if (n == 0) {
        RK_CUDA(cudaMemsetAsync(result, 0, sizeof(rk_metrics_result_t), s));
        return 0;
    }
    RK_CHECK_ARG(score && label && ws, "rk_metrics_compute: NULL input or workspace");
    RK_CHECK_ARG(ws_bytes >= rk_metrics_workspace_bytes(n, G), "rk_metrics_compute: workspace %zu < %zu bytes",
                 ws_bytes, rk_metrics_workspace_bytes(n, G));
    const MetricsWs w = metrics_layout((char*)ws, n, G);
    unsigned long long* all = w.counters;   // [2U, P, N] of the whole set, then per group
    unsigned long long* gu2 = all + 3;
    RK_CUDA(cudaMemsetAsync(all, 0, (size_t)(3 + 3 * G) * 8, s));
    const int tiles = (int)ceil_div(n, kMetricTile);

    metrics_key_kernel<<<tiles, kKeyThreads, 0, s>>>(score, label, n, w.k, w.v, w.ll_part, w.acc_part);
    RK_LAUNCH_CHECK();
    int rc = radix_sort_u32(w.k, w.v, w.sk, w.sp, n, 32, w.sort_ws, s);
    if (rc) return rc;
    rc = auc_pass(w, score, label, w.sp, nullptr, n, all, all + 1, all + 2, s);
    if (rc) return rc;
    if (G > 0) {
        group_key_kernel<<<(unsigned)ceil_div(n, 256), 256, 0, s>>>(group, w.sp, n, G, w.k, w.v);
        RK_LAUNCH_CHECK();
        int bits = 1;
        while ((1ll << bits) < G) ++bits;
        rc = radix_sort_u32(w.k, w.v, w.sk, w.sp, n, bits, w.sort_ws, s);
        if (rc) return rc;
        rc = auc_pass(w, score, label, w.sp, w.sk, n, gu2, gu2 + G, gu2 + 2 * G, s);
        if (rc) return rc;
    }
    metrics_final_kernel<<<1, kFinalThreads, 0, s>>>(w.ll_part, w.acc_part, tiles, all, G, gu2, gu2 + G,
                                                      gu2 + 2 * G, result);
    RK_LAUNCH_CHECK();
    return 0;
}

int rk_metrics_merge(const float* score_g, const float* label_g, const int64_t* group_g, const int64_t* state_g,
                     int64_t world, int64_t capacity, float* score_out, float* label_out, int64_t* group_out,
                     int64_t* state_out, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(world >= 1 && capacity >= 1 && world <= ((1ll << 31) - 1) / capacity,
                 "rk_metrics_merge: world=%lld capacity=%lld (need >= 1 each and world*capacity < 2^31)",
                 (long long)world, (long long)capacity);
    RK_CHECK_ARG(score_g && label_g && state_g && score_out && label_out && state_out,
                 "rk_metrics_merge: NULL buffer");
    RK_CHECK_ARG(!group_g || group_out, "rk_metrics_merge: group_g needs group_out");
    RK_CHECK_ARG(state_out + 3 <= state_g || state_out >= state_g + 3 * world,
                 "rk_metrics_merge: state_out overlaps state_g");
    const int64_t per = ceil_div(capacity, kMergeThreads);
    const int64_t ctas_per_rank = per < kMergeMaxCtasPerRank ? per : kMergeMaxCtasPerRank;
    metrics_merge_kernel<<<(unsigned)(world * ctas_per_rank), kMergeThreads, 0, (cudaStream_t)stream_>>>(
        score_g, label_g, group_g, state_g, world, capacity, ctas_per_rank, score_out, label_out, group_out,
        state_out);
    RK_LAUNCH_CHECK();
    return 0;
}

}  // extern "C"
