// direct_reduce.cu — rk_embgrad_direct_reduce: dense [rows, dim] embedding gradients of tables read
// through a per-sample index column (n <= 8192 occurrences), in ONE launch, with no prior
// rk_plan_build and no pre-zeroed output.  Replaces ATen embedding_dense_backward (autograd of
// nn.Embedding, reached from loss.backward(), e.g. DCN/dcn.py:166, DeepFM/deepfm.py:170).
//
// Output-partitioned: every CTA owns up to 1024 consecutive rows of one table (about 384 occurrences: fewer rows
// for small tables whose rows are hit many times each).  It
//   1. writes zeros over its rows (the caller's gradient buffer needs no memset),
//   2. scans the WHOLE index column (<= 64 KB, L2-resident; every CTA of the table reads it) and
//      keeps the occurrences whose row falls into its range,
//   3. orders them by (row, occurrence) with one stable counting pass over its rows in shared memory
//      (warp-match ranking in occurrence order, as rk_plan_build's sort does),
//   4. sums every row's gradient rows in that order: short runs one after the other by a lane
//      group, runs of more than 32 occurrences by a warp / the whole CTA over fixed interleaved
//      slots folded by a fixed shuffle tree.
// No atomics on floats, no dependence on scheduling: the result is a function of the inputs only.
// Tables that share an index column (DeepFM / FwFM: first-order [rows,1] and second-order
// [rows,D] tables of a field) are one job with several outputs: the column is scanned and ordered once.
//
// HBM/L2-bound integer + float work: per table, n*8 B of indices per CTA (L2), n*dim*4 B of gradient
// rows once, rows*dim*4 B of output once.
#include <string.h>
#include "common.cuh"

namespace rk {

constexpr int kDirThreads = 256;
constexpr int kDirWarps   = kDirThreads / 32;
constexpr int kDirMaxN    = RK_DIRECT_MAX_N;             // 8192
constexpr int kDirRows    = 1024;                        // most rows per CTA = bins of the counting pass
constexpr int kDirRpt     = kDirRows / kDirThreads;      // rows per thread in the prefix step
constexpr int kDirOccBits = 13;                          // packed entry: local row << 13 | occurrence
constexpr int kDirMaxOut  = 3;
constexpr int kDirMaxJobs = RK_MAX_FIELDS;
constexpr int kSeqRun     = 8;                           // runs up to this length: one lane group, in order
constexpr int kWarpRun    = 128;                         // up to this: one warp; longer: the whole CTA
constexpr int kDirTarget  = 384;                         // occurrences a CTA should own on average
constexpr int kDirMaxDim  = 128;                         // widest table row

struct DirectOut {
    const float* g;
    float*       dw;
    int32_t      ld;
    int16_t      dim;
    int8_t       vec;
    int8_t       lanes;
};
struct DirectJob {
    const int64_t* idx;
    int32_t        n;
    int32_t        rows;
    int32_t        cta_start;
    int16_t        n_out;
    int16_t        rows_per_cta;   // power of two <= 256: fewer for small, densely hit tables (balance)
    DirectOut      out[kDirMaxOut];
};
struct DirectParams {
    DirectJob job[kDirMaxJobs];
    int32_t   n_jobs;
};

// Sum of the gradient rows of entries start+slot, start+slot+nslots, ... (< start+len), in that order.
template <int V>
__device__ __forceinline__ Vec<V> strided_sum(const uint32_t* __restrict__ ent, int start, int len, int slot,
                                              int nslots, const float* __restrict__ g, int64_t ld, int col) {
    constexpr uint32_t kOccMask = (1u << kDirOccBits) - 1u;
    Vec<V> acc;
    vec_zero(acc);
    int j = slot;
    for (; j + 7 * nslots < len; j += 8 * nslots) {                 // eight loads in flight
        Vec<V> q[8];
#pragma unroll
        for (int u = 0; u < 8; ++u)
            q[u].load_plain(g + (int64_t)(ent[start + j + u * nslots] & kOccMask) * ld + col);
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int e = 0; e < V; ++e) acc.v[e] += q[u].v[e];
    }
    if (j < len) {                                                  // up to seven more, loaded together
        Vec<V> q[7];
#pragma unroll
        for (int u = 0; u < 7; ++u) {
            vec_zero(q[u]);
            if (j + u * nslots < len) q[u].load_plain(g + (int64_t)(ent[start + j + u * nslots] & kOccMask) * ld + col);
        }
#pragma unroll
        for (int u = 0; u < 7; ++u)
            if (j + u * nslots < len) {
#pragma unroll
                for (int e = 0; e < V; ++e) acc.v[e] += q[u].v[e];
            }
    }
    return acc;
}

// The rows of this CTA's range that have occurrences, by run length: lists built once per CTA.
struct RunLists {
    uint16_t* short_rows;              // 1 .. kSeqRun occurrences
    uint16_t* mid_rows;                // kSeqRun+1 .. kWarpRun
    uint16_t* long_rows;               // more
    int*      n;                       // [3]: n_short, n_mid, n_long
};

// All rows of this CTA's range for one output table.  run_start[d] / run_len[d]: where local row d's
// occurrences sit in ent[].  red: [kDirWarps][kDirMaxDim] floats of scratch.
template <int V>
__device__ __forceinline__ void reduce_rows(const DirectOut& o, const uint32_t* __restrict__ ent,
                                            const uint32_t* __restrict__ run_start,
                                            const uint32_t* __restrict__ run_len, const RunLists& L, int row0,
                                            float* red) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int CL = o.lanes;                          // column lanes per row
    // ---- short runs: one lane group per row, occurrences added one after the other
    const int n_short = L.n[0], n_mid = L.n[1], n_long = L.n[2];
    for (int item = tid; item < n_short * CL; item += kDirThreads) {
        const int i = item / CL, cl = item - i * CL;
        const int d = L.short_rows[i];
        Vec<V> acc = strided_sum<V>(ent, (int)run_start[d], (int)run_len[d], 0, 1, o.g, o.ld, cl * V);
        acc.store(o.dw + (int64_t)(row0 + d) * o.dim + cl * V);
    }
    // ---- medium runs: one warp per row, RL interleaved slots per column lane, fixed shuffle tree
    int RL = 1;
    while (RL * 2 * CL <= 32) RL *= 2;
    const int rl = lane / CL, cl = lane - rl * CL;
    const bool on = rl < RL;
    for (int i = warp; i < n_mid; i += kDirWarps) {
        const int d = L.mid_rows[i];
        Vec<V> acc;
        vec_zero(acc);
        if (on) acc = strided_sum<V>(ent, (int)run_start[d], (int)run_len[d], rl, RL, o.g, o.ld, cl * V);
        for (int s = RL >> 1; s > 0; s >>= 1) {
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const float other = __shfl_down_sync(kFull, acc.v[e], s * CL);
                if (on && rl < s) acc.v[e] += other;
            }
        }
        if (on && rl == 0) acc.store(o.dw + (int64_t)(row0 + d) * o.dim + cl * V);
    }
    // ---- long runs (a few per CTA): all warps, warp w takes slots [w*RL, (w+1)*RL) of 8*RL
    for (int i = 0; i < n_long; ++i) {                         // uniform over the CTA
        const int d = L.long_rows[i];
        Vec<V> acc;
        vec_zero(acc);
        if (on) acc = strided_sum<V>(ent, (int)run_start[d], (int)run_len[d], warp * RL + rl, kDirWarps * RL, o.g, o.ld, cl * V);
        for (int s = RL >> 1; s > 0; s >>= 1) {
#pragma unroll
            for (int e = 0; e < V; ++e) {
                const float other = __shfl_down_sync(kFull, acc.v[e], s * CL);
                if (on && rl < s) acc.v[e] += other;
            }
        }
        if (on && rl == 0) {
#pragma unroll
            for (int e = 0; e < V; ++e) red[warp * kDirMaxDim + cl * V + e] = acc.v[e];
        }
        __syncthreads();
        if (warp == 0 && lane < CL) {
            Vec<V> tot;
            vec_zero(tot);
            for (int ww = 0; ww < kDirWarps; ++ww) {
#pragma unroll
                for (int e = 0; e < V; ++e) tot.v[e] += red[ww * kDirMaxDim + lane * V + e];
            }
            tot.store(o.dw + (int64_t)(row0 + d) * o.dim + lane * V);
        }
        __syncthreads();
    }
}

// shared memory: staged[8192] | ent[8192] (u32) | rank[8192] (u16) | cnt[warps][R] (u16) | run_start[R] | run_len[R] |
// three row lists [R] (u16)
constexpr size_t kDirSmemBytes = 2 * sizeof(uint32_t) * kDirMaxN + sizeof(uint16_t) * kDirMaxN +
                                 sizeof(uint16_t) * kDirWarps * kDirRows + 2 * sizeof(uint32_t) * kDirRows +
                                 3 * sizeof(uint16_t) * kDirRows;

__global__ void __launch_bounds__(kDirThreads, 2)
direct_reduce_kernel(const __grid_constant__ DirectParams p, int32_t* err_flag) {
    extern __shared__ __align__(16) uint8_t dir_smem[];
    uint32_t* staged    = reinterpret_cast<uint32_t*>(dir_smem);               // compacted, occurrence order, per warp
    uint32_t* ent       = staged + kDirMaxN;                                   // ordered by (row, occurrence)
    uint16_t* rank      = reinterpret_cast<uint16_t*>(ent + kDirMaxN);         // rank of staged[i] inside its warp's part
    uint16_t* cnt       = rank + kDirMaxN;                                     // [warps][R]
    uint32_t* run_start = reinterpret_cast<uint32_t*>(cnt + kDirWarps * kDirRows);
    uint32_t* run_len   = run_start + kDirRows;
    RunLists lists;
    lists.short_rows = reinterpret_cast<uint16_t*>(run_len + kDirRows);
    lists.mid_rows   = lists.short_rows + kDirRows;
    lists.long_rows  = lists.mid_rows + kDirRows;
    __shared__ int      list_n[3];
    __shared__ uint32_t warp_tot[kDirWarps];
    lists.n = list_n;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int j = 0;
#pragma unroll 1
    while (j + 1 < p.n_jobs && (int)blockIdx.x >= p.job[j + 1].cta_start) ++j;
    const DirectJob& jb = p.job[j];
    const int R      = jb.rows_per_cta;          // power of two, 1 .. kDirRows
    const int row0   = ((int)blockIdx.x - jb.cta_start) * R;
    const int n_rows = jb.rows - row0 < R ? jb.rows - row0 : R;
    const int n      = jb.n;

    // 1. zeros over this CTA's rows of every output (fire and forget; the sums land after a barrier)
    for (int q = 0; q < jb.n_out; ++q) {
        const DirectOut& o = jb.out[q];
        float* base = o.dw + (int64_t)row0 * o.dim;
        const int total = n_rows * o.dim;
        if (o.vec == 4) {
            for (int i = tid * 4; i < total; i += kDirThreads * 4)
                *reinterpret_cast<float4*>(base + i) = make_float4(0.f, 0.f, 0.f, 0.f);
        } else {
            for (int i = tid; i < total; i += kDirThreads) base[i] = 0.f;
        }
    }
    for (int i = tid; i < kDirWarps * R / 2; i += kDirThreads) reinterpret_cast<uint32_t*>(cnt)[i] = 0;
    if (tid < 3) list_n[tid] = 0;

    // 2. the whole index column, warp-blocked so that (warp, round, lane) order = occurrence order; the
    //    occurrences that fall into this CTA's rows are compacted, in that order, into the warp's part of
    //    staged[] as (local row << 13 | occurrence)
    const int per_warp = ((n + kDirWarps * 32 - 1) / (kDirWarps * 32)) * 32;     // multiple of 32
    const int wbase    = warp * per_warp;
    const unsigned lt  = (1u << lane) - 1u;
    const int64_t* col = jb.idx;
    const int64_t rows64 = jb.rows;
    int wcount = 0;
#pragma unroll 1
    for (int h = 0; h < per_warp; h += 16 * 32) {         // 16 index loads in flight per thread
        int64_t raw[16];
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int i = wbase + h + r * 32 + lane;
            raw[r] = (h + r * 32 < per_warp && i < n) ? __ldg(col + i) : 0;
        }
#pragma unroll
        for (int r = 0; r < 16; ++r) {
            const int i = wbase + h + r * 32 + lane;
            bool mine = false;
            uint32_t key = 0;
            if (h + r * 32 < per_warp && i < n) {
                const int64_t row = checked_row(raw[r], rows64, err_flag);
                const int64_t d = row - row0;
                if (d >= 0 && d < n_rows) { mine = true; key = ((uint32_t)d << kDirOccBits) | (uint32_t)i; }
            }
            const unsigned bal = __ballot_sync(kFull, mine);
            if (mine) staged[wbase + wcount + __popc(bal & lt)] = key;
            wcount += __popc(bal);
        }
    }
    if (lane == 0) warp_tot[warp] = (uint32_t)wcount;
    __syncthreads();          // cnt is zero, the warp totals are known (each warp ranks its own part: no staging hazard)

    // 3. stable rank inside the warp's part of the compacted sequence
    uint16_t* my_cnt = cnt + warp * R;
#pragma unroll 1
    for (int e = lane; e - lane < wcount; e += 32) {
        const bool valid = e < wcount;
        const uint32_t d = valid ? staged[wbase + e] >> kDirOccBits : 0u;
        const uint32_t tag = valid ? d : (0x10000u | lane);       // the padding matches nobody
        const unsigned mm  = __match_any_sync(kFull, tag);
        const uint32_t old = valid ? my_cnt[d] : 0u;
        __syncwarp();
        if (valid && (mm & lt) == 0) my_cnt[d] = (uint16_t)(old + __popc(mm));
        __syncwarp();
        if (valid) rank[wbase + e] = (uint16_t)(old + __popc(mm & lt));
    }
    __syncthreads();

    // 4. per row: exclusive prefix over the warps; exclusive scan over the rows (thread = R/256 consecutive rows)
    {
        const int rpt = R >= kDirThreads ? R / kDirThreads : 1;
        uint32_t tot[kDirRpt];
        uint32_t mine = 0;
#pragma unroll
        for (int u = 0; u < kDirRpt; ++u) {
            tot[u] = 0;
            const int d = tid * rpt + u;
            if (u < rpt && d < R) {
                uint32_t t = 0;
#pragma unroll
                for (int ww = 0; ww < kDirWarps; ++ww) {
                    const uint32_t c = cnt[ww * R + d];
                    cnt[ww * R + d] = (uint16_t)t;
                    t += c;
                }
                tot[u] = t;
                mine += t;
            }
        }
        uint32_t inc = mine;
#pragma unroll
        for (int s = 1; s < 32; s <<= 1) {
            const uint32_t v = __shfl_up_sync(kFull, inc, s);
            if (lane >= s) inc += v;
        }
        __shared__ uint32_t scan_tot[kDirWarps];
        if (lane == 31) scan_tot[warp] = inc;
        __syncthreads();
        uint32_t run = inc - mine;
        for (int ww = 0; ww < warp; ++ww) run += scan_tot[ww];
#pragma unroll
        for (int u = 0; u < kDirRpt; ++u) {
            const int d = tid * rpt + u;
            if (u < rpt && d < R) {
                run_start[d] = run;
                run_len[d]   = tot[u];
                run += tot[u];
                // which rows have work, by run length (the order inside a list does not matter: rows are independent)
                if (tot[u] > (uint32_t)kWarpRun)     lists.long_rows[atomicAdd(&list_n[2], 1)] = (uint16_t)d;
                else if (tot[u] > (uint32_t)kSeqRun) lists.mid_rows[atomicAdd(&list_n[1], 1)] = (uint16_t)d;
                else if (tot[u] > 0)                 lists.short_rows[atomicAdd(&list_n[0], 1)] = (uint16_t)d;
            }
        }
    }
    __syncthreads();

    // 5. scatter into (row, occurrence) order
#pragma unroll 1
    for (int e = lane; e < wcount; e += 32) {
        const uint32_t key = staged[wbase + e];
        const uint32_t d = key >> kDirOccBits;
        ent[run_start[d] + my_cnt[d] + rank[wbase + e]] = key;
    }
    __syncthreads();          // also orders the zero stores of step 1 before the sums below

    // 6. the sums; the long runs' partial rows go where staged[] was (dead from here on)
    static_assert(kDirWarps * kDirMaxDim <= kDirMaxN, "long-run scratch");
    float* red = reinterpret_cast<float*>(staged);
    for (int q = 0; q < jb.n_out; ++q) {
        const DirectOut& o = jb.out[q];
        if (o.vec == 4)      reduce_rows<4>(o, ent, run_start, run_len, lists, row0, red);
        else if (o.vec == 2) reduce_rows<2>(o, ent, run_start, run_len, lists, row0, red);
        else                 reduce_rows<1>(o, ent, run_start, run_len, lists, row0, red);
    }
}

}  // namespace rk

extern "C" {

int rk_embgrad_direct_reduce(const rk_direct_table_t* tables, int n_tables, int32_t* err_flag,
                             rk_stream_t stream_) {
    using namespace rk;
    cudaStream_t s = (cudaStream_t)stream_;
    RK_CHECK_ARG(tables && n_tables >= 1 && n_tables <= RK_MAX_TABLES, "direct_reduce: n_tables=%d", n_tables);
    DirectParams p;
    memset(&p, 0, sizeof(p));
    int ctas = 0;
    auto flush = [&]() -> int {
        if (p.n_jobs == 0) return 0;
        RK_CUDA(cudaFuncSetAttribute(direct_reduce_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)kDirSmemBytes));      // per device: set on every call
        direct_reduce_kernel<<<ctas, kDirThreads, kDirSmemBytes, s>>>(p, err_flag);
        RK_LAUNCH_CHECK();
        memset(&p, 0, sizeof(p));
        ctas = 0;
        return 0;
    };
    for (int t = 0; t < n_tables; ++t) {
        const rk_direct_table_t& tb = tables[t];
        RK_CHECK_ARG(tb.dw && tb.rows > 0 && tb.dim > 0 && tb.dim <= kDirMaxDim && tb.n >= 0, "direct_reduce: table %d rows=%lld dim=%d n=%lld",
                     t, (long long)tb.rows, tb.dim, (long long)tb.n);
        RK_CHECK_ARG(tb.n <= kDirMaxN, "direct_reduce: table %d has %lld occurrences (max %d: use rk_plan_build + "
                     "rk_embgrad_segment_reduce)", t, (long long)tb.n, kDirMaxN);
        RK_CHECK_ARG(tb.rows < (1ll << 31) && tb.ld < (1ll << 31), "direct_reduce: table %d too large", t);
        RK_CHECK_ARG(tb.n == 0 || (tb.idx && tb.g), "direct_reduce: table %d NULL idx / g", t);
        int v = tb.dim % 4 == 0 ? 4 : (tb.dim % 2 == 0 ? 2 : 1);
        while (v > 1 && ((tb.ld % v) != 0 || ((uintptr_t)tb.g % (4 * v)) != 0 || ((uintptr_t)tb.dw % (4 * v)) != 0))
            v >>= 1;
        RK_CHECK_ARG(tb.dim / v <= 32, "direct_reduce: table %d dim %d too wide", t, tb.dim);
        DirectOut o;
        o.g = tb.g; o.dw = tb.dw; o.ld = (int32_t)tb.ld; o.dim = (int16_t)tb.dim; o.vec = (int8_t)v;
        o.lanes = (int8_t)(tb.dim / v);
        // same index column, height and length as an earlier table of this launch: one more output of that job
        int j = -1;
        for (int k = 0; k < p.n_jobs; ++k)
            if (p.job[k].idx == tb.idx && p.job[k].rows == (int32_t)tb.rows && p.job[k].n == (int32_t)tb.n &&
                p.job[k].n_out < kDirMaxOut) { j = k; break; }
        if (j < 0) {
            if (p.n_jobs == kDirMaxJobs) { int rc = flush(); if (rc) return rc; }
            j = p.n_jobs++;
            p.job[j].idx = tb.idx;
            p.job[j].n = (int32_t)tb.n;
            p.job[j].rows = (int32_t)tb.rows;
            p.job[j].cta_start = ctas;
            // rows per CTA: every CTA of a table scans the table's whole index column, so the fewer CTAs the
            // less redundant work; a CTA should own ~kDirTarget occurrences: up to 2048 rows of a large sparsely
            // hit table, a few rows of a small table whose rows are hit thousands of times each (balance)
            int R = 1;
            const double want = tb.n > 0 ? (double)tb.rows * (double)kDirTarget / (double)tb.n : (double)kDirRows;
            while (R < kDirRows && 2 * R <= want) R *= 2;
            p.job[j].rows_per_cta = (int16_t)R;
            ctas += (int)ceil_div(tb.rows, R);
        }
        p.job[j].out[p.job[j].n_out++] = o;
    }
    return flush();
}

}  // extern "C"
