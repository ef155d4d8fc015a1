// plan_sort.cu — rk_plan_build: stable LSD radix sort of every index occurrence of a batch
// by (field, row).  Replaces the sort inside ATen's embedding_dense_backward (reached from
// loss.backward(), e.g. DeepFM/deepfm.py:170, DIN/din.py:346); the order it produces makes the
// later segment reduction sum each row's gradients in occurrence order (deterministic,
// atomics-free).  Keys are uint32 = key_base[field] + row, where every field owns rows+1 keys
// (the last one parks padded history positions that carry no gradient); payload = occurrence
// number inside its field.  Fields sort independently into their own slice of the output.
//
// HBM/latency-bound integer work, two paths:
//   * every field has <= 8192 occurrences (all per-sample columns at batch <= 8192): ONE launch,
//     one 1024-thread CTA per field, the whole sort in shared memory (packed key|occurrence
//     words, up to 9-bit digits, warp-match ranking) — no global round trips between passes;
//   * otherwise (DIN/BST history columns, larger batches): one multi-CTA sort of ALL fields by the
//     global key — key building + first histogram, then per pass tile histogram, per-digit scan and
//     stable scatter with up to 10-bit digits — 6 launches for a 20-bit key space, independent of F.
#include <string.h>
#include "common.cuh"
#include "radix_sort.cuh"

namespace rk {

// --------------------------------------------------------------------------- shared pieces
struct FieldKeys {              // how to turn occurrence o of one field into its key
    const int64_t* idx;
    const int64_t* len;         // sequence fields: per-sample length, else NULL
    int64_t        n;           // occurrences
    int64_t        rows;
    int64_t        start;       // first slot of the field in sorted_keys / perm
    uint32_t       key_base;
    int32_t        T;
    int32_t        mode;        // RK_LIVE_*
    int32_t        bits;        // bits of rows (+ sentinel)
};

__device__ __forceinline__ uint32_t key_of(const FieldKeys& f, int64_t o, int64_t raw_index, int32_t* err_flag) {
    int64_t row = checked_row(raw_index, f.rows, err_flag);
    if (f.mode != RK_LIVE_ALL) {
        // padded history positions carry no gradient: park them on the field's sentinel row
        const int64_t b = o / f.T, t = o - b * f.T;
        const int64_t l = f.len[b];
        const bool dead = t >= l && !(f.mode == RK_LIVE_PREFIX_OR_EMPTY && l <= 0);
        if (dead) row = f.rows;
    }
    return (uint32_t)row;
}
__device__ __forceinline__ uint32_t local_key(const FieldKeys& f, int64_t o, int32_t* err_flag) {
    return key_of(f, o, f.idx[o], err_flag);
}

// --------------------------------------------------------------------------- small fields
constexpr int kSmallN       = 8192;
constexpr int kSmallThreads = 1024;
constexpr int kSmallWarps   = kSmallThreads / 32;
constexpr int kSmallRounds  = kSmallN / kSmallThreads;   // 8 keys per thread
constexpr int kSmallOccBits = 13;                        // occurrence number packed under the key
constexpr int kSmallMaxBits = 32 - kSmallOccBits;        // 19 key bits fit above the occurrence
constexpr int kSmallBins    = 512;                       // up to 9-bit digits

struct SmallBatch {
    FieldKeys f[RK_MAX_FIELDS];
};

__global__ void __launch_bounds__(kSmallThreads, 1)
small_field_sort_kernel(const __grid_constant__ SmallBatch batch, uint32_t* __restrict__ sorted_keys,
                        uint32_t* __restrict__ perm, int32_t* err_flag) {
    extern __shared__ __align__(16) uint32_t sm_u32[];
    uint32_t* buf0 = sm_u32;                       // [kSmallN] packed (key << 13 | occurrence)
    uint32_t* buf1 = sm_u32 + kSmallN;
    uint16_t* cnt  = reinterpret_cast<uint16_t*>(sm_u32 + 2 * kSmallN);   // [warps][bins]
    __shared__ uint32_t digit_base[kSmallBins];
    __shared__ uint32_t warp_tot[32];

    const FieldKeys& f = batch.f[blockIdx.x];
    const int tid = threadIdx.x, w = tid >> 5, lane = tid & 31;
    const int n = (int)f.n;
    {   // all of a thread's index loads in flight at once (the column is cold in HBM)
        int64_t raw[kSmallRounds];
#pragma unroll
        for (int r = 0; r < kSmallRounds; ++r) {
            const int i = tid + r * kSmallThreads;
            raw[r] = i < n ? __ldg(f.idx + i) : 0;
        }
#pragma unroll
        for (int r = 0; r < kSmallRounds; ++r) {
            const int i = tid + r * kSmallThreads;
            if (i < n) buf0[i] = (key_of(f, i, raw[r], err_flag) << kSmallOccBits) | (uint32_t)i;
        }
    }

    const int passes = (f.bits + 8) / 9;
    const int dbits  = (f.bits + passes - 1) / passes;
    const int bins   = 1 << dbits;
    const unsigned lt = (1u << lane) - 1u;
    uint32_t* in = buf0;
    uint32_t* out = buf1;
    for (int p = 0; p < passes; ++p) {
        const int shift = kSmallOccBits + p * dbits;
        for (int i = tid; i < kSmallWarps * bins / 2; i += kSmallThreads)
            reinterpret_cast<uint32_t*>(cnt)[i] = 0;
        __syncthreads();
        uint32_t key[kSmallRounds];
        uint16_t rank[kSmallRounds];
        const int wbase = w * (kSmallRounds * 32);
#pragma unroll
        for (int r = 0; r < kSmallRounds; ++r) key[r] = wbase + r * 32 + lane < n ? in[wbase + r * 32 + lane] : 0u;
#pragma unroll
        for (int r = 0; r < kSmallRounds; ++r) {
            const bool     valid = wbase + r * 32 + lane < n;   // the first n slots hold the keys
            const uint32_t d     = (key[r] >> shift) & (bins - 1);
            const uint32_t tag   = valid ? d : (kSmallBins | lane);   // padding matches nobody
            const unsigned m     = __match_any_sync(kFull, tag);
            const uint32_t old   = valid ? cnt[w * bins + d] : 0u;
            __syncwarp();
            if (valid && (m & lt) == 0) cnt[w * bins + d] = (uint16_t)(old + __popc(m));
            __syncwarp();
            rank[r] = (uint16_t)(old + __popc(m & lt));
        }
        __syncthreads();
        // per digit: exclusive prefix over the warps, then exclusive scan over the digits
        uint32_t tot = 0;
        if (tid < bins) {
            for (int ww = 0; ww < kSmallWarps; ++ww) {
                const uint32_t c = cnt[ww * bins + tid];
                cnt[ww * bins + tid] = (uint16_t)tot;
                tot += c;
            }
        }
        uint32_t inc = tot;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(kFull, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) warp_tot[w] = inc;
        __syncthreads();
        if (w == 0) {
            const uint32_t t = warp_tot[lane];
            uint32_t winc = t;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t v = __shfl_up_sync(kFull, winc, o);
                if (lane >= o) winc += v;
            }
            warp_tot[lane] = winc - t;
        }
        __syncthreads();
        if (tid < bins) digit_base[tid] = warp_tot[w] + inc - tot;
        __syncthreads();
#pragma unroll
        for (int r = 0; r < kSmallRounds; ++r) {
            if (wbase + r * 32 + lane < n) {
                const uint32_t d = (key[r] >> shift) & (bins - 1);
                out[digit_base[d] + cnt[w * bins + d] + rank[r]] = key[r];
            }
        }
        __syncthreads();
        uint32_t* t = in; in = out; out = t;
    }
    for (int i = tid; i < n; i += kSmallThreads) {
        const uint32_t v = in[i];
        sorted_keys[f.start + i] = f.key_base + (v >> kSmallOccBits);
        perm[f.start + i]        = v & ((1u << kSmallOccBits) - 1u);
    }
}

// --------------------------------------------------------------------------- large fields
constexpr int kSortThreads = 256;
constexpr int kSortWarps   = kSortThreads / 32;
constexpr int kSortRounds  = 8;
constexpr int kSortTile    = kSortThreads * kSortRounds;   // 2048 keys per CTA
constexpr int kMaxBins     = 1024;                         // up to 10-bit digits

__global__ void __launch_bounds__(kSortThreads)
tile_hist_kernel(const uint32_t* __restrict__ keys, int64_t n, int shift, int bins, int n_tiles,
                 uint32_t* __restrict__ hist) {
    __shared__ uint32_t h[kMaxBins];
    for (int i = threadIdx.x; i < bins; i += kSortThreads) h[i] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * kSortTile;
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int64_t i = base + r * kSortThreads + threadIdx.x;
        if (i < n) atomicAdd(&h[(keys[i] >> shift) & (bins - 1)], 1u);
    }
    __syncthreads();
    for (int d = threadIdx.x; d < bins; d += kSortThreads)
        hist[(int64_t)d * n_tiles + blockIdx.x] = h[d];
}

// Keys of ALL fields at once (global key = key_base[field] + row, payload = occurrence number inside
// its field), fused with the first pass's tile histogram (same tiling as tile_hist_kernel).  Sorting
// the concatenation by the global key sorts every field into its own slice, so the number of
// launches no longer grows with the number of fields.
__global__ void __launch_bounds__(kSortThreads)
build_keys_hist_kernel(const __grid_constant__ SmallBatch fields, int F, int64_t n_total, uint32_t* __restrict__ keys,
                       uint32_t* __restrict__ vals, int bins, int n_tiles, uint32_t* __restrict__ hist,
                       int32_t* err_flag) {
    __shared__ uint32_t h[kMaxBins];
    for (int i = threadIdx.x; i < bins; i += kSortThreads) h[i] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * kSortTile;
    int f = 0;
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int64_t i = base + r * kSortThreads + threadIdx.x;
        if (i < n_total) {
            while (f + 1 < F && i >= fields.f[f + 1].start) ++f;     // i grows with r: the search resumes where it was
            const FieldKeys& fk = fields.f[f];
            const int64_t o = i - fk.start;
            const uint32_t k = fk.key_base + local_key(fk, o, err_flag);
            keys[i] = k;
            vals[i] = (uint32_t)o;
            atomicAdd(&h[k & (bins - 1)], 1u);
        }
    }
    __syncthreads();
    for (int d = threadIdx.x; d < bins; d += kSortThreads)
        hist[(int64_t)d * n_tiles + blockIdx.x] = h[d];
}

// Per digit (one CTA each): exclusive scan of that digit's tile counts in place, and its total.
__global__ void __launch_bounds__(256)
row_scan_kernel(uint32_t* __restrict__ hist, int n_tiles, uint32_t* __restrict__ totals) {
    __shared__ uint32_t warp_tot[8];
    __shared__ uint32_t carry_s;
    uint32_t* row = hist + (int64_t)blockIdx.x * n_tiles;
    const int t = threadIdx.x, lane = t & 31, w = t >> 5;
    if (t == 0) carry_s = 0;
    __syncthreads();
    for (int base = 0; base < n_tiles; base += 256) {
        const int i = base + t;
        const uint32_t c = i < n_tiles ? row[i] : 0u;
        uint32_t inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(kFull, inc, o);
            if (lane >= o) inc += v;
        }
        if (lane == 31) warp_tot[w] = inc;
        __syncthreads();
        uint32_t before = carry_s;
        for (int ww = 0; ww < w; ++ww) before += warp_tot[ww];
        if (i < n_tiles) row[i] = before + inc - c;
        __syncthreads();
        if (t == 255) carry_s = before + inc;
        __syncthreads();
    }
    if (t == 0) totals[blockIdx.x] = carry_s;
}

// Stable scatter of one tile: ranks are taken in (warp, round, lane) = input order.  On the
// last pass the keys get their field base and land in the caller's slice.
__global__ void __launch_bounds__(kSortThreads)
scatter_kernel(const uint32_t* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
               uint32_t* __restrict__ keys_out, uint32_t* __restrict__ vals_out, int64_t n,
               int shift, int bins, int n_tiles, const uint32_t* __restrict__ hist_scanned,
               const uint32_t* __restrict__ totals, uint32_t add_base) {
    extern __shared__ uint32_t cnt[];   // [kSortWarps][bins]
    __shared__ uint32_t dbase[kMaxBins];   // keys with a smaller digit, over all tiles
    __shared__ uint32_t wsum[kSortWarps];
    const int t = threadIdx.x, w = t >> 5, lane = t & 31;
    for (int i = t; i < kSortWarps * bins; i += kSortThreads) cnt[i] = 0;
    {   // exclusive scan of the digit totals: 4 consecutive digits per thread
        uint32_t v[4], sum = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) { v[j] = 4 * t + j < bins ? totals[4 * t + j] : 0u; sum += v[j]; }
        uint32_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t x = __shfl_up_sync(kFull, inc, o);
            if (lane >= o) inc += x;
        }
        if (lane == 31) wsum[w] = inc;
        __syncthreads();
        uint32_t run = inc - sum;
        for (int ww = 0; ww < w; ++ww) run += wsum[ww];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (4 * t + j < bins) dbase[4 * t + j] = run;
            run += v[j];
        }
    }
    __syncthreads();

    const int64_t  wbase = (int64_t)blockIdx.x * kSortTile + (int64_t)w * (kSortRounds * 32);
    const unsigned lt    = (1u << lane) - 1u;
    uint32_t key[kSortRounds];
    uint16_t rank[kSortRounds];
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int64_t i = wbase + r * 32 + lane;
        key[r] = i < n ? keys_in[i] : 0u;
    }
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int64_t  i     = wbase + r * 32 + lane;
        const bool     valid = i < n;
        const uint32_t d     = (key[r] >> shift) & (bins - 1);
        const uint32_t tag   = valid ? d : (kMaxBins | lane);   // invalid lanes match nobody
        const unsigned m     = __match_any_sync(kFull, tag);
        const uint32_t old   = valid ? cnt[w * bins + d] : 0u;
        __syncwarp();
        if (valid && (m & lt) == 0) cnt[w * bins + d] = old + __popc(m);
        __syncwarp();
        rank[r] = (uint16_t)(old + __popc(m & lt));
    }
    __syncthreads();
    for (int d = t; d < bins; d += kSortThreads) {
        uint32_t run = dbase[d] + hist_scanned[(int64_t)d * n_tiles + blockIdx.x];
#pragma unroll
        for (int ww = 0; ww < kSortWarps; ++ww) {
            uint32_t c = cnt[ww * bins + d];
            cnt[ww * bins + d] = run;
            run += c;
        }
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < kSortRounds; ++r) {
        const int64_t i = wbase + r * 32 + lane;
        if (i < n) {
            const uint32_t d   = (key[r] >> shift) & (bins - 1);
            const uint32_t pos = cnt[w * bins + d] + rank[r];
            keys_out[pos] = key[r] + add_base;
            vals_out[pos] = vals_in[i];
        }
    }
}

static int bits_for(int64_t rows_plus_sentinel) {
    int bits = 1;
    while (bits < 32 && (1ull << bits) < (unsigned long long)rows_plus_sentinel) ++bits;
    return bits;
}
static bool is_small(int64_t n, int bits) { return n <= kSmallN && bits <= kSmallMaxBits; }
static size_t al256(size_t b) { return (b + 255) & ~(size_t)255; }

size_t radix_sort_ws_bytes(int64_t n) {
    const size_t tiles = (size_t)ceil_div(n > 0 ? n : 1, kSortTile);
    return 2 * al256((size_t)(n > 0 ? n : 0) * 4) + al256((tiles + 1) * kMaxBins * 4);
}

int radix_sort_u32(uint32_t* keys, uint32_t* vals, uint32_t* keys_out, uint32_t* vals_out, int64_t n,
                   int bits, void* ws, cudaStream_t s) {
    RK_CHECK_ARG(bits >= 1 && bits <= 32 && n >= 0 && n < (1ll << 31), "radix_sort_u32: n=%lld bits=%d",
                 (long long)n, bits);
    if (n == 0) return 0;
    const size_t arr = al256((size_t)n * 4);
    uint32_t* kT = (uint32_t*)ws;
    uint32_t* vT = (uint32_t*)((char*)ws + arr);
    uint32_t* hist = (uint32_t*)((char*)ws + 2 * arr);
    const int tiles  = (int)ceil_div(n, kSortTile);
    uint32_t* totals = hist + (size_t)tiles * kMaxBins;
    const int passes = (bits + 9) / 10;
    const int dbits  = (bits + passes - 1) / passes;
    const int bins   = 1 << dbits;
    uint32_t *kin = keys, *vin = vals;
    for (int p = 0; p < passes; ++p) {
        const bool last = p == passes - 1;
        uint32_t* kout = last ? keys_out : (kin == keys ? kT : keys);
        uint32_t* vout = last ? vals_out : (vin == vals ? vT : vals);
        tile_hist_kernel<<<tiles, kSortThreads, 0, s>>>(kin, n, p * dbits, bins, tiles, hist);
        RK_LAUNCH_CHECK();
        row_scan_kernel<<<bins, 256, 0, s>>>(hist, tiles, totals);
        RK_LAUNCH_CHECK();
        scatter_kernel<<<tiles, kSortThreads, (size_t)kSortWarps * bins * 4, s>>>(
            kin, vin, kout, vout, n, p * dbits, bins, tiles, hist, totals, 0u);
        RK_LAUNCH_CHECK();
        kin = kout;
        vin = vout;
    }
    return 0;
}

}  // namespace rk

extern "C" {

size_t rk_plan_workspace_bytes(int64_t n_total) {
    if (n_total < 0) n_total = 0;
    // sized for the large-field path: ping-pong keys + vals (n_total bounds the largest field)
    // and the tile histograms
    const size_t n     = (size_t)n_total;
    const size_t tiles = (size_t)rk::ceil_div(n_total > 0 ? n_total : 1, rk::kSortTile);
    return 4 * rk::al256(n * 4) + rk::al256((tiles + 1) * rk::kMaxBins * 4);   // + the digit totals
}

int rk_plan_build(const int64_t* const* idx, const int64_t* n, const int64_t* rows, int F,
                  const int64_t* const* seq_len, const int32_t* seq_T, const int32_t* live_mode,
                  uint32_t* sorted_keys, uint32_t* perm, void* ws, size_t ws_bytes,
                  int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    cudaStream_t s = (cudaStream_t)stream_;
    RK_CHECK_ARG(F >= 1 && F <= RK_MAX_FIELDS, "rk_plan_build: F=%d outside [1,%d]", F,
                 RK_MAX_FIELDS);
    RK_CHECK_ARG(idx && n && rows, "rk_plan_build: NULL host array");
    FieldKeys fk[RK_MAX_FIELDS];
    memset(fk, 0, sizeof(fk));
    int64_t total = 0, space = 0;
    for (int f = 0; f < F; ++f) {
        RK_CHECK_ARG(n[f] >= 0 && rows[f] > 0, "rk_plan_build: field %d n=%lld rows=%lld", f,
                     (long long)n[f], (long long)rows[f]);
        RK_CHECK_ARG(idx[f] != nullptr || n[f] == 0, "rk_plan_build: field %d idx is NULL", f);
        fk[f].idx      = idx[f];
        fk[f].n        = n[f];
        fk[f].rows     = rows[f];
        fk[f].start    = total;
        fk[f].key_base = (uint32_t)space;
        fk[f].bits     = bits_for(rows[f] + 1);
        fk[f].mode     = live_mode ? live_mode[f] : RK_LIVE_ALL;
        if (fk[f].mode != RK_LIVE_ALL) {
            RK_CHECK_ARG(fk[f].mode == RK_LIVE_PREFIX || fk[f].mode == RK_LIVE_PREFIX_OR_EMPTY,
                         "rk_plan_build: field %d live_mode %d", f, fk[f].mode);
            RK_CHECK_ARG(seq_len && seq_len[f] && seq_T && seq_T[f] > 0 && n[f] % seq_T[f] == 0,
                         "rk_plan_build: field %d needs lengths and T dividing n", f);
            fk[f].len = seq_len[f];
            fk[f].T   = seq_T[f];
        }
        total += n[f];
        space += rows[f] + 1;   // +1: the sentinel row of dead occurrences sorts last in the field
    }
    RK_CHECK_ARG(total < (1ll << 31) && space < (1ll << 32),
                 "rk_plan_build: %lld occurrences / %lld rows exceed the 32-bit key space",
                 (long long)total, (long long)space);
    if (total == 0) return 0;
    RK_CHECK_ARG(sorted_keys && perm && ws, "rk_plan_build: NULL output or workspace");
    RK_CHECK_ARG(ws_bytes >= rk_plan_workspace_bytes(total),
                 "rk_plan_build: workspace %zu < %zu bytes", ws_bytes,
                 rk_plan_workspace_bytes(total));

    // ---- every field fits one CTA's shared memory: one launch, one CTA per field
    bool all_small = true;
    for (int f = 0; f < F; ++f)
        if (n[f] > 0 && !is_small(n[f], fk[f].bits)) all_small = false;
    if (all_small) {
        SmallBatch small;
        int n_small = 0;
        for (int f = 0; f < F; ++f)
            if (n[f] > 0) small.f[n_small++] = fk[f];
        const size_t smem = 2 * (size_t)kSmallN * 4 + (size_t)kSmallWarps * kSmallBins * 2;
        // per call: the attribute belongs to the current DEVICE, a process may drive several
        RK_CUDA(cudaFuncSetAttribute(small_field_sort_kernel,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        small_field_sort_kernel<<<n_small, kSmallThreads, smem, s>>>(small, sorted_keys, perm, err_flag);
        RK_LAUNCH_CHECK();
        return 0;
    }

    // ---- otherwise ONE multi-CTA sort of all fields by the global key: 1 + 3 * passes - 1 launches
    // whatever the number of fields (DCN at batch 32768: 186 us with a sort per field, ~45 us like this)
    SmallBatch all;
    for (int f = 0; f < F; ++f) all.f[f] = fk[f];
    char* base = (char*)ws;
    const size_t arr = al256((size_t)total * 4);
    uint32_t* kA = (uint32_t*)base;
    uint32_t* vA = (uint32_t*)(base + arr);
    uint32_t* kB = (uint32_t*)(base + 2 * arr);
    uint32_t* vB = (uint32_t*)(base + 3 * arr);
    uint32_t* hist = (uint32_t*)(base + 4 * arr);
    uint32_t* totals = hist + (size_t)ceil_div(total, kSortTile) * kMaxBins;
    const int bits   = bits_for(space);
    const int passes = (bits + 9) / 10;
    const int dbits  = (bits + passes - 1) / passes;
    const int bins   = 1 << dbits;
    const int tiles  = (int)ceil_div(total, kSortTile);
    build_keys_hist_kernel<<<tiles, kSortThreads, 0, s>>>(all, F, total, kA, vA, bins, tiles, hist, err_flag);
    RK_LAUNCH_CHECK();
    uint32_t *kin = kA, *vin = vA;
    for (int p = 0; p < passes; ++p) {
        const bool last = p == passes - 1;
        uint32_t* kout = last ? sorted_keys : (kin == kA ? kB : kA);
        uint32_t* vout = last ? perm : (vin == vA ? vB : vA);
        if (p > 0) {                     // pass 0's histogram came with the keys
            tile_hist_kernel<<<tiles, kSortThreads, 0, s>>>(kin, total, p * dbits, bins, tiles, hist);
            RK_LAUNCH_CHECK();
        }
        row_scan_kernel<<<bins, 256, 0, s>>>(hist, tiles, totals);
        RK_LAUNCH_CHECK();
        scatter_kernel<<<tiles, kSortThreads, (size_t)kSortWarps * bins * 4, s>>>(
            kin, vin, kout, vout, total, p * dbits, bins, tiles, hist, totals, 0u);
        RK_LAUNCH_CHECK();
        kin = kout;
        vin = vout;
    }
    return 0;
}

}  // extern "C"
