// batch.cu — one training batch gathered on the device from an encoded frame resident in HBM.
// Replaces each script's WechatDataset.__getitem__ + DataLoader collation (DIN/din.py:86-222 with
// din_collate_fn's padding, BST/bst.py:94-159, DCN/dcn.py:52-112, DeepFM/deepfm.py:26-70), which
// rank_b200.loader.EncodedWechat does with numpy fancy indexing on one host thread.
//
// Output row i of every column is source row order[*cursor + row0 + i].  Bytes are copied, never
// converted.  A plain column is cut into units of 16, 8, 4 or 1 bytes (the widest that divides the
// row and both base addresses); consecutive threads take consecutive units of the output, so the
// writes are coalesced and a row of several units is read by neighbouring threads.  The ragged DIN
// history is one unit per int64 of the padded [B, width] output.  Every column and the history are
// one launch: a CTA finds its column from the prefix of per-column CTA counts.  The bound is the
// latency of the random row reads (each thread keeps kPer independent loads in flight).
#include <string.h>
#include "common.cuh"

namespace rk {

constexpr int kGatherThreads = 256;
constexpr int kPer = 4;                                   // units per thread, loads issued before stores
constexpr int kUnitsPerCta = kGatherThreads * kPer;

struct GatherJob {
    const void*    src;      // plain: [n_rows, units_per_row] units; history: the flat ids
    void*          dst;      // plain: [B, units_per_row] units; history: [B, width] int64
    const int64_t* offsets;  // history only: [n_rows + 1]
    int64_t*       dst_len;  // history only: [B]
    int64_t        units_per_row;
    int64_t        units;
    int32_t        unit_bytes;  // 16, 8, 4 or 1; 0 marks the history
    int32_t        cta_start;
};

struct GatherParams {
    GatherJob      job[RK_BATCH_MAX_COLS + 1];
    int32_t        n;
    const int64_t* order;
    int64_t        n_order, n_rows, row0, B;
    const int64_t* cursor;
    uint32_t*      status;
};

template <typename U>
__device__ __forceinline__ void gather_plain(const GatherJob& j, const GatherParams& P, int64_t base, int64_t u0) {
    const U* __restrict__ src = static_cast<const U*>(j.src);
    U* __restrict__ dst = static_cast<U*>(j.dst);
    U v[kPer];
    bool bad = false;
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        const int64_t u = u0 + k * kGatherThreads;
        if (u >= j.units) break;
        const int64_t i = u / j.units_per_row;
        const int64_t r = __ldg(P.order + base + i);
        if ((uint64_t)r >= (uint64_t)P.n_rows) {          // the row is written as zeros
            bad = true;
            memset(&v[k], 0, sizeof(U));
        } else {
            v[k] = src[r * j.units_per_row + (u - i * j.units_per_row)];
        }
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        const int64_t u = u0 + k * kGatherThreads;
        if (u < j.units) dst[u] = v[k];
    }
    if (bad) atomicOr(P.status, RK_BATCH_BAD_ROW);
}

__device__ __forceinline__ void gather_history(const GatherJob& j, const GatherParams& P, int64_t base, int64_t u0) {
    const int64_t* __restrict__ values = static_cast<const int64_t*>(j.src);
    int64_t* __restrict__ dst = static_cast<int64_t*>(j.dst);
    const int64_t width = j.units_per_row;
    int64_t v[kPer];
    uint32_t bits = 0;
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        const int64_t u = u0 + k * kGatherThreads;
        v[k] = 0;
        if (u >= j.units) break;
        const int64_t i = u / width, t = u - i * width;
        const int64_t r = __ldg(P.order + base + i);
        int64_t first = 0, len = 0;
        if ((uint64_t)r >= (uint64_t)P.n_rows) {
            bits |= RK_BATCH_BAD_ROW;
        } else {
            first = __ldg(j.offsets + r);
            len = __ldg(j.offsets + r + 1) - first;
        }
        if (t == 0) {
            if (len > width) bits |= RK_BATCH_SEQ_OVERFLOW;
            j.dst_len[i] = len < width ? len : width;      // the ids kept, so a reader never passes width
        }
        if (t < len) v[k] = __ldg(values + first + t);
    }
#pragma unroll
    for (int k = 0; k < kPer; ++k) {
        const int64_t u = u0 + k * kGatherThreads;
        if (u < j.units) dst[u] = v[k];
    }
    if (bits) atomicOr(P.status, bits);
}

__global__ void __launch_bounds__(kGatherThreads)
batch_gather_kernel(const __grid_constant__ GatherParams P) {
    const int64_t cur = *(volatile const int64_t*)P.cursor;
    const int64_t base = cur + P.row0;
    if (cur < 0 || base > P.n_order - P.B) {             // the whole batch must lie inside order
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(P.status, RK_BATCH_WINDOW);
        return;
    }
    int jn = 0;
    while (jn + 1 < P.n && P.job[jn + 1].cta_start <= (int)blockIdx.x) ++jn;
    const GatherJob& j = P.job[jn];
    const int64_t u0 = (int64_t)(blockIdx.x - j.cta_start) * kUnitsPerCta + threadIdx.x;
    switch (j.unit_bytes) {
        case 16: gather_plain<uint4>(j, P, base, u0); break;
        case 8:  gather_plain<uint2>(j, P, base, u0); break;
        case 4:  gather_plain<uint32_t>(j, P, base, u0); break;
        case 1:  gather_plain<uint8_t>(j, P, base, u0); break;
        default: gather_history(j, P, base, u0); break;
    }
}

}  // namespace rk

static_assert(sizeof(rk_batch_col_t) == 24, "rk_batch_col_t layout (mirrored by _lib.RkBatchCol)");
static_assert(sizeof(rk_batch_seq_t) == 40, "rk_batch_seq_t layout (mirrored by _lib.RkBatchSeq)");

extern "C" int rk_batch_gather(const rk_batch_col_t* cols, int n_cols, const rk_batch_seq_t* seq,
                               const int64_t* order, int64_t n_order, int64_t n_rows, const int64_t* cursor,
                               int64_t row0, int64_t B, uint32_t* status, rk_stream_t stream_) {
    using namespace rk;
    RK_CHECK_ARG(n_cols >= 0 && n_cols <= RK_BATCH_MAX_COLS && (n_cols == 0 || cols),
                 "batch_gather: n_cols=%d (max %d)", n_cols, RK_BATCH_MAX_COLS);
    RK_CHECK_ARG(order && cursor && status, "batch_gather: NULL order / cursor / status");
    RK_CHECK_ARG(B > 0, "batch_gather: B=%lld", (long long)B);
    RK_CHECK_ARG(n_order >= 0 && n_rows >= 0 && row0 >= 0, "batch_gather: n_order=%lld n_rows=%lld row0=%lld",
                 (long long)n_order, (long long)n_rows, (long long)row0);
    GatherParams P;
    memset(&P, 0, sizeof(P));
    int64_t ctas = 0;
    auto add = [&](GatherJob& j) {
        j.units = B * j.units_per_row;
        j.cta_start = (int32_t)ctas;
        ctas += ceil_div(j.units, kUnitsPerCta);
    };
    for (int c = 0; c < n_cols; ++c) {
        const rk_batch_col_t& col = cols[c];
        RK_CHECK_ARG(col.src && col.dst, "batch_gather: column %d: NULL src / dst", c);
        RK_CHECK_ARG(col.row_bytes > 0 && col.row_bytes <= INT64_MAX / B / 2, "batch_gather: column %d: row_bytes=%lld",
                     c, (long long)col.row_bytes);
        int ub = 16;
        while (ub > 1 && ((uintptr_t)col.src % ub || (uintptr_t)col.dst % ub || col.row_bytes % ub)) ub >>= 1;
        if (ub == 2) ub = 1;                             // no 2-byte path: such columns go byte by byte
        GatherJob& j = P.job[P.n++];
        j.src = col.src;
        j.dst = col.dst;
        j.unit_bytes = ub;
        j.units_per_row = col.row_bytes / ub;
        add(j);
    }
    if (seq) {
        RK_CHECK_ARG(seq->values && seq->offsets && seq->dst && seq->dst_len,
                     "batch_gather: history: NULL values / offsets / dst / dst_len");
        RK_CHECK_ARG(seq->width > 0, "batch_gather: history width=%d", seq->width);
        GatherJob& j = P.job[P.n++];
        j.src = seq->values;
        j.dst = seq->dst;
        j.offsets = seq->offsets;
        j.dst_len = seq->dst_len;
        j.unit_bytes = 0;
        j.units_per_row = seq->width;
        add(j);
    }
    RK_CHECK_ARG(ctas < INT32_MAX, "batch_gather: %lld CTAs in one launch", (long long)ctas);
    if (P.n == 0) return 0;
    P.order = order;
    P.n_order = n_order;
    P.n_rows = n_rows;
    P.row0 = row0;
    P.B = B;
    P.cursor = cursor;
    P.status = status;
    batch_gather_kernel<<<(unsigned)ctas, kGatherThreads, 0, (cudaStream_t)stream_>>>(P);
    RK_LAUNCH_CHECK();
    return 0;
}
