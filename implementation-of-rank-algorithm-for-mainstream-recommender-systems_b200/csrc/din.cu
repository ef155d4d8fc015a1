// din.cu — DIN hot path: every gather of DIN.forward (DIN/din.py:294-305), the local activation
// unit din_attention (DIN/din.py:42-84), the concat (:310) and the per-sample L2 norm of the
// mini-batch-aware regulariser (:318-322), forward and backward.  fp32 SIMT at any history width
// T >= 0; the tensor-core activation unit further down takes T <= 128.
//
// One CTA owns kSamples consecutive samples.  Only history positions t < len feed the
// activation-unit MLP (padded positions get weight 0 in raw mode and exp(-2^32/sqrt(D)) = 0 in
// softmax mode, so their scores are never observable).  The CTA's live (b,t) rows are cut into
// tiles of at most kRows rows in sample order: whole samples while they fit (a sample with
// len <= kRows is never split, so short samples pack several to a tile), and a sample with
// len > kRows is cut at the tile edge and continues in the next tile.  Segment j of a tile = the
// rows of sample s_begin + j it holds.  Per tile:
//   gather   K rows (64 B each at D=16) -> shared memory, feature-major, with q, q-k, q*k
//   MLP      [rows,4D]x[4D,64] -> ReLU -> [rows,64]x[64,32] -> ReLU -> .w3   (tile_gemm.cuh)
//   pooling  one warp per segment:
//     raw      the pooled vector sum_t s_t k_t is accumulated segment after segment (fixed order)
//     softmax  online: per sample a running max m and sum S of exp(z - m); a segment with max m'
//              rescales (S, pooled) by exp(m - max(m, m')).  att_w holds the scaled scores z_t until
//              the sample's last segment, which rewrites them as exp(z_t - m) / S.
// The backward never needs dW of the unit (its weights are drawn per call and unregistered,
// DIN/din.py:61-67), so the forward keeps only the two ReLU masks as bits (12 B per row) and the
// weights w_t; the backward is g_score -> 32 -> 64 -> 4D through the transposed weights.  Its
// softmax term sum_u w_u (g_att . k_u) = g_att . pooled, and pooled is saved in concat_all, so
// every row's score gradient is local; g_q is summed segment after segment.
#include <string.h>
#include "common.cuh"
#include <cuda_bf16.h>
#include "tile_gemm.cuh"
#include "umma.cuh"
#include "prof.cuh"

namespace rk {

constexpr int kDinThreads = 256;
constexpr int kRows       = 128;   // (b,t) rows per MLP tile
constexpr int kSamples    = 8;     // samples per CTA
constexpr int kH1 = 64, kH2 = 32;
constexpr int kMaxDense   = 32;

struct DinParams {
    FieldSet       cat;                      // off = column in the concat row
    const float*   dense_col[kMaxDense];
    int64_t        dense_stride;
    int32_t        n_dense;
    const float*   tgt_w;  const int64_t* tgt_idx;  int64_t tgt_rows;  int32_t tgt_off;
    const float*   his_w;  const int64_t* his_idx;  int64_t his_rows;
    const int64_t* his_len;
    int32_t        T, D, att_off, width, l2_from, use_softmax;
    const float*   mlp;
    const uint8_t* mlp_tiles;               // operand tiles made once per forward (tensor-core path)
    int64_t        B;
};

// Offsets (floats) inside the packed per-call weights; K1 = 4*D.
struct MlpLayout {
    int w1t, b1, w2t, b2, w3, b3, w1, w2, total;
    __host__ __device__ explicit MlpLayout(int D) {
        const int K1 = 4 * D;
        w1t = 0;                 // [K1][64]   W1t[k][n] = W1[n][k]
        b1  = w1t + K1 * kH1;    // [64]
        w2t = b1 + kH1;          // [64][32]   W2t[k][n] = W2[n][k]
        b2  = w2t + kH1 * kH2;   // [32]
        w3  = b2 + kH2;          // [32]
        b3  = w3 + kH2;          // [1] (+3 pad)
        w1  = b3 + 4;            // [64][K1]   as registered: W1[n][k]
        w2  = w1 + kH1 * K1;     // [32][64]   W2[n][k]
        total = w2 + kH2 * kH1;
    }
};

// Shared-memory carve-up shared by forward and backward.
struct DinSmem {
    float *wA, *wB, *vec;          // weights: fwd (W1t, W2t) / bwd (W1, W2); vec = b1,b2,w3,b3
    float *x, *h1, *h2;            // [4D][kRows], [64][kRows], [32][kRows]
    float *score, *gw;             // [kRows]
    float *q, *gatt, *gq;          // [kSamples][D]
    int   *row_s, *row_t;          // row -> (local sample, t)
    int   *len;                    // [kSamples] clipped length
    float *run_max, *run_sum;      // [kSamples] softmax running max / sum (backward: run_sum = g_att . pooled)
    int   *seg_r0, *seg_t0;        // [kSamples + 1], [kSamples]: segment j = rows [seg_r0[j], seg_r0[j+1]),
                                   // positions seg_t0[j] + (row - seg_r0[j]) of sample s_begin + j
    int   *cursor;                 // [4] n_segments, n_rows, next sample, next position
    uint32_t* mask;                // [3][kRows] (backward)
    __device__ DinSmem(float* base, int D) {
        const int K1 = 4 * D;
        float* p = base;
        wA = p;     p += K1 * kH1;
        wB = p;     p += kH1 * kH2;
        vec = p;    p += 2 * kH1 + 2 * kH2 + 4;
        x = p;      p += K1 * kRows;
        h1 = p;     p += kH1 * kRows;
        h2 = p;     p += kH2 * kRows;
        score = p;  p += kRows;
        gw = p;     p += kRows;
        q = p;      p += kSamples * D;
        gatt = p;   p += kSamples * D;
        gq = p;     p += kSamples * D;
        row_s = (int*)p;  p += kRows;
        row_t = (int*)p;  p += kRows;
        len = (int*)p;    p += kSamples;
        run_max = p;      p += kSamples;
        run_sum = p;      p += kSamples;
        seg_r0 = (int*)p; p += kSamples + 1;
        seg_t0 = (int*)p; p += kSamples;
        cursor = (int*)p; p += 4;
        mask = (uint32_t*)p;  p += 3 * kRows;
    }
    static size_t bytes(int D) {
        const int K1 = 4 * D;
        return sizeof(float) * (size_t)(K1 * kH1 + kH1 * kH2 + 2 * kH1 + 2 * kH2 + 4 + K1 * kRows +
                                        kH1 * kRows + kH2 * kRows + 2 * kRows + 3 * kSamples * D +
                                        2 * kRows + 4 * kSamples + 1 + kSamples + 4 + 3 * kRows);
    }
};

template <int TN, class Epi>
__device__ __forceinline__ void tile_gemm_rows(const float* As, const float* Bs, int K, int N,
                                               int m_used, Epi epi) {
    tile_gemm<TN, kDinThreads>(As, kRows, Bs, N, K, N, m_used, epi);
}

// History positions that carry gradient / attention weight: t < len, or every t when len == 0 in
// softmax mode (all scores equal the padding value -> uniform weights 1/T, DIN/din.py:74-77).
__device__ __forceinline__ int clip_len(int64_t len, int T) {
    return len < 0 ? 0 : (len > T ? T : (int)len);
}

// Stage the K rows of a tile feature-major into x[D..2D), optionally with q, q-k, q*k.
template <bool FULL_CROSS>
__device__ __forceinline__ void stage_rows(const DinParams& p, const DinSmem& sm, int64_t b0,
                                           int n_rows, int32_t* err_flag) {
    const int D = p.D, D4 = D / 4;
    for (int item = threadIdx.x; item < D4 * kRows; item += kDinThreads) {
        const int c4 = item / kRows, m = item - c4 * kRows;
        float4 k = make_float4(0.f, 0.f, 0.f, 0.f), q = k;
        if (m < n_rows) {
            const int s = sm.row_s[m], t = sm.row_t[m];
            const int64_t row = checked_row(__ldg(p.his_idx + (b0 + s) * p.T + t), p.his_rows, err_flag);
            k = __ldg(reinterpret_cast<const float4*>(p.his_w + row * D) + c4);
            q = *reinterpret_cast<const float4*>(sm.q + s * D + c4 * 4);
        }
        const float kv[4] = {k.x, k.y, k.z, k.w}, qv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int c = c4 * 4 + e;
            sm.x[(D + c) * kRows + m] = kv[e];
            if (FULL_CROSS) {
                sm.x[c * kRows + m]           = qv[e];
                sm.x[(2 * D + c) * kRows + m] = qv[e] - kv[e];
                sm.x[(3 * D + c) * kRows + m] = qv[e] * kv[e];
            }
        }
    }
}

// Thread 0 plans the tile that starts at position t_begin of sample s_begin (tests/test_din_long.py
// restates this planner).
__device__ __forceinline__ void plan_tile(const DinSmem& sm, int n_samples, int s_begin, int t_begin) {
    int rows = 0, j = 0, s = s_begin, t0 = t_begin;
    while (s < n_samples) {
        const int rem = sm.len[s] - t0;
        if (rem <= kRows - rows) {                      // the rest of the sample fits
            sm.seg_r0[j] = rows;  sm.seg_t0[j] = t0;  ++j;
            rows += rem;  ++s;  t0 = 0;
            continue;
        }
        if (sm.len[s] <= kRows || rows == kRows) break;  // a short sample is never split
        sm.seg_r0[j] = rows;  sm.seg_t0[j] = t0;  ++j;   // a long one fills the tile
        t0 += kRows - rows;  rows = kRows;
        break;
    }
    sm.seg_r0[j] = rows;
    sm.cursor[0] = j;  sm.cursor[1] = rows;  sm.cursor[2] = s;  sm.cursor[3] = t0;
}

__device__ __forceinline__ void row_map(const DinSmem& sm, int n_seg, int s_begin) {
    for (int m = threadIdx.x; m < kRows; m += kDinThreads) {
        int j = 0;
        while (j + 1 < n_seg && m >= sm.seg_r0[j + 1]) ++j;
        sm.row_s[m] = s_begin + j;
        sm.row_t[m] = sm.seg_t0[j] + m - sm.seg_r0[j];
    }
}

// The activation unit on one staged tile: layers 1-3, scores -> sm.score, mask bits -> masks.
__device__ __forceinline__ void mlp_fwd(const DinParams& p, const DinSmem& sm, int64_t b0, int n_rows,
                                        uint32_t* masks) {
    const int K1 = 4 * p.D, tid = threadIdx.x;
    const float* b1 = sm.vec;
    const float* b2 = sm.vec + kH1;
    const float* w3 = sm.vec + kH1 + kH2;
    const float  b3 = sm.vec[kH1 + 2 * kH2];
    const int m_used = (n_rows + 3) / 4 * 4;
    tile_gemm_rows<8>(sm.x, sm.wA, K1, kH1, m_used, [&](int m0, int n0, float (&acc)[4][8]) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i][j] = fmaxf(acc[i][j] + b1[n0 + j], 0.f);
        store_tile_kmajor<8>(sm.h1, kRows, m0, n0, acc);
    });
    __syncthreads();
    tile_gemm_rows<4>(sm.h1, sm.wB, kH1, kH2, m_used, [&](int m0, int n0, float (&acc)[4][4]) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i][j] = fmaxf(acc[i][j] + b2[n0 + j], 0.f);
        store_tile_kmajor<4>(sm.h2, kRows, m0, n0, acc);
    });
    __syncthreads();
    if (tid < n_rows) {
        const int m = tid;
        float sc = b3;
        uint32_t m2 = 0, m1a = 0, m1b = 0;
#pragma unroll 8
        for (int n = 0; n < kH2; ++n) {
            const float h = sm.h2[n * kRows + m];
            sc = fmaf(h, w3[n], sc);
            m2 |= (h > 0.f ? 1u : 0u) << n;
        }
#pragma unroll 8
        for (int n = 0; n < 32; ++n) {
            m1a |= (sm.h1[n * kRows + m] > 0.f ? 1u : 0u) << n;
            m1b |= (sm.h1[(32 + n) * kRows + m] > 0.f ? 1u : 0u) << n;
        }
        sm.score[m] = sc;
        if (masks) {
            uint32_t* mk = masks + ((b0 + sm.row_s[m]) * p.T + sm.row_t[m]) * 3;
            mk[0] = m1a; mk[1] = m1b; mk[2] = m2;
        }
    }
    __syncthreads();
}

// Softmax mode, len == 0, T > 0: every position holds the padding score, so the weights are 1/T over
// all T positions (the reference's quirk).  Each row is weighted by u = 1/T before it is added, as the
// reference weights it: a batch of empty histories over the same padding row gives every sample the
// same pooled vector, and the tower's batch norm turns any ulp by which it differs into its bias
// gradients.  One warp; each lane sums whole rows in t order, then the lanes reduce.
__device__ __forceinline__ void pool_empty(const DinParams& p, int64_t b, float* pooled, int32_t* err_flag) {
    const int D = p.D, D4 = D / 4, T = p.T, lane = threadIdx.x & 31;
    const float u = 1.0f / (float)T;
    float4 a[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) a[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int t = lane; t < T; t += 32) {
        const int64_t row = checked_row(__ldg(p.his_idx + b * T + t), p.his_rows, err_flag);
        const float4* k = reinterpret_cast<const float4*>(p.his_w + row * D);
#pragma unroll
        for (int c = 0; c < 8; ++c)
            if (c < D4) {
                const float4 v = __ldg(k + c);
                a[c].x = fmaf(u, v.x, a[c].x); a[c].y = fmaf(u, v.y, a[c].y);
                a[c].z = fmaf(u, v.z, a[c].z); a[c].w = fmaf(u, v.w, a[c].w);
            }
    }
#pragma unroll
    for (int c = 0; c < 8; ++c)
        if (c < D4) {
            const float v[4] = {warp_sum(a[c].x), warp_sum(a[c].y), warp_sum(a[c].z), warp_sum(a[c].w)};
            if (lane == 0)
                for (int e = 0; e < 4; ++e) pooled[4 * c + e] = v[e];
        }
}

// The forward's last step: the rest of the concat row and the L2 norm, one warp per sample.
__device__ __forceinline__ void concat_norm(const DinParams& p, const DinSmem& sm, int64_t b0, int n_samples,
                                            float* concat_all, float* norm_out, int32_t* err_flag) {
    const int D = p.D, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int s = warp; s < n_samples; s += kDinThreads / 32) {
        const int64_t b = b0 + s;
        float* out = concat_all + b * p.width;
        float ss = 0.f;
        for (int c = lane; c < p.width; c += 32) {
            float v;
            if (c < p.n_dense) {
                v = __ldg(p.dense_col[c] + b * p.dense_stride);
                out[c] = v;
            } else if (c >= p.att_off && c < p.att_off + D) {
                v = sm.gatt[s * D + c - p.att_off];        // pooled (kept in shared memory)
            } else if (c >= p.tgt_off && c < p.tgt_off + D) {
                v = sm.q[s * D + c - p.tgt_off];
                out[c] = v;
            } else {
                v = 0.f;
                for (int f = 0; f < p.cat.F; ++f)
                    if (c >= p.cat.off[f] && c < p.cat.off[f] + p.cat.dim[f]) {
                        const int64_t row = checked_row(__ldg(p.cat.idx[f] + b), p.cat.rows[f], err_flag);
                        v = __ldg(p.cat.weight[f] + row * p.cat.dim[f] + c - p.cat.off[f]);
                    }
                out[c] = v;
            }
            if (c >= p.l2_from) ss = fmaf(v, v, ss);
        }
        ss = warp_sum(ss);
        if (lane == 0 && norm_out) norm_out[b] = sqrtf(ss);
    }
}

// Shared memory holds this kernel at 2 CTAs per SM, so it may use up to 128 registers at no cost in
// occupancy; with that bound stated ptxas schedules it at ~100 registers, which measured 0.4-2.4 % faster
// (hot path, T = 1..256) than the ~75 it picks unbounded.
__global__ void __launch_bounds__(kDinThreads, 2)
din_fwd_kernel(const __grid_constant__ DinParams p, float* __restrict__ concat_all,
               float* __restrict__ norm_out, float* __restrict__ att_w, uint32_t* __restrict__ masks,
               int32_t* err_flag) {
    extern __shared__ __align__(16) float smem_raw[];
    const int D = p.D, K1 = 4 * D, T = p.T;
    DinSmem sm(smem_raw, D);
    const MlpLayout L(D);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b0 = (int64_t)blockIdx.x * kSamples;
    const int n_samples = (int)((p.B - b0) < kSamples ? (p.B - b0) : kSamples);

    // ---- stage the per-call weights and the CTA's q rows / lengths
    for (int i = tid; i < K1 * kH1; i += kDinThreads) sm.wA[i] = __ldg(p.mlp + L.w1t + i);
    for (int i = tid; i < kH1 * kH2; i += kDinThreads) sm.wB[i] = __ldg(p.mlp + L.w2t + i);
    for (int i = tid; i < kH1; i += kDinThreads) sm.vec[i] = __ldg(p.mlp + L.b1 + i);
    for (int i = tid; i < kH2; i += kDinThreads) {
        sm.vec[kH1 + i]       = __ldg(p.mlp + L.b2 + i);
        sm.vec[kH1 + kH2 + i] = __ldg(p.mlp + L.w3 + i);
    }
    if (tid == 0) sm.vec[kH1 + 2 * kH2] = __ldg(p.mlp + L.b3);
    for (int i = tid; i < n_samples * D; i += kDinThreads) {
        const int s = i / D, e = i - s * D;
        const int64_t row = checked_row(__ldg(p.tgt_idx + b0 + s), p.tgt_rows, err_flag);
        sm.q[i] = __ldg(p.tgt_w + row * D + e);
    }
    for (int i = tid; i < kSamples * D; i += kDinThreads) sm.gatt[i] = 0.f;   // pooled, accumulated per segment
    if (tid < kSamples) {
        sm.len[tid] = tid < n_samples ? clip_len(__ldg(p.his_len + b0 + tid), T) : 0;
        sm.run_max[tid] = -INFINITY;
        sm.run_sum[tid] = 0.f;
    }
    __syncthreads();
    const float inv_sqrt_d = 1.0f / sqrtf((float)D);

    int s_begin = 0, t_begin = 0;
    while (s_begin < n_samples) {
        if (tid == 0) plan_tile(sm, n_samples, s_begin, t_begin);
        __syncthreads();
        const int n_seg = sm.cursor[0], n_rows = sm.cursor[1], s_next = sm.cursor[2], t_next = sm.cursor[3];
        row_map(sm, n_seg, s_begin);
        __syncthreads();
        if (n_rows > 0) {
            stage_rows<true>(p, sm, b0, n_rows, err_flag);
            __syncthreads();
            mlp_fwd(p, sm, b0, n_rows, masks);
        }
        // ---- pooling: one warp per segment
        for (int j = warp; j < n_seg; j += kDinThreads / 32) {
            const int s = s_begin + j, len = sm.len[s];
            const int r0 = sm.seg_r0[j], n = sm.seg_r0[j + 1] - r0, t0 = sm.seg_t0[j];
            float* wrow = att_w + (b0 + s) * T;
            float* pooled = sm.gatt + s * D;
            if (len == 0) {
                if (p.use_softmax && T > 0) {          // at T == 0 there is nothing to pool: pooled stays 0
                    for (int t = lane; t < T; t += 32) wrow[t] = 1.0f / (float)T;
                    pool_empty(p, b0 + s, pooled, err_flag);
                } else {
                    for (int t = lane; t < T; t += 32) wrow[t] = 0.f;
                }
            } else {
                float scale = 1.f;
                if (p.use_softmax) {
                    float mx = -INFINITY;
                    for (int r = lane; r < n; r += 32) mx = fmaxf(mx, sm.score[r0 + r] * inv_sqrt_d);
                    mx = fmaxf(warp_max(mx), sm.run_max[s]);
                    scale = expf(sm.run_max[s] - mx);
                    float sum = 0.f;
                    for (int r = lane; r < n; r += 32) {
                        const float z = sm.score[r0 + r] * inv_sqrt_d, e = expf(z - mx);
                        sm.gw[r0 + r] = e;
                        sum += e;
                        wrow[t0 + r] = z;
                    }
                    sum = warp_sum(sum);
                    __syncwarp();
                    if (lane == 0) { sm.run_sum[s] = fmaf(sm.run_sum[s], scale, sum); sm.run_max[s] = mx; }
                } else {
                    for (int r = lane; r < n; r += 32) {
                        const float w = sm.score[r0 + r];
                        sm.gw[r0 + r] = w;
                        wrow[t0 + r] = w;
                    }
                }
                __syncwarp();
                for (int e = 0; e < D; ++e) {
                    float a = 0.f;
                    for (int r = lane; r < n; r += 32) a = fmaf(sm.gw[r0 + r], sm.x[(D + e) * kRows + r0 + r], a);
                    a = warp_sum(a);
                    if (lane == 0) pooled[e] = fmaf(pooled[e], scale, a);
                }
                if (t0 + n == len) {                       // the sample's last segment
                    __syncwarp();
                    if (p.use_softmax) {
                        const float mx = sm.run_max[s], inv_sum = 1.0f / sm.run_sum[s];
                        for (int t = lane; t < T; t += 32) wrow[t] = t < len ? expf(wrow[t] - mx) * inv_sum : 0.f;
                        for (int e = lane; e < D; e += 32) pooled[e] *= inv_sum;
                    } else {
                        for (int t = len + lane; t < T; t += 32) wrow[t] = 0.f;
                    }
                }
            }
            __syncwarp();
            if (t0 + n == len)
                for (int e = lane; e < D; e += 32) concat_all[(b0 + s) * p.width + p.att_off + e] = pooled[e];
        }
        __syncthreads();
        s_begin = s_next;
        t_begin = t_next;
    }
    concat_norm(p, sm, b0, n_samples, concat_all, norm_out, err_flag);
}

// Backward.  g_row[B,width]: gradient w.r.t. every column of the concat row INCLUDING what flows
// back through the attention into q (target columns) — these are the per-occurrence gradients of
// the category / target tables.  g_hist[B,T,D]: per-occurrence gradients of the history table
// (written for live positions only).
__global__ void __launch_bounds__(kDinThreads)
din_bwd_kernel(const __grid_constant__ DinParams p, const float* __restrict__ concat_all,
               const float* __restrict__ norm, const float* __restrict__ att_w,
               const uint32_t* __restrict__ masks, const float* __restrict__ g_concat,
               const float* __restrict__ g_norm, float* __restrict__ g_row,
               float* __restrict__ g_hist, int32_t* err_flag) {
    extern __shared__ __align__(16) float smem_raw[];
    const int D = p.D, K1 = 4 * D, T = p.T;
    DinSmem sm(smem_raw, D);
    const MlpLayout L(D);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t b0 = (int64_t)blockIdx.x * kSamples;
    const int n_samples = (int)((p.B - b0) < kSamples ? (p.B - b0) : kSamples);

    // weights in their registered orientation: B operands of the transposed products
    for (int i = tid; i < kH1 * K1; i += kDinThreads) sm.wA[i] = __ldg(p.mlp + L.w1 + i);   // [64][K1]
    for (int i = tid; i < kH2 * kH1; i += kDinThreads) sm.wB[i] = __ldg(p.mlp + L.w2 + i);  // [32][64]
    for (int i = tid; i < kH2; i += kDinThreads) sm.vec[i] = __ldg(p.mlp + L.w3 + i);
    if (tid < kSamples) sm.len[tid] = tid < n_samples ? clip_len(__ldg(p.his_len + b0 + tid), T) : 0;
    // per sample: q, and g_att = upstream gradient of the attention output (tower + L2 term)
    for (int i = tid; i < n_samples * D; i += kDinThreads) {
        const int s = i / D, e = i - s * D;
        const int64_t b = b0 + s;
        sm.q[i] = concat_all[b * p.width + p.tgt_off + e];
        float g = g_concat ? g_concat[b * p.width + p.att_off + e] : 0.f;
        if (g_norm) {
            const float nv = norm[b];
            if (nv > 0.f) g = fmaf(g_norm[b] / nv, concat_all[b * p.width + p.att_off + e], g);
        }
        sm.gatt[i] = g;
        sm.gq[i]   = 0.f;
    }
    __syncthreads();
    // softmax: sum_u w_u (g_att . k_u) = g_att . pooled, one scalar per sample
    if (tid < n_samples) {
        float dot = 0.f;
        for (int e = 0; e < D; ++e) dot = fmaf(sm.gatt[tid * D + e], concat_all[(b0 + tid) * p.width + p.att_off + e], dot);
        sm.run_sum[tid] = dot;
    }
    __syncthreads();
    const float* w3 = sm.vec;
    const float  inv_sqrt_d = 1.0f / sqrtf((float)D);

    int s_begin = 0, t_begin = 0;
    while (s_begin < n_samples) {
        if (tid == 0) plan_tile(sm, n_samples, s_begin, t_begin);
        __syncthreads();
        const int n_seg = sm.cursor[0], n_rows = sm.cursor[1], s_next = sm.cursor[2], t_next = sm.cursor[3];
        row_map(sm, n_seg, s_begin);
        __syncthreads();
        if (n_rows > 0) {
            stage_rows<false>(p, sm, b0, n_rows, err_flag);      // K rows -> x[D..2D)
            __syncthreads();
            // score gradient of every row, local to the row: raw g_att . k; softmax w (g_att . k - g_att . pooled) / sqrt(D)
            if (tid < kRows) {
                const int m = tid;
                float gs = 0.f, w = 0.f;
                uint32_t k0 = 0, k1 = 0, k2 = 0;
                if (m < n_rows) {
                    const int s = sm.row_s[m], t = sm.row_t[m];
                    float gw = 0.f;
                    for (int e = 0; e < D; ++e) gw = fmaf(sm.gatt[s * D + e], sm.x[(D + e) * kRows + m], gw);
                    w = att_w[(b0 + s) * T + t];
                    gs = p.use_softmax ? w * (gw - sm.run_sum[s]) * inv_sqrt_d : gw;
                    const uint32_t* mk = masks + ((b0 + s) * T + t) * 3;
                    k0 = mk[0]; k1 = mk[1]; k2 = mk[2];
                }
                sm.score[m] = w;
                sm.mask[m] = k0; sm.mask[kRows + m] = k1; sm.mask[2 * kRows + m] = k2;
                // g_z2[n][m] = g_s[m] * w3[n] * relu2'  -> h2 region
#pragma unroll 8
                for (int n = 0; n < kH2; ++n) sm.h2[n * kRows + m] = ((k2 >> n) & 1u) ? gs * w3[n] : 0.f;
            }
            __syncthreads();
            const int m_used = (n_rows + 3) / 4 * 4;
            // g_z1 = (g_z2 x W2) * relu1'   [rows,32]x[32,64]
            tile_gemm_rows<8>(sm.h2, sm.wB, kH2, kH1, m_used, [&](int m0, int n0, float (&acc)[4][8]) {
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const uint32_t bits = sm.mask[(n0 >> 5) * kRows + m0 + i] >> (n0 & 31);
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = ((bits >> j) & 1u) ? acc[i][j] : 0.f;
                }
                store_tile_kmajor<8>(sm.h1, kRows, m0, n0, acc);
            });
            __syncthreads();
            // g_cross = g_z1 x W1   [rows,64]x[64,4D]: h1 is this product's A operand, so its k-block
            // [D,2D) goes to h2 (free now, D <= 32 rows) and the rest over x, keeping the K rows in x[D..2D)
            tile_gemm_rows<4>(sm.h1, sm.wA, kH1, K1, m_used, [&](int m0, int n0, float (&acc)[4][4]) {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int c = n0 + j;
                    float* dst = (c >= D && c < 2 * D) ? sm.h2 + (c - D) * kRows : sm.x + c * kRows;
                    *reinterpret_cast<float4*>(dst + m0) = make_float4(acc[0][j], acc[1][j], acc[2][j], acc[3][j]);
                }
            });
            __syncthreads();
            // per row: g_k = w_t g_att + gc_k - gc_d + gc_p * q ; g_q_row = gc_q + gc_d + gc_p * k
            for (int item = tid; item < D * kRows; item += kDinThreads) {
                const int e = item / kRows, m = item - e * kRows;
                if (m < n_rows) {
                    const int s = sm.row_s[m];
                    const float k  = sm.x[(D + e) * kRows + m];
                    const float gd = sm.x[(2 * D + e) * kRows + m];
                    const float gp = sm.x[(3 * D + e) * kRows + m];
                    sm.x[e * kRows + m]       = sm.x[e * kRows + m] + gd + gp * k;
                    sm.x[(D + e) * kRows + m] = fmaf(sm.score[m], sm.gatt[s * D + e], sm.h2[e * kRows + m] - gd + gp * sm.q[s * D + e]);
                }
            }
            __syncthreads();
            // write g_k rows (coalesced over e inside a row)
            for (int item = tid; item < (D / 4) * kRows; item += kDinThreads) {
                const int c4 = item / kRows, m = item - c4 * kRows;
                if (m < n_rows) {
                    const float* src = sm.x + (D + 4 * c4) * kRows + m;
                    *reinterpret_cast<float4*>(g_hist + ((b0 + sm.row_s[m]) * T + sm.row_t[m]) * D + 4 * c4) =
                        make_float4(src[0], src[kRows], src[2 * kRows], src[3 * kRows]);
                }
            }
            // g_q: each segment's rows, added to the sample's sum segment after segment
            for (int j = warp; j < n_seg; j += kDinThreads / 32) {
                const int s = s_begin + j, r0 = sm.seg_r0[j], n = sm.seg_r0[j + 1] - r0;
                if (n == 0) continue;
                for (int e = 0; e < D; ++e) {
                    float a = 0.f;
                    for (int r = lane; r < n; r += 32) a += sm.x[e * kRows + r0 + r];
                    a = warp_sum(a);
                    if (lane == 0) sm.gq[s * D + e] += a;
                }
            }
        }
        // softmax, len == 0: uniform weights over all T positions, gradient g_att / T everywhere
        if (p.use_softmax) {
            for (int j = 0; j < n_seg; ++j) {
                const int s = s_begin + j;
                if (sm.len[s] != 0) continue;
                const float u = 1.0f / (float)T;
                for (int64_t i = tid; i < (int64_t)T * D; i += kDinThreads)
                    g_hist[(b0 + s) * T * D + i] = u * sm.gatt[s * D + (int)(i % D)];
            }
        }
        __syncthreads();
        s_begin = s_next;
        t_begin = t_next;
    }

    // ---- gradient of the concat row: tower gradient + L2 term (+ attention's d/dq on the target)
    for (int s = warp; s < n_samples; s += kDinThreads / 32) {
        const int64_t b = b0 + s;
        float scale = 0.f;
        if (g_norm) {
            const float nv = norm[b];
            scale = nv > 0.f ? g_norm[b] / nv : 0.f;
        }
        for (int c = lane; c < p.width; c += 32) {
            float g = g_concat ? g_concat[b * p.width + c] : 0.f;
            if (c >= p.l2_from) g = fmaf(scale, concat_all[b * p.width + c], g);
            if (c >= p.tgt_off && c < p.tgt_off + D) g += sm.gq[s * D + c - p.tgt_off];
            g_row[b * p.width + c] = g;
        }
    }
}

// ===========================================================================================
// Tensor-core forward (D = 16): the activation-unit MLP on tcgen05, bf16 operands, fp32
// accumulators in TMEM.  One thread = one (b,t) row = one TMEM lane; 128 rows per tile.
//   A1[128x64] = [q,k,q-k,q*k] (split bf16 hi+lo, K-major, 128-byte swizzle, built by the row's thread)
//   D1 = A1 . W1^T (4 x tcgen05.mma M128 N64 K16) -> tcgen05.ld -> +b1, ReLU, mask bits, bf16
//   A2 = relu(D1) rewritten in place over A1;  D2 = A2 . W2^T (M128 N32) -> +b2, ReLU, . w3
// Gathered K rows stay in fp32 registers for the pooling.  Everything outside the two GEMMs is
// the same math as din_fwd_kernel; tolerance of this path is the bf16 bar (2e-2).
// ===========================================================================================
namespace tc {

constexpr int kTcThreads  = 128;
constexpr int kTcTmemCols = 128;     // 64 (layer 1) + 32 (layer 2), power of two

// Dynamic group scheduler of the persistent tensor-core kernels: [0] forward, [1] backward.
// CTAs draw sample groups from `next`; the last CTA to finish re-arms both counters, so every
// launch (and every CUDA-graph replay) starts from zero without a memset.  One launch of a
// kernel at a time per device (launches are stream-ordered; one process per GPU).
__device__ unsigned int g_din_next[2];
__device__ unsigned int g_din_done[2];

__device__ __forceinline__ int64_t next_group(int which, unsigned int* slot) {
    if (threadIdx.x == 0) *slot = atomicAdd(&g_din_next[which], 1u);
    __syncthreads();
    return (int64_t)*slot;
}
__device__ __forceinline__ void scheduler_exit(int which) {
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(&g_din_done[which], 1u) == gridDim.x - 1) {
            g_din_next[which] = 0;
            g_din_done[which] = 0;
            __threadfence();
        }
    }
}

// ---- forward -------------------------------------------------------------------------------
constexpr int kTcGroup = kSamples;   // samples per scheduler draw (16 was measured slower: 93 vs 82 us)

struct TcFwdSmem {
    uint8_t *a, *a_lo, *w1, *w1_lo, *w2, *w2_lo;   // swizzled split-bf16 tiles; a_lo doubles as pooling scratch
    float *kstage;                                 // [128][16] history rows landed by cp.async.bulk
    float *vec, *q, *att, *score, *wt;
    int *len;
    int64_t *ix_his, *ix_tgt, *ix_len, *ix_cat;    // the group's raw indices, landed by cp.async
    int16_t* colmap;                               // concat column -> categorical field; -1 dense/none, -2 target/attention
    uint64_t *bar_mma, *bar_w;
    uint32_t* tmem_slot;
    __device__ TcFwdSmem(uint8_t* base, int T, int F) {
        uint8_t* p = base;
        a = p;       p += 128 * 128;
        a_lo = p;    p += 128 * 128;
        w1 = p;      p += 64 * 128;
        w1_lo = p;   p += 64 * 128;
        w2 = p;      p += 32 * 128;
        w2_lo = p;   p += 32 * 128;
        kstage = (float*)p;  p += sizeof(float) * kRows * 16;
        vec = (float*)p;     p += sizeof(float) * (kH1 + 2 * kH2 + 4);
        q = (float*)p;       p += sizeof(float) * kTcGroup * 16;
        att = (float*)p;     p += sizeof(float) * kTcGroup * 16;
        score = (float*)p;   p += sizeof(float) * kRows;
        wt = (float*)p;      p += sizeof(float) * kRows;
        len = (int*)p;       p += sizeof(int) * 3 * kTcGroup;      // [0,8) lengths, [8,17) their prefix sums
        bar_mma = (uint64_t*)p;   p += 8;
        tmem_slot = (uint32_t*)p; p += 8;
        bar_w = (uint64_t*)p;     p += 8;
        p += 8;
        ix_his = (int64_t*)p;     p += sizeof(int64_t) * kTcGroup * T;
        ix_tgt = (int64_t*)p;     p += sizeof(int64_t) * kTcGroup;
        ix_len = (int64_t*)p;     p += sizeof(int64_t) * kTcGroup;
        ix_cat = (int64_t*)p;     p += sizeof(int64_t) * kTcGroup * F;
        colmap = (int16_t*)p;
    }
    static size_t bytes(int width, int T, int F) {
        return 1024 /* alignment slack */ + 2 * (128 * 128 + 64 * 128 + 32 * 128) + sizeof(float) * kRows * 16 +
               sizeof(float) * (kH1 + 2 * kH2 + 4 + 2 * kTcGroup * 16 + 2 * kRows) + sizeof(int) * 3 * kTcGroup + 32 +
               sizeof(int64_t) * kTcGroup * (size_t)(T + 2 + F) + sizeof(int16_t) * (size_t)width;
    }
};

// A tile = whole samples [s_begin, s_end) of the group, n_rows <= 128 live (b,t) rows; this
// thread's row is (my_s, my_t) when `on`.
struct TcTile {
    int s_end, n_rows, my_s, my_t;
    bool on;
};
// len[0..8) are the group's clipped lengths, len[8 + i] = len[0] + ... + len[i-1] (i = 0..8): the rows of samples
// [s_begin, i) are a difference of two prefix sums, so planning a tile is straight-line code on registers instead
// of a loop of dependent shared-memory loads.
__device__ __forceinline__ void store_len_prefix(int* len, const int64_t* ix_len, int n_samples, int T, int tid) {
    if (tid < kTcGroup) len[tid] = tid < n_samples ? clip_len(ix_len[tid], T) : 0;
    else if (tid < 2 * kTcGroup + 1) {
        int a = 0;
        for (int j = 0; j < tid - kTcGroup; ++j) a += j < n_samples ? clip_len(ix_len[j], T) : 0;
        len[tid] = a;
    }
}
__device__ __forceinline__ TcTile plan_tile_tc(const int* len, int n_samples, int s_begin, int tid) {
    const int4 p0 = *reinterpret_cast<const int4*>(len + kTcGroup), p1 = *reinterpret_cast<const int4*>(len + kTcGroup + 4);
    const int pre[kTcGroup + 1] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w, len[2 * kTcGroup]};
    const int base = len[kTcGroup + s_begin];
    TcTile t;
    t.s_end = s_begin; t.n_rows = 0;
    int my_s = s_begin, start = 0;
#pragma unroll
    for (int i = 0; i < kTcGroup; ++i) {
        const int end_i = pre[i + 1] - base;         // rows of samples [s_begin, i]
        // whole samples while they fit: the prefix sums are monotone, so this holds on one run starting at s_begin
        const bool fits = i >= s_begin && i < n_samples && end_i <= kRows;
        if (fits) { t.s_end = i + 1; t.n_rows = end_i; }
        if (fits && tid >= end_i) { my_s = i + 1; start = end_i; }
    }
    t.on = tid < t.n_rows;
    t.my_s = t.on ? my_s : s_begin;
    t.my_t = t.on ? tid - start : 0;
    return t;
}
__device__ __forceinline__ int tile_row0(const int* len, int s_begin, int s) {
    return len[kTcGroup + s] - len[kTcGroup + s_begin];
}

// kstage rows are 64 bytes apart, so the same 16-byte chunk of 32 consecutive rows would fall on two
// bank groups (16-way conflict for the LDGSTS writes and the LDS.128 read-back).  Chunk c of row r
// lives at position c ^ ((r >> 1) & 3): eight consecutive rows then cover all eight bank groups.
__device__ __forceinline__ int kstage_chunk(int row, int c) { return c ^ ((row >> 1) & 3); }

// Asynchronous staging of the tile's history rows: a thread that owns a live row issues four 16-byte
// cp.async (LDGSTS) copies of it into its own slot of kstage and commits the group; it later waits
// for its own group only (each thread reads back just the row it copied, so no barrier is needed).
// No registers are tied up while the rows are in flight: this is issued for tile i+1 while the
// tensor core works on tile i.  (One 64-byte cp.async.bulk per row was measured slower — 96 vs
// 82 us for the whole kernel — the TMA unit is built for few large copies, not 200k small ones.)
__device__ __forceinline__ void issue_rows(const DinParams& p, const TcFwdSmem& sm, const TcTile& t, int tid,
                                           int32_t* err_flag) {
    if (t.on) {
        const int64_t row = checked_row(sm.ix_his[t.my_s * p.T + t.my_t], p.his_rows, err_flag);
        const float* src = p.his_w + row * 16;
        const uint32_t dst = smem_u32(sm.kstage + tid * 16);
#pragma unroll
        for (int c = 0; c < 4; ++c)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16 * kstage_chunk(tid, c)), "l"(src + 4 * c) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}
__device__ __forceinline__ void wait_rows() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// Every index the group needs — history ids, target id, length, categorical ids — in one round of
// 8-byte cp.async copies: issued one group ahead (during the last tile of the previous group), so
// that a group starts with its indices in shared memory and pays one memory latency (the rows)
// instead of an index -> row chain per feature.
__device__ __forceinline__ void issue_idx(const DinParams& p, const TcFwdSmem& sm, int64_t group, int tid) {
    const int64_t b0 = group * kTcGroup;
    const int n = (int)((p.B - b0) < kTcGroup ? (p.B - b0) : kTcGroup);
    for (int i = tid; i < n * p.T; i += kTcThreads) cp_async8(sm.ix_his + i, p.his_idx + b0 * p.T + i);
    if (tid < n) {
        cp_async8(sm.ix_tgt + tid, p.tgt_idx + b0 + tid);
        cp_async8(sm.ix_len + tid, p.his_len + b0 + tid);
    }
    for (int i = tid; i < p.cat.F * kTcGroup; i += kTcThreads) {
        const int f = i / kTcGroup, s_ = i - f * kTcGroup;
        if (s_ < n) cp_async8(sm.ix_cat + i, p.cat.idx[f] + b0 + s_);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}


// The operand tiles of the per-call weights, laid out once per forward by din_weight_tiles_kernel in exactly
// the swizzled split-bf16 image the kernels keep in shared memory, so that a CTA fetches them with ONE bulk
// (TMA) copy instead of converting 24-32 KB itself (8 % of the forward, 9 % of the backward before):
//   forward image   [W1 hi 8K][W1 lo 8K][W2 hi 4K][W2 lo 4K]                  (B operands [n][k], K-major)
//   backward image  [W1^T hi 8K][W1^T lo 8K][W2^T hi 8K][W2^T lo 8K]
constexpr uint32_t kTileFwdBytes = 2 * (64 * 128 + 32 * 128);
constexpr uint32_t kTileBwdBytes = 2 * (64 * 128 + 64 * 128);

__global__ void __launch_bounds__(256)
din_weight_tiles_kernel(const float* __restrict__ mlp, uint8_t* __restrict__ tiles) {
    const MlpLayout L(16);
    uint8_t* f_w1 = tiles;            uint8_t* f_w1_lo = f_w1 + 64 * 128;
    uint8_t* f_w2 = f_w1_lo + 64 * 128;  uint8_t* f_w2_lo = f_w2 + 32 * 128;
    uint8_t* b_w1 = tiles + kTileFwdBytes;  uint8_t* b_w1_lo = b_w1 + 64 * 128;
    uint8_t* b_w2 = b_w1_lo + 64 * 128;     uint8_t* b_w2_lo = b_w2 + 64 * 128;
    // rows of a tile that no weight fills (backward W2^T: chunks 4..7 of a line) are never read by an MMA
    for (int item = blockIdx.x * blockDim.x + threadIdx.x; item < 1536; item += gridDim.x * blockDim.x) {
        float v[8];
        if (item < 512) {                                   // forward W1[n][k]: 64 rows x 8 chunks
            const int n = item >> 3, c = item & 7;
            ld8(mlp + L.w1 + n * 64 + c * 8, v);
            store_chunk_split(f_w1, f_w1_lo, n, c, v);
        } else if (item < 768) {                            // forward W2[n][k]: 32 rows x 8 chunks
            const int i = item - 512, n = i >> 3, c = i & 7;
            ld8(mlp + L.w2 + n * 64 + c * 8, v);
            store_chunk_split(f_w2, f_w2_lo, n, c, v);
        } else if (item < 1024) {                           // backward W2^T[n][k]: 64 rows x 4 chunks
            const int i = item - 768, n = i >> 2, c = i & 3;
            ld8(mlp + L.w2t + n * 32 + c * 8, v);
            store_chunk_split(b_w2, b_w2_lo, n, c, v);
        } else {                                            // backward W1^T[c][n]: 64 rows x 8 chunks
            const int i = item - 1024, n = i >> 3, c = i & 7;
            ld8(mlp + L.w1t + n * 64 + c * 8, v);
            store_chunk_split(b_w1, b_w1_lo, n, c, v);
        }
    }
}

__global__ void __launch_bounds__(kTcThreads)
din_fwd_tc_kernel(const __grid_constant__ DinParams p, float* __restrict__ concat_all,
                  float* __restrict__ norm_out, float* __restrict__ att_w, uint32_t* __restrict__ masks,
                  int32_t* err_flag) {
    extern __shared__ uint8_t smem_raw_tc[];
    uint8_t* base = smem_raw_tc + ((1024u - (smem_u32(smem_raw_tc) & 1023u)) & 1023u);   // swizzle atoms need 1024 B
    TcFwdSmem sm(base, p.T, p.cat.F);
    PROF_DECL
    constexpr int D = 16;
    const int T = p.T;
    const MlpLayout L(D);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n_groups = (p.B + kTcGroup - 1) / kTcGroup;

    // The first group is static (blockIdx.x <= n_groups - 1: the grid never exceeds the group count);
    // later ones are drawn from the device counter.  Its indices start flying before the set-up.
    int64_t group = blockIdx.x;
    issue_idx(p, sm, group, tid);

    // ---- one-time setup: barriers, TMEM, weights (fp32 -> split bf16, swizzled, K-major = as registered)
    if (tid == 0) {
        mbar_init(sm.bar_mma, 1);
        mbar_init(sm.bar_w, 1);
        // the four weight tiles in one bulk (TMA) copy: w1 | w1_lo | w2 | w2_lo are contiguous
        mbar_expect_tx(sm.bar_w, kTileFwdBytes);
        bulk_copy_g2s(sm.w1, p.mlp_tiles, kTileFwdBytes, sm.bar_w);
    }
    if (warp == 0) tmem_alloc(sm.tmem_slot, kTcTmemCols);
    for (int i = tid; i < kH1; i += kTcThreads) sm.vec[i] = __ldg(p.mlp + L.b1 + i);
    for (int i = tid; i < kH2; i += kTcThreads) {
        sm.vec[kH1 + i]       = __ldg(p.mlp + L.b2 + i);
        sm.vec[kH1 + kH2 + i] = __ldg(p.mlp + L.w3 + i);
    }
    if (tid == 0) sm.vec[kH1 + 2 * kH2] = __ldg(p.mlp + L.b3);
    for (int c = tid; c < p.width; c += kTcThreads) {
        int m = -1;
        for (int f = 0; f < p.cat.F; ++f)
            if (c >= p.cat.off[f] && c < p.cat.off[f] + p.cat.dim[f]) m = f;
        if ((c >= p.att_off && c < p.att_off + D) || (c >= p.tgt_off && c < p.tgt_off + D)) m = -2;
        sm.colmap[c] = (int16_t)m;
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    mbar_wait(sm.bar_w, 0);
    const uint32_t tmem = *sm.tmem_slot;
    const float* b1 = sm.vec;
    const float* b2 = sm.vec + kH1;
    const float* w3 = sm.vec + kH1 + kH2;
    const float  b3 = sm.vec[kH1 + 2 * kH2];
    const float  inv_sqrt_d = 0.25f;
    const uint64_t a_desc[2]  = {umma_desc(smem_u32(sm.a)), umma_desc(smem_u32(sm.a_lo))};
    const uint64_t w1_desc[2] = {umma_desc(smem_u32(sm.w1)), umma_desc(smem_u32(sm.w1_lo))};
    const uint64_t w2_desc[2] = {umma_desc(smem_u32(sm.w2)), umma_desc(smem_u32(sm.w2_lo))};
    const uint32_t my_tmem = tmem + ((uint32_t)(warp * 32) << 16);
    float* pool = reinterpret_cast<float*>(sm.a_lo);     // [128][17], free once the second MMA has read a_lo
    uint32_t ph_mma = 0;

    PROF(0);
    __shared__ unsigned int group_slot;
    while (group < n_groups) {                   // persistent: groups of 8 samples
        // the next draw is issued now and published at the first barrier of a tile: its latency is
        // never exposed, and the last tile of this group prefetches the indices of the next one
        unsigned int next_draw = 0;
        if (tid == 0) next_draw = gridDim.x + atomicAdd(&g_din_next[0], 1u);
        const int64_t b0 = group * kTcGroup;
        const int n_samples = (int)((p.B - b0) < kTcGroup ? (p.B - b0) : kTcGroup);
        wait_rows();                             // this group's indices (issue_idx) have landed ...
        __syncthreads();                         // ... for every thread
        store_len_prefix(sm.len, sm.ix_len, n_samples, T, tid);
        if (tid < n_samples * 4) {               // target rows: 4 x 16 bytes per sample, same commit group as the tile rows
            const int s = tid >> 2, c = tid & 3;
            const int64_t row = checked_row(sm.ix_tgt[s], p.tgt_rows, err_flag);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                         ::"r"(smem_u32(sm.q + s * D + 4 * c)), "l"(p.tgt_w + row * D + 4 * c) : "memory");
        }
        __syncthreads();
        PROF(1); PROF_COUNT(13);

        int s_begin = 0;
        TcTile cur = plan_tile_tc(sm.len, n_samples, 0, tid);
        issue_rows(p, sm, cur, tid, err_flag);               // first tile of the group: exposed latency

        // ---- while those rows fly: every column of the concat rows except the attention output.
        // Warp w owns samples w and w + 4; all index loads, then all row loads are issued back to
        // back (registers), so the group pays two memory latencies instead of two per column.
        constexpr int kSlots = kTcGroup / 4;
        float ss_part[kSlots];
#pragma unroll
        for (int slot = 0; slot < kSlots; ++slot) ss_part[slot] = 0.f;
        for (int c0 = 0; c0 < p.width; c0 += 128) {
            const float* src[kSlots][4];
#pragma unroll
            for (int slot = 0; slot < kSlots; ++slot)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int s = warp + 4 * slot, c = c0 + lane + 32 * j;
                    src[slot][j] = nullptr;
                    if (s < n_samples && c < p.width) {
                        const int64_t b = b0 + s;
                        const int f = sm.colmap[c];
                        if (f >= 0) {
                            const int64_t row = checked_row(sm.ix_cat[f * kTcGroup + s], p.cat.rows[f], err_flag);
                            src[slot][j] = p.cat.weight[f] + row * p.cat.dim[f] + (c - p.cat.off[f]);
                        } else if (c < p.n_dense) {
                            src[slot][j] = p.dense_col[c] + b * p.dense_stride;
                        }
                    }
                }
            float v[kSlots][4];
#pragma unroll
            for (int slot = 0; slot < kSlots; ++slot)
#pragma unroll
                for (int j = 0; j < 4; ++j) v[slot][j] = src[slot][j] ? __ldg(src[slot][j]) : 0.f;
#pragma unroll
            for (int slot = 0; slot < kSlots; ++slot)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int s = warp + 4 * slot, c = c0 + lane + 32 * j;
                    if (s < n_samples && c < p.width && sm.colmap[c] != -2) {
                        const float x = v[slot][j];
                        concat_all[(b0 + s) * p.width + c] = x;
                        if (c >= p.l2_from) ss_part[slot] = fmaf(x, x, ss_part[slot]);
                    }
                }
        }
        // Softmax over an empty history: every position holds the padding score, so the weights are
        // uniform 1/T over ALL T positions.  One warp per such sample, lanes = (16-byte chunk, t mod 8).
        if (p.use_softmax) {
            const float u = 1.0f / (float)T;
            for (int s = warp; s < n_samples; s += kTcThreads / 32) {
                if (sm.len[s] != 0) continue;
                const int c4 = lane & 3;
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
                for (int t = lane >> 2; t < T; t += 8) {
                    const int64_t row = checked_row(sm.ix_his[s * T + t], p.his_rows, err_flag);
                    const float4 v = __ldg(reinterpret_cast<const float4*>(p.his_w + row * D) + c4);
                    acc.x = fmaf(u, v.x, acc.x); acc.y = fmaf(u, v.y, acc.y);
                    acc.z = fmaf(u, v.z, acc.z); acc.w = fmaf(u, v.w, acc.w);
                }
#pragma unroll
                for (int o = 4; o < 32; o <<= 1) {
                    acc.x += __shfl_xor_sync(kFull, acc.x, o); acc.y += __shfl_xor_sync(kFull, acc.y, o);
                    acc.z += __shfl_xor_sync(kFull, acc.z, o); acc.w += __shfl_xor_sync(kFull, acc.w, o);
                }
                if (lane < 4) *reinterpret_cast<float4*>(sm.att + s * 16 + 4 * c4) = acc;
            }
        }
        while (s_begin < n_samples) {
            // ---- the tile's history rows have landed in shared memory
            wait_rows();
            if (s_begin == 0) __syncthreads();   // the target rows were copied by other threads
            PROF(2); PROF_COUNT(12);
            float k[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) k[e] = 0.f;
            if (cur.on) {
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 v = *reinterpret_cast<const float4*>(sm.kstage + tid * 16 + 4 * kstage_chunk(tid, c));
                    k[4 * c] = v.x; k[4 * c + 1] = v.y; k[4 * c + 2] = v.z; k[4 * c + 3] = v.w;
                }
            }
            const bool has_next = cur.s_end < n_samples;
            TcTile nxt = cur;
            // issued while the tensor core works: the rows of the next tile or, on the last tile of
            // the group, the indices of the next group (kstage / ix_* were consumed before the barrier)
            auto shadow_work = [&]() {
                if (has_next) {
                    nxt = plan_tile_tc(sm.len, n_samples, cur.s_end, tid);
                    issue_rows(p, sm, nxt, tid, err_flag);
                } else if ((int64_t)group_slot < n_groups) {
                    issue_idx(p, sm, (int64_t)group_slot, tid);
                }
            };
            if (cur.n_rows > 0) {
                // ---- this thread's row of A1 = [q, k, q-k, q*k]
                float qv[16];
#pragma unroll
                for (int e = 0; e < 16; ++e) qv[e] = cur.on ? sm.q[cur.my_s * D + e] : 0.f;
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    float a[8], b[8], c[8], d[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        a[j] = qv[8 * half + j];
                        b[j] = k[8 * half + j];
                        c[j] = a[j] - b[j];
                        d[j] = a[j] * b[j];
                    }
                    store_chunk_split(sm.a, sm.a_lo, tid, 0 + half, a);
                    store_chunk_split(sm.a, sm.a_lo, tid, 2 + half, b);
                    store_chunk_split(sm.a, sm.a_lo, tid, 4 + half, c);
                    store_chunk_split(sm.a, sm.a_lo, tid, 6 + half, d);
                }
                if (tid == 0) group_slot = next_draw;
                fence_async_smem();
                fence_before();
                __syncthreads();
                if (tid == 0) {                          // layer 1 on the tensor core
                    PROF(3);
                    fence_after();
#pragma unroll
                    for (int term = 0; term < 3; ++term)   // hi.hi + lo.hi + hi.lo
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)     // K = 64 = 4 x 16; +32 B per step inside the swizzle atom
                            umma_bf16(tmem, a_desc[term == 1] + 2 * kk, w1_desc[term == 2] + 2 * kk, umma_idesc(64),
                                      (term | kk) > 0);
                    umma_commit(sm.bar_mma);
                }
                shadow_work();
                mbar_wait(sm.bar_mma, ph_mma);
                ph_mma ^= 1;
                fence_after();
                uint32_t m1a = 0, m1b = 0;
                PROF(4);
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    float v[32];
                    tmem_ld32(my_tmem + 32 * half, v);
                    uint32_t bits = 0;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {            // 16-byte broadcast loads of the bias
                        const float4 bb = *reinterpret_cast<const float4*>(b1 + 32 * half + 4 * c);
                        v[4 * c]     = fmaxf(v[4 * c] + bb.x, 0.f);
                        v[4 * c + 1] = fmaxf(v[4 * c + 1] + bb.y, 0.f);
                        v[4 * c + 2] = fmaxf(v[4 * c + 2] + bb.z, 0.f);
                        v[4 * c + 3] = fmaxf(v[4 * c + 3] + bb.w, 0.f);
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) bits |= (v[j] > 0.f ? 1u : 0u) << j;
                    if (half == 0) m1a = bits; else m1b = bits;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float h8[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) h8[j] = v[8 * c + j];
                        store_chunk_split(sm.a, sm.a_lo, tid, 4 * half + c, h8);   // A2 = relu(layer 1), in place
                    }
                }
                fence_async_smem();
                fence_before();
                __syncthreads();
                if (tid == 0) {                          // layer 2 on the tensor core
                    PROF(5);
                    fence_after();
#pragma unroll
                    for (int term = 0; term < 3; ++term)
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            umma_bf16(tmem + 64, a_desc[term == 1] + 2 * kk, w2_desc[term == 2] + 2 * kk,
                                      umma_idesc(32), (term | kk) > 0);
                    umma_commit(sm.bar_mma);
                }
                mbar_wait(sm.bar_mma, ph_mma);
                ph_mma ^= 1;
                fence_after();
                {
                    PROF(6);
                    float v[32];
                    tmem_ld32(my_tmem + 64, v);
                    float sc = b3;
                    uint32_t m2 = 0;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const float4 bb = *reinterpret_cast<const float4*>(b2 + 4 * c);
                        const float4 ww = *reinterpret_cast<const float4*>(w3 + 4 * c);
                        const float h0 = fmaxf(v[4 * c] + bb.x, 0.f), h1 = fmaxf(v[4 * c + 1] + bb.y, 0.f);
                        const float h2 = fmaxf(v[4 * c + 2] + bb.z, 0.f), h3 = fmaxf(v[4 * c + 3] + bb.w, 0.f);
                        m2 |= ((h0 > 0.f ? 1u : 0u) | (h1 > 0.f ? 2u : 0u) | (h2 > 0.f ? 4u : 0u) | (h3 > 0.f ? 8u : 0u)) << (4 * c);
                        sc = fmaf(h0, ww.x, sc); sc = fmaf(h1, ww.y, sc);
                        sc = fmaf(h2, ww.z, sc); sc = fmaf(h3, ww.w, sc);
                    }
                    sm.score[tid] = sc;
                    if (cur.on && masks) {
                        uint32_t* mk = masks + ((b0 + cur.my_s) * T + cur.my_t) * 3;
                        mk[0] = m1a; mk[1] = m1b; mk[2] = m2;
                    }
                }
                fence_before();
                __syncthreads();
            } else {                                     // a tile of empty histories: nothing for the tensor core
                if (tid == 0) group_slot = next_draw;
                __syncthreads();
                shadow_work();
            }
            PROF(7);
            // ---- attention weights per sample (warp per sample), then weighted pooling through smem
            for (int s = s_begin + warp; s < cur.s_end; s += kTcThreads / 32) {
                const int len = sm.len[s], r0 = tile_row0(sm.len, s_begin, s);
                float* wrow = att_w + (b0 + s) * T;
                if (len == 0) {
                    const float u = p.use_softmax ? 1.0f / (float)T : 0.f;
                    for (int t = lane; t < T; t += 32) wrow[t] = u;
                    continue;
                }
                float inv_sum = 1.f, mx = 0.f;
                if (p.use_softmax) {
                    mx = -INFINITY;
                    for (int t = lane; t < len; t += 32) mx = fmaxf(mx, sm.score[r0 + t] * inv_sqrt_d);
                    mx = warp_max(mx);
                    float sum = 0.f;
                    for (int t = lane; t < len; t += 32) sum += expf(sm.score[r0 + t] * inv_sqrt_d - mx);
                    inv_sum = 1.0f / warp_sum(sum);
                }
                for (int t = lane; t < T; t += 32) {
                    float w = 0.f;
                    if (t < len) {
                        w = p.use_softmax ? expf(sm.score[r0 + t] * inv_sqrt_d - mx) * inv_sum : sm.score[r0 + t];
                        sm.wt[r0 + t] = w;
                    }
                    wrow[t] = w;
                }
            }
            __syncthreads();
            PROF(8);
            {
                const float w = cur.on ? sm.wt[tid] : 0.f;
#pragma unroll
                for (int e = 0; e < 16; ++e) pool[tid * 17 + e] = w * k[e];
            }
            __syncthreads();
            for (int item = tid; item < (cur.s_end - s_begin) * 16; item += kTcThreads) {
                const int s = s_begin + (item >> 4), e = item & 15;
                const int len = sm.len[s], r0 = tile_row0(sm.len, s_begin, s);
                float a = 0.f;
                for (int t = 0; t < len; ++t) a += pool[(r0 + t) * 17 + e];
                if (len > 0 || !p.use_softmax) sm.att[s * 16 + e] = a;     // (softmax, no history): set at group start
            }
            __syncthreads();
            s_begin = cur.s_end;
            cur = nxt;
            PROF(9);
        }

        // ---- the attention output columns and the L2 norm of the finished rows
#pragma unroll
        for (int slot = 0; slot < kSlots; ++slot) {
            const int s = warp + 4 * slot;
            if (s >= n_samples) continue;
            const int64_t b = b0 + s;
            float ss = ss_part[slot];
            {                                    // lanes 0..15: attention output, 16..31: target row
                const int e = lane & 15;
                const int c = (lane < D ? p.att_off : p.tgt_off) + e;
                const float x = lane < D ? sm.att[s * 16 + e] : sm.q[s * D + e];
                concat_all[b * p.width + c] = x;
                if (c >= p.l2_from) ss = fmaf(x, x, ss);
            }
            ss = warp_sum(ss);
            if (lane == 0 && norm_out) norm_out[b] = sqrtf(ss);
        }
        __syncthreads();      // q / len / att are rewritten by the next group
        group = (int64_t)group_slot;     // rewritten only after the next group's first barrier
        PROF(10);
    }
    scheduler_exit(0);
    PROF_END;
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kTcTmemCols);
}

// ---- backward ------------------------------------------------------------------------------
struct TcBwdSmem {
    uint8_t *a, *a_lo, *w1, *w1_lo, *w2, *w2_lo;   // w1 = W1^T, w2 = W2^T (64 rows each); a_lo doubles as pooling scratch
    float *kstage;                                 // [128][16] history rows landed by cp.async
    float *vec, *q, *att, *gq, *gt, *dot, *score, *wt;
    float *ca, *gc;                                // the group's concat_all / g_concat rows [8][width]
    float *attw;                                   // the group's attention weights [8][T]
    uint32_t* mask;                                // the group's ReLU masks [8][T][3]
    float *nrm, *gnrm;                             // [8]
    int64_t *ix_his, *ix_len;
    int* len;
    uint64_t *bar, *bar_w;
    uint32_t* tmem_slot;
    static __host__ __device__ size_t pad16(size_t n) { return (n + 15) & ~(size_t)15; }
    __device__ TcBwdSmem(uint8_t* base, int T, int width) {
        uint8_t* p = base;
        a = p;       p += 128 * 128;
        a_lo = p;    p += 128 * 128;
        w1 = p;      p += 64 * 128;
        w1_lo = p;   p += 64 * 128;
        w2 = p;      p += 64 * 128;
        w2_lo = p;   p += 64 * 128;
        kstage = (float*)p;   p += sizeof(float) * kRows * 16;
        ca = (float*)p;       p += pad16(sizeof(float) * kSamples * width);
        gc = (float*)p;       p += pad16(sizeof(float) * kSamples * width);
        attw = (float*)p;     p += pad16(sizeof(float) * kSamples * T);
        mask = (uint32_t*)p;  p += pad16(sizeof(uint32_t) * kSamples * T * 3);
        ix_his = (int64_t*)p; p += pad16(sizeof(int64_t) * kSamples * T);
        ix_len = (int64_t*)p; p += sizeof(int64_t) * kSamples;
        nrm = (float*)p;      p += sizeof(float) * kSamples;
        gnrm = (float*)p;     p += sizeof(float) * kSamples;
        vec = (float*)p;      p += sizeof(float) * kH2;
        q = (float*)p;        p += sizeof(float) * kSamples * 16;
        att = (float*)p;      p += sizeof(float) * kSamples * 16;
        gq = (float*)p;       p += sizeof(float) * kSamples * 16;
        gt = (float*)p;       p += sizeof(float) * kSamples * 16;
        dot = (float*)p;      p += sizeof(float) * 8;
        score = (float*)p;    p += sizeof(float) * kRows;
        wt = (float*)p;       p += sizeof(float) * kRows;
        len = (int*)p;        p += sizeof(int) * 3 * kSamples;     // [0,8) lengths, [8,17) their prefix sums
        bar = (uint64_t*)p;   p += 8;
        bar_w = (uint64_t*)p; p += 8;
        tmem_slot = (uint32_t*)p;
    }
    static size_t bytes(int T, int width) {
        return 16 + 1024 /* alignment slack */ + 2 * (128 * 128 + 2 * 64 * 128) + sizeof(float) * kRows * 16 +
               2 * pad16(sizeof(float) * kSamples * width) + pad16(sizeof(float) * kSamples * T) +
               pad16(sizeof(uint32_t) * kSamples * T * 3) + pad16(sizeof(int64_t) * kSamples * T) +
               sizeof(int64_t) * kSamples + sizeof(float) * (2 * kSamples + kH2 + 4 * kSamples * 16 + 8 + 2 * kRows) +
               sizeof(int) * 3 * kSamples + 16;
    }
};

// n 4-byte words, global -> shared, asynchronously: 16-byte copies when the block allows it.
__device__ __forceinline__ void copy_words_async(void* dst_smem, const void* src, int n, int tid) {
    const uint32_t dst = smem_u32(dst_smem);
    const char* s = reinterpret_cast<const char*>(src);
    if ((n & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        for (int i = tid; i < (n >> 2); i += kTcThreads)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16 * i), "l"(s + 16 * (size_t)i) : "memory");
    } else {
        for (int i = tid; i < n; i += kTcThreads)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4 * i), "l"(s + 4 * (size_t)i) : "memory");
    }
}

// Everything the backward of a group reads that does not depend on an index: issued one group ahead.
__device__ __forceinline__ void issue_group_bwd(const DinParams& p, const TcBwdSmem& sm, int64_t group, int tid,
                                                const float* concat_all, const float* norm, const float* att_w,
                                                const uint32_t* masks, const float* g_concat, const float* g_norm) {
    const int64_t b0 = group * kSamples;
    const int n = (int)((p.B - b0) < kSamples ? (p.B - b0) : kSamples);
    copy_words_async(sm.ix_his, p.his_idx + b0 * p.T, 2 * n * p.T, tid);
    copy_words_async(sm.attw, att_w + b0 * p.T, n * p.T, tid);
    copy_words_async(sm.mask, masks + b0 * p.T * 3, 3 * n * p.T, tid);
    copy_words_async(sm.ca, concat_all + b0 * p.width, n * p.width, tid);
    if (g_concat) copy_words_async(sm.gc, g_concat + b0 * p.width, n * p.width, tid);
    else for (int i = tid; i < n * p.width; i += kTcThreads) sm.gc[i] = 0.f;
    if (tid < n) {
        cp_async8(sm.ix_len + tid, p.his_len + b0 + tid);
        if (g_norm) {
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(sm.nrm + tid)), "l"(norm + b0 + tid) : "memory");
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(sm.gnrm + tid)), "l"(g_norm + b0 + tid) : "memory");
        } else {
            sm.nrm[tid] = 0.f;
            sm.gnrm[tid] = 0.f;
        }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// Tensor-core backward (D = 16): g_score -> (x W2) -> relu' -> (x W1) -> g_cross on tcgen05 with
// split-bf16 operands; B operands are the transposed weights of the pack (W2^T [64][32] and
// W1^T [64][64], both K-major for these products).  Same outputs as din_bwd_kernel.
__global__ void __launch_bounds__(kTcThreads)
din_bwd_tc_kernel(const __grid_constant__ DinParams p, const float* __restrict__ concat_all,
                  const float* __restrict__ norm, const float* __restrict__ att_w,
                  const uint32_t* __restrict__ masks, const float* __restrict__ g_concat,
                  const float* __restrict__ g_norm, float* __restrict__ g_row,
                  float* __restrict__ g_hist, int32_t* err_flag) {
    extern __shared__ uint8_t smem_raw_tc[];
    uint8_t* base = smem_raw_tc + ((1024u - (smem_u32(smem_raw_tc) & 1023u)) & 1023u);
    TcBwdSmem sm(base, p.T, p.width);
    constexpr int D = 16;
    const int T = p.T, W = p.width;
    const MlpLayout L(D);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t n_groups = (p.B + kSamples - 1) / kSamples;

    // first group static (the grid never exceeds the group count); its inputs fly during the set-up
    int64_t group = blockIdx.x;
    issue_group_bwd(p, sm, group, tid, concat_all, norm, att_w, masks, g_concat, g_norm);

    if (tid == 0) {
        mbar_init(sm.bar, 1);
        mbar_init(sm.bar_w, 1);
        // w1 | w1_lo | w2 | w2_lo (W1^T, W2^T) in one bulk (TMA) copy
        mbar_expect_tx(sm.bar_w, kTileBwdBytes);
        bulk_copy_g2s(sm.w1, p.mlp_tiles + kTileFwdBytes, kTileBwdBytes, sm.bar_w);
    }
    if (warp == 0) tmem_alloc(sm.tmem_slot, kTcTmemCols);
    for (int i = tid; i < kH2; i += kTcThreads) sm.vec[i] = __ldg(p.mlp + L.w3 + i);
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    mbar_wait(sm.bar_w, 0);
    const uint32_t tmem = *sm.tmem_slot;
    const float* w3 = sm.vec;
    const uint64_t a_desc[2]  = {umma_desc(smem_u32(sm.a)), umma_desc(smem_u32(sm.a_lo))};
    const uint64_t w1_desc[2] = {umma_desc(smem_u32(sm.w1)), umma_desc(smem_u32(sm.w1_lo))};
    const uint64_t w2_desc[2] = {umma_desc(smem_u32(sm.w2)), umma_desc(smem_u32(sm.w2_lo))};
    const uint32_t my_tmem = tmem + ((uint32_t)(warp * 32) << 16);
    float* pool = reinterpret_cast<float*>(sm.a_lo);     // [128][17], free once the second MMA has read a_lo
    uint32_t phase = 0;

    __shared__ unsigned int group_slot;
    while (group < n_groups) {                       // persistent: groups of 8 samples
        unsigned int next_draw = 0;                  // drawn now, published at a tile barrier, used by the last tile
        if (tid == 0) next_draw = gridDim.x + atomicAdd(&g_din_next[1], 1u);
        const int64_t b0 = group * kSamples;
        const int n_samples = (int)((p.B - b0) < kSamples ? (p.B - b0) : kSamples);
        wait_rows();                                 // the group's inputs (issue_group_bwd) have landed ...
        __syncthreads();                             // ... for every thread
        store_len_prefix(sm.len, sm.ix_len, n_samples, T, tid);
        for (int i = tid; i < n_samples * D; i += kTcThreads) {
            const int s = i / D, e = i - s * D;
            sm.q[i] = sm.ca[s * W + p.tgt_off + e];
            const float nv = sm.nrm[s];
            const float scale = nv > 0.f ? sm.gnrm[s] / nv : 0.f;
            sm.att[i] = fmaf(scale, sm.ca[s * W + p.att_off + e], sm.gc[s * W + p.att_off + e]);   // g_att
            sm.gq[i]  = 0.f;
        }
        // g_row of every column but the target's (those wait for g_q): smem -> coalesced stores
        for (int i = tid; i < n_samples * W; i += kTcThreads) {
            const int s = i / W, c = i - s * W;
            const float nv = sm.nrm[s];
            const float scale = nv > 0.f ? sm.gnrm[s] / nv : 0.f;
            float g = sm.gc[i];
            if (c >= p.l2_from) g = fmaf(scale, sm.ca[i], g);
            if (c >= p.tgt_off && c < p.tgt_off + D) sm.gt[s * D + c - p.tgt_off] = g;
            else g_row[b0 * W + i] = g;
        }
        __syncthreads();

        int s_begin = 0;
        TcTile cur = plan_tile_tc(sm.len, n_samples, 0, tid);
        {                                            // first tile of the group: exposed latency
            if (cur.on) {
                const int64_t row = checked_row(sm.ix_his[cur.my_s * T + cur.my_t], p.his_rows, err_flag);
                const uint32_t dst = smem_u32(sm.kstage + tid * 16);
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16 * kstage_chunk(tid, c)), "l"(p.his_w + row * 16 + 4 * c) : "memory");
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
        }
        while (s_begin < n_samples) {
            wait_rows();
            const bool on = cur.on;
            const int my_s = cur.my_s, my_t = cur.my_t;
            const bool has_next = cur.s_end < n_samples;
            TcTile nxt = cur;
            // issued while the tensor core works: the rows of the next tile or, on the last tile of the
            // group, the inputs of the next group (everything staged was consumed before the barrier)
            auto shadow_work = [&]() {
                if (has_next) {
                    nxt = plan_tile_tc(sm.len, n_samples, cur.s_end, tid);
                    if (nxt.on) {
                        const int64_t row = checked_row(sm.ix_his[nxt.my_s * T + nxt.my_t], p.his_rows, err_flag);
                        const uint32_t dst = smem_u32(sm.kstage + tid * 16);
#pragma unroll
                        for (int c = 0; c < 4; ++c)
                            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16 * kstage_chunk(tid, c)), "l"(p.his_w + row * 16 + 4 * c) : "memory");
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                } else if ((int64_t)group_slot < n_groups) {
                    issue_group_bwd(p, sm, (int64_t)group_slot, tid, concat_all, norm, att_w, masks, g_concat, g_norm);
                }
            };
            if (cur.n_rows > 0) {
                float k[16], gatt[16];
                float w = 0.f, gw = 0.f;
                uint32_t m1a = 0, m1b = 0, m2 = 0;
#pragma unroll
                for (int e = 0; e < 16; ++e) { k[e] = 0.f; gatt[e] = 0.f; }
                if (on) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float4 v = *reinterpret_cast<const float4*>(sm.kstage + tid * 16 + 4 * kstage_chunk(tid, c));
                        k[4 * c] = v.x; k[4 * c + 1] = v.y; k[4 * c + 2] = v.z; k[4 * c + 3] = v.w;
                    }
#pragma unroll
                    for (int e = 0; e < 16; ++e) { gatt[e] = sm.att[my_s * D + e]; gw = fmaf(gatt[e], k[e], gw); }
                    w = sm.attw[my_s * T + my_t];
                    const uint32_t* mk = sm.mask + (my_s * T + my_t) * 3;
                    m1a = mk[0]; m1b = mk[1]; m2 = mk[2];
                }
                if (p.use_softmax) {          // g_s = w (g_w - sum_u w_u g_w_u) / sqrt(D)
                    sm.wt[tid] = w;
                    sm.score[tid] = gw;
                    __syncthreads();
                    for (int s = s_begin + warp; s < cur.s_end; s += kTcThreads / 32) {
                        const int len = sm.len[s], r0 = tile_row0(sm.len, s_begin, s);
                        float dsum = 0.f;
                        for (int t = lane; t < len; t += 32) dsum = fmaf(sm.wt[r0 + t], sm.score[r0 + t], dsum);
                        dsum = warp_sum(dsum);
                        if (lane == 0) sm.dot[s] = dsum;
                    }
                    __syncthreads();
                    gw = w * (gw - sm.dot[my_s]) * 0.25f;
                }
                if (!on) gw = 0.f;
                // ---- A = g_z2 [128 x 32]
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) v[j] = ((m2 >> (8 * c + j)) & 1u) ? gw * w3[8 * c + j] : 0.f;
                    store_chunk_split(sm.a, sm.a_lo, tid, c, v);
                }
                if (tid == 0) group_slot = next_draw;
                fence_async_smem();
                fence_before();
                __syncthreads();
                if (tid == 0) {
                    fence_after();
#pragma unroll
                    for (int term = 0; term < 3; ++term)
#pragma unroll
                        for (int kk = 0; kk < 2; ++kk)     // K = 32
                            umma_bf16(tmem, a_desc[term == 1] + 2 * kk, w2_desc[term == 2] + 2 * kk, umma_idesc(64),
                                      (term | kk) > 0);
                    umma_commit(sm.bar);
                }
                shadow_work();
                mbar_wait(sm.bar, phase);
                phase ^= 1;
                fence_after();
                // ---- g_z1 = (g_z2 x W2) * relu1'  -> A [128 x 64]
#pragma unroll
                for (int half = 0; half < 2; ++half) {
                    float v[32];
                    tmem_ld32(my_tmem + 32 * half, v);
                    const uint32_t bits = half == 0 ? m1a : m1b;
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        float h8[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) h8[j] = ((bits >> (8 * c + j)) & 1u) ? v[8 * c + j] : 0.f;
                        store_chunk_split(sm.a, sm.a_lo, tid, 4 * half + c, h8);
                    }
                }
                fence_async_smem();
                fence_before();
                __syncthreads();
                if (tid == 0) {
                    fence_after();
#pragma unroll
                    for (int term = 0; term < 3; ++term)
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)     // K = 64
                            umma_bf16(tmem + 64, a_desc[term == 1] + 2 * kk, w1_desc[term == 2] + 2 * kk, umma_idesc(64),
                                      (term | kk) > 0);
                    umma_commit(sm.bar);
                }
                mbar_wait(sm.bar, phase);
                phase ^= 1;
                fence_after();
                // ---- g_cross = [gc_q | gc_k | gc_d | gc_p] -> g_k row, and this row's share of g_q
                float gk[16], gqr[16];
                {
                    float v[32];
                    tmem_ld32(my_tmem + 64, v);
#pragma unroll
                    for (int e = 0; e < 16; ++e) { gqr[e] = v[e]; gk[e] = fmaf(w, gatt[e], v[16 + e]); }
                    tmem_ld32(my_tmem + 96, v);
#pragma unroll
                    for (int e = 0; e < 16; ++e) {
                        const float qe = sm.q[my_s * D + e];
                        gqr[e] += v[e] + v[16 + e] * k[e];
                        gk[e]  += v[16 + e] * qe - v[e];
                    }
                }
                if (on) {
                    float4* dst = reinterpret_cast<float4*>(g_hist + ((b0 + my_s) * T + my_t) * D);
#pragma unroll
                    for (int c = 0; c < 4; ++c) dst[c] = make_float4(gk[4 * c], gk[4 * c + 1], gk[4 * c + 2], gk[4 * c + 3]);
                }
#pragma unroll
                for (int e = 0; e < 16; ++e) pool[tid * 17 + e] = on ? gqr[e] : 0.f;
                fence_before();
                __syncthreads();
                for (int item = tid; item < (cur.s_end - s_begin) * 16; item += kTcThreads) {
                    const int s = s_begin + (item >> 4), e = item & 15;
                    const int len = sm.len[s], r0 = tile_row0(sm.len, s_begin, s);
                    float a = 0.f;
                    for (int t = 0; t < len; ++t) a += pool[(r0 + t) * 17 + e];
                    sm.gq[s * 16 + e] = a;
                }
            } else {                                     // a tile of empty histories: nothing for the tensor core
                if (tid == 0) group_slot = next_draw;
                __syncthreads();
                shadow_work();
            }
            if (p.use_softmax) {      // no history: uniform weights, gradient g_att / T on every position
                for (int s = s_begin; s < cur.s_end; ++s) {
                    if (sm.len[s] != 0) continue;
                    const float u = 1.0f / (float)T;
                    for (int i = tid; i < T * D; i += kTcThreads)
                        g_hist[(b0 + s) * T * D + i] = u * sm.att[s * D + (i % D)];
                }
            }
            __syncthreads();
            s_begin = cur.s_end;
            cur = nxt;
        }

        // the target's columns of g_row: upstream + L2-norm share (gt) + the attention unit's g_q
        for (int i = tid; i < n_samples * D; i += kTcThreads) {
            const int s = i / D, e = i - s * D;
            g_row[(b0 + s) * W + p.tgt_off + e] = sm.gt[i] + sm.gq[i];
        }
        __syncthreads();      // q / len / att / gq / gt are rewritten by the next group
        group = (int64_t)group_slot;     // rewritten only after the next group's first barrier
    }
    scheduler_exit(1);
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, kTcTmemCols);
}

}  // namespace tc

}  // namespace rk

// The fp32 kernels: one CTA per kSamples samples, the DinSmem carve-up as dynamic shared memory.
template <class Kernel, class... Args>
static int din_launch(Kernel kernel, int grid, int D, rk_stream_t stream, Args... args) {
    using namespace rk;
    const size_t smem = DinSmem::bytes(D);
    RK_CHECK_ARG(smem <= 227 * 1024, "din: %zu bytes of shared memory", smem);
    RK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kernel<<<grid, kDinThreads, smem, (cudaStream_t)stream>>>(args...);
    RK_LAUNCH_CHECK();
    return 0;
}

extern "C" {

int rk_din_mlp_floats(int D) { return rk::MlpLayout(D).total; }

int rk_din_tile_bytes(void) { return (int)(rk::tc::kTileFwdBytes + rk::tc::kTileBwdBytes); }

static int din_pack(const rk_din_args_t* a, rk::DinParams* p) {
    using namespace rk;
    RK_CHECK_ARG(a, "din: args is NULL");
    memset(p, 0, sizeof(*p));
    if (int rc = pack_fields(a->cat, a->n_cat, &p->cat)) return rc;
    RK_CHECK_ARG(a->n_dense >= 0 && a->n_dense <= kMaxDense, "din: n_dense=%d", a->n_dense);
    for (int c = 0; c < a->n_dense; ++c) {
        RK_CHECK_ARG(a->dense_cols && a->dense_cols[c], "din: dense column %d is NULL", c);
        p->dense_col[c] = a->dense_cols[c];
    }
    p->dense_stride = a->dense_stride;
    p->n_dense = a->n_dense;
    const int D = a->history.dim;
    RK_CHECK_ARG(D >= 4 && D <= 32 && D % 4 == 0, "din: embedding dim %d not in {4,8,..,32}", D);
    RK_CHECK_ARG(a->target.dim == D, "din: target dim %d != history dim %d", a->target.dim, D);
    RK_CHECK_ARG(a->T >= 0, "din: history length %d is negative", a->T);
    RK_CHECK_ARG(a->precision != RK_DIN_BF16_TENSOR || a->T <= kRows,
                 "din: the tensor-core activation unit takes histories of at most %d positions (got %d); "
                 "use RK_DIN_FP32 for longer ones", kRows, a->T);
    RK_CHECK_ARG(a->target.weight && a->target.idx && ((a->history.weight && a->history.idx) || a->T == 0) &&
                 a->hist_len && a->mlp, "din: NULL pointer");
    RK_CHECK_ARG(((uintptr_t)a->history.weight % 16) == 0, "din: history table must be 16-byte aligned");
    p->tgt_w = a->target.weight;   p->tgt_idx = a->target.idx;   p->tgt_rows = a->target.rows;
    p->tgt_off = a->target.out_off;
    p->his_w = a->history.weight;  p->his_idx = a->history.idx;  p->his_rows = a->history.rows;
    p->his_len = a->hist_len;
    p->T = a->T;  p->D = D;  p->att_off = a->att_off;  p->width = a->width;
    p->l2_from = a->l2_from;  p->use_softmax = a->use_softmax;
    p->mlp = a->mlp;  p->B = a->B;
    p->mlp_tiles = (const uint8_t*)a->mlp_tiles;
    RK_CHECK_ARG(a->precision != RK_DIN_BF16_TENSOR || a->mlp_tiles,
                 "din: mlp_tiles is NULL (RK_DIN_BF16_TENSOR needs rk_din_tile_bytes() bytes of scratch)");
    RK_CHECK_ARG(((uintptr_t)a->mlp_tiles % 128) == 0, "din: mlp_tiles must be 128-byte aligned");
    RK_CHECK_ARG(p->width > 0 && p->att_off + D <= p->width && p->tgt_off + D <= p->width, "din: bad layout");
    return 0;
}

int rk_din_fwd(const rk_din_args_t* args, float* concat_all, float* norm, float* att_w,
               uint32_t* relu_masks, int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    DinParams p;
    if (int rc = din_pack(args, &p)) return rc;
    RK_CHECK_ARG(concat_all && (att_w || p.T == 0), "din_fwd: NULL output");
    if (p.B == 0) return 0;
    if (args->precision == RK_DIN_BF16_TENSOR && p.T > 0) {
        RK_CHECK_ARG(p.D == 16, "din_fwd: the tensor-core activation unit is built for D = 16 (got %d)", p.D);
        const size_t smem_tc = tc::TcFwdSmem::bytes(p.width, p.T, p.cat.F);
        constexpr int per_sm = 3;
        auto kernel = tc::din_fwd_tc_kernel;
        RK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc));
        // Persistent CTAs drawing groups of samples from a device-side counter: static striding was
        // measured slower than one CTA per group (158 vs 101 us) because group work varies with the
        // history lengths; dynamic draws keep the balance and pay the per-CTA setup once.
        const int n_groups = (int)ceil_div(p.B, tc::kTcGroup);
        const int grid_tc = n_groups < sm_count() * per_sm ? n_groups : sm_count() * per_sm;
        // both directions' operand tiles, once per forward
        tc::din_weight_tiles_kernel<<<6, 256, 0, (cudaStream_t)stream_>>>(p.mlp, (uint8_t*)args->mlp_tiles);
        RK_LAUNCH_CHECK();
        kernel<<<grid_tc, tc::kTcThreads, smem_tc, (cudaStream_t)stream_>>>(
            p, concat_all, norm, att_w, relu_masks, err_flag);
        RK_LAUNCH_CHECK();
        return 0;
    }
    // T == 0 (every history empty) runs no activation unit, so both precisions take the fp32 kernel
    RK_CHECK_ARG(args->precision == RK_DIN_FP32 || p.T == 0, "din_fwd: unknown precision %d", args->precision);
    return din_launch(din_fwd_kernel, (int)ceil_div(p.B, kSamples), p.D, stream_, p, concat_all, norm, att_w,
                      relu_masks, err_flag);
}

int rk_din_bwd(const rk_din_args_t* args, const float* concat_all, const float* norm,
               const float* att_w, const uint32_t* relu_masks, const float* g_concat,
               const float* g_norm, float* g_row, float* g_hist, int32_t* err_flag,
               rk_stream_t stream_) {
    using namespace rk;
    DinParams p;
    if (int rc = din_pack(args, &p)) return rc;
    RK_CHECK_ARG(concat_all && g_row && ((att_w && relu_masks && g_hist) || p.T == 0), "din_bwd: NULL pointer");
    RK_CHECK_ARG(!g_norm || norm, "din_bwd: g_norm without the saved norms");
    if (p.B == 0) return 0;
    const int grid = (int)ceil_div(p.B, kSamples);
    if (args->precision == RK_DIN_BF16_TENSOR && p.T > 0) {
        RK_CHECK_ARG(p.D == 16, "din_bwd: the tensor-core activation unit is built for D = 16 (got %d)", p.D);
        const size_t smem_tc = tc::TcBwdSmem::bytes(p.T, p.width);
        RK_CHECK_ARG(smem_tc <= 227 * 1024, "din_bwd: %zu bytes of shared memory (width %d)", smem_tc, p.width);
        RK_CUDA(cudaFuncSetAttribute(tc::din_bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)smem_tc));
        // Two CTAs need ~190 KB; with the carve-out the driver would pick for that (196 KB) nothing else fits on
        // the SM while they are resident, and the sort of the history ids (plan_sort.cu, 21 KB per CTA, on its own
        // stream) would have to wait for this kernel to drain.  The full 228 KB leaves it room to run alongside;
        // this kernel's global traffic is cp.async / streaming and does not miss the L1 it gives up.
        RK_CUDA(cudaFuncSetAttribute(tc::din_bwd_tc_kernel, cudaFuncAttributePreferredSharedMemoryCarveout,
                                     (int)cudaSharedmemCarveoutMaxShared));
        // persistent CTAs, two per SM by shared memory; the grid never exceeds the group count
        constexpr int per_sm = 2;
        const int grid_tc = grid < sm_count() * per_sm ? grid : sm_count() * per_sm;
        tc::din_bwd_tc_kernel<<<grid_tc, tc::kTcThreads, smem_tc, (cudaStream_t)stream_>>>(
            p, concat_all, norm, att_w, relu_masks, g_concat, g_norm, g_row, g_hist, err_flag);
        RK_LAUNCH_CHECK();
        return 0;
    }
    RK_CHECK_ARG(args->precision == RK_DIN_FP32 || p.T == 0, "din_bwd: unknown precision %d", args->precision);
    return din_launch(din_bwd_kernel, grid, p.D, stream_, p, concat_all, norm, att_w, relu_masks, g_concat, g_norm,
                      g_row, g_hist, err_flag);
}

}  // extern "C"
