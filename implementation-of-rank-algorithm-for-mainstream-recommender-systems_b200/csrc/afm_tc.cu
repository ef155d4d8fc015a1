// afm_tc.cu — AFM's attention pooling (AFM/afm.py:92-115) with the attention MLP on tcgen05.
// Same contract as afm.cu (rk_afm_fwd / rk_afm_bwd); selected per module (AFM.attention_precision).
//
// Rows of a tile are (sample, pair) couples: S = 128 / P whole samples per 128-row tile.
//   forward : pre = V W1^T on the tensor core (V = e_i * e_j, split-bf16: hi.hi + lo.hi + hi.lo,
//             fp32 accumulation in TMEM), then per row s = w2 . relu(pre + b1) + b2 straight from
//             TMEM, softmax over the sample's rows, out = sum_p a_p v_p.
// Operand tiles: one 128-byte line per row holding [hi(Kp) | lo(Kp)] bf16 (Kp = D rounded up to
// 16, <= 32), so the three split terms are three (A k-slice, B k-slice) pairings of the same two
// tiles.  HBM traffic is the same as the SIMT kernel's (idx + rows in, out written once).
#include <string.h>
#include "common.cuh"
#include "umma.cuh"
#include "prof.cuh"

namespace rk {
namespace tc {

constexpr int kAfmTcThreads = 128;
constexpr int kAfmTcRows    = 128;
constexpr int kAfmTcMaxS    = 16;
constexpr int kAfmTcMaxSF   = 64;    // S * F <= 64 for every F in [2,16]

struct AfmTcParams {
    FieldSet     fs;
    const float* w1;   // [A][D]
    const float* b1;   // [A]
    const float* w2;   // [A]
    const float* b2;   // [1]
    int32_t      D, Kp, A, Ap, P, S, estride;
    int64_t      B, n_tiles;
    const uint8_t* tiles;   // operand tiles made once per forward by afm_weight_tiles_kernel
};

// Image written once per forward by afm_weight_tiles_kernel and fetched by one / two bulk (TMA) copies per CTA:
//   [B1 16 KB: W1 as the B operand, line n = [hi | lo] of W1[n][:]] [B2 16 KB: w2[a] W1[a][d] transposed, hi lines | lo
//   lines, two K panels] [max |W1| as one float]
constexpr uint32_t kAfmTileB1 = 128 * 128, kAfmTileB2 = 2 * 64 * 128, kAfmTileBytes = kAfmTileB1 + kAfmTileB2 + 16;

struct AfmTcFwdSmem {
    uint8_t *a1, *b1t;              // [128][128 B], [Ap][128 B]  (b1t = W1 as the B operand)
    float   *e[2];                  // gathered rows of the tile, [S][F][estride], double buffered
    int64_t *ix[2];                 // raw indices of the tiles after next
    float   *bias, *w2, *score, *attn;
    int     *pi, *pj;
    uint64_t *bar, *bar_w;
    uint32_t* tmem_slot;
    __device__ AfmTcFwdSmem(uint8_t* base, const AfmTcParams& p) {
        uint8_t* q = base;
        a1 = q;   q += 128 * 128;
        b1t = q;  q += 128 * 128;
        const size_t eb = sizeof(float) * p.S * p.fs.F * p.estride;
        e[0] = (float*)q;  q += eb;
        e[1] = (float*)q;  q += eb;
        ix[0] = (int64_t*)q;  q += sizeof(int64_t) * kAfmTcMaxSF;
        ix[1] = (int64_t*)q;  q += sizeof(int64_t) * kAfmTcMaxSF;
        bias = (float*)q;  q += sizeof(float) * p.Ap;
        w2 = (float*)q;    q += sizeof(float) * p.Ap;
        score = (float*)q; q += sizeof(float) * kAfmTcRows;
        attn = (float*)q;  q += sizeof(float) * kAfmTcRows;
        pi = (int*)q;      q += sizeof(int) * 128;
        pj = (int*)q;      q += sizeof(int) * 128;
        bar = (uint64_t*)q; q += 8;
        bar_w = (uint64_t*)q; q += 8;
        tmem_slot = (uint32_t*)q;
    }
    static size_t bytes(const AfmTcParams& p) {
        return 1024 + 2 * 128 * 128 + 2 * sizeof(float) * p.S * p.fs.F * p.estride + sizeof(float) * (2 * p.Ap + 2 * kAfmTcRows) +
               sizeof(int) * 256 + 32 + 2 * sizeof(int64_t) * 64;
    }
};

// fp32 x[n] (n <= 32, zero padded to Kp) -> line `r` of a [hi | lo] operand tile
template <int KP>
__device__ __forceinline__ void store_line_split(uint8_t* tile, int r, const float (&x)[KP]) {
    constexpr int CH = KP / 8;                       // 16-byte chunks per half
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        float hi8[8], lo8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            hi8[j] = x[8 * c + j];
            lo8[j] = x[8 * c + j] - __bfloat162float(__float2bfloat16_rn(x[8 * c + j]));
        }
        store_chunk(tile, r, c, hi8);
        store_chunk(tile, r, CH + c, lo8);
    }
}

// Input staging, two tiles deep: the indices of tile t+2 are copied to shared memory (8-byte
// cp.async) while the rows of tile t+1 are gathered with 16-byte cp.async from the indices that
// landed one tile earlier, all of it issued in the shadow of tile t's first MMA.  Only the very
// first tile of a CTA reads its indices with ordinary loads.
// item / d for 0 <= item < 1024, 1 <= d <= 16, through a float reciprocal (exact there: (item + 0.5) / d is at
// least 1/32 away from an integer, the product's rounding error is below 1e-4); a runtime integer division is
// ~20 instructions, and these loops decompose two or three item numbers per tile
__device__ __forceinline__ int small_div(int item, float inv_d) { return (int)(((float)item + 0.5f) * inv_d); }

__device__ __forceinline__ void afm_issue_idx(const AfmTcParams& p, int64_t* ix, int64_t tile, int tid) {
    const int F = p.fs.F;
    const float inv_f = 1.0f / (float)F;
    const int64_t b0 = tile * p.S;
    const int n_s = (int)((p.B - b0) < p.S ? (p.B - b0) : p.S);
    for (int item = tid; item < n_s * F; item += kAfmTcThreads) {
        const int s = small_div(item, inv_f), f = item - s * F;
        cp_async8(ix + item, p.fs.idx[f] + b0 + s);
    }
}
__device__ __forceinline__ void afm_issue_rows(const AfmTcParams& p, float* e, const int64_t* ix, int64_t tile, int tid,
                                               int32_t* err_flag) {
    const int F = p.fs.F, c4 = p.D >> 2;
    const int64_t b0 = tile * p.S;
    const int n_s = (int)((p.B - b0) < p.S ? (p.B - b0) : p.S);
    const float inv_c4 = 1.0f / (float)c4, inv_f = 1.0f / (float)F;
    for (int item = tid; item < n_s * F * c4; item += kAfmTcThreads) {
        const int sf = small_div(item, inv_c4), c = item - sf * c4, s = small_div(sf, inv_f), f = sf - s * F;
        const int64_t raw = ix ? ix[sf] : __ldg(p.fs.idx[f] + b0 + s);
        const int64_t row = checked_row(raw, p.fs.rows[f], err_flag);
        cp_async16(e + (s * F + f) * p.estride + 4 * c, p.fs.weight[f] + row * p.D + 4 * c);
    }
}

// ---- the weight operand tiles, written into the global image by afm_weight_tiles_kernel
// B1 line n = [hi | lo] of W1[n][:], zero beyond A / D
template <int KP>
__device__ __forceinline__ void afm_build_b1(uint8_t* b1t, const float* __restrict__ w1, int A, int D, int lines, int tid,
                                             int n_threads) {
    for (int item = tid; item < lines * (KP / 8); item += n_threads) {
        const int n = item / (KP / 8), c = item - n * (KP / 8);
        float hi8[8], lo8[8];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n < A && 8 * c + 4 * h < D) w = __ldg(reinterpret_cast<const float4*>(w1 + n * D + 8 * c + 4 * h));
            hi8[4 * h] = w.x; hi8[4 * h + 1] = w.y; hi8[4 * h + 2] = w.z; hi8[4 * h + 3] = w.w;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) lo8[j] = hi8[j] - __bfloat162float(__float2bfloat16_rn(hi8[j]));
        store_chunk(b1t, n, c, hi8);
        store_chunk(b1t, n, KP / 8 + c, lo8);
    }
}
// B2 lines n < KP: hi of w2[a] W1[a][n]; n >= KP: lo.  K = a, 64 per panel.  W1 is read row-major (coalesced
// float4) and scattered into the transposed, pre-zeroed tile two bytes at a time.
template <int KP>
__device__ __forceinline__ void afm_scatter_b2(uint8_t* b2t, const float* __restrict__ w1, const float* __restrict__ w2,
                                               int A, int D, int tid, int n_threads) {
    for (int item = tid; item < A * (D >> 2); item += n_threads) {
        const int a = item / (D >> 2), d0 = 4 * (item - a * (D >> 2));
        const float4 w4 = __ldg(reinterpret_cast<const float4*>(w1 + a * D + d0));
        const float w2a = __ldg(w2 + a);
        const float w[4] = {w2a * w4.x, w2a * w4.y, w2a * w4.z, w2a * w4.w};
        uint8_t* panel = b2t + (a >> 6) * (64 * 128);
        const int c = (a & 63) >> 3, e = (a & 7) * 2;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const __nv_bfloat16 hi = __float2bfloat16_rn(w[j]);
            const __nv_bfloat16 lo = __float2bfloat16_rn(w[j] - __bfloat162float(hi));
            const int nh = d0 + j, nl = KP + d0 + j;
            *reinterpret_cast<__nv_bfloat16*>(panel + nh * 128 + ((c ^ (nh & 7)) << 4) + e) = hi;
            *reinterpret_cast<__nv_bfloat16*>(panel + nl * 128 + ((c ^ (nl & 7)) << 4) + e) = lo;
        }
    }
}

// Once per forward: both directions' weight tiles + max |W1| into the global image (CTA 0: B2, CTA 1: B1 and the max).
// The attention weights are registered parameters, the same for every CTA of both kernels: 592 + 296 CTAs used to
// convert them each for themselves (13 % / 9 % of the forward / backward).
template <int KP>
__global__ void __launch_bounds__(256)
afm_weight_tiles_kernel(const float* __restrict__ w1, const float* __restrict__ w2, int A, int D, uint8_t* __restrict__ tiles) {
    __shared__ float red[8];
    const int tid = threadIdx.x;
    if (blockIdx.x == 0) {
        uint8_t* b2t = tiles + kAfmTileB1;
        for (int i = tid; i < (int)kAfmTileB2 / 16; i += 256) reinterpret_cast<uint4*>(b2t)[i] = make_uint4(0u, 0u, 0u, 0u);
        __syncthreads();
        afm_scatter_b2<KP>(b2t, w1, w2, A, D, tid, 256);
    } else {
        afm_build_b1<KP>(tiles, w1, A, D, 128, tid, 256);
        float m = 0.f;
        for (int i = tid; i < A * D; i += 256) m = fmaxf(m, fabsf(__ldg(w1 + i)));
        m = warp_max(m);
        if ((tid & 31) == 0) red[tid >> 5] = m;
        __syncthreads();
        if (tid == 0) {
            float t = 0.f;
            for (int w = 0; w < 8; ++w) t = fmaxf(t, red[w]);
            *reinterpret_cast<float*>(tiles + kAfmTileB1 + kAfmTileB2) = t;
        }
    }
}

template <int KP>
__global__ void __launch_bounds__(kAfmTcThreads, 4)      // 4 CTAs / SM: at most 128 registers
afm_fwd_tc_kernel(const __grid_constant__ AfmTcParams p, float* __restrict__ out, int32_t* err_flag) {
    extern __shared__ uint8_t afm_tc_raw[];
    uint8_t* base = afm_tc_raw + ((1024u - (smem_u32(afm_tc_raw) & 1023u)) & 1023u);
    AfmTcFwdSmem sm(base, p);
    PROF_DECL
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int F = p.fs.F, D = p.D, P = p.P;
    constexpr int LO = KP / 8;                       // 16-byte units from the hi half to the lo half of a line

    int64_t tile = blockIdx.x;
    if (tile < p.n_tiles) {
        afm_issue_rows(p, sm.e[0], nullptr, tile, tid, err_flag);
        if (tile + gridDim.x < p.n_tiles) afm_issue_idx(p, sm.ix[1], tile + gridDim.x, tid);
        cp_async_commit();
    }

    if (tid == 0) {
        mbar_init(sm.bar, 1);
        mbar_init(sm.bar_w, 1);
        mbar_expect_tx(sm.bar_w, (uint32_t)p.Ap * 128u);          // W1's operand tile in one bulk (TMA) copy
        bulk_copy_g2s(sm.b1t, p.tiles, (uint32_t)p.Ap * 128u, sm.bar_w);
    }
    if (warp == 0) tmem_alloc(sm.tmem_slot, 128);
    for (int n = tid; n < p.Ap; n += kAfmTcThreads) {
        sm.bias[n] = n < p.A ? __ldg(p.b1 + n) : 0.f;
        sm.w2[n]   = n < p.A ? __ldg(p.w2 + n) : 0.f;
    }
    if (tid == 0) {
        int q = 0;
        for (int i = 0; i < F; ++i)
            for (int j = i + 1; j < F; ++j) { sm.pi[q] = i; sm.pj[q] = j; ++q; }
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    mbar_wait(sm.bar_w, 0);
    const uint32_t tmem = *sm.tmem_slot;
    const uint32_t my_tmem = tmem + ((uint32_t)(warp * 32) << 16);
    const uint64_t a_desc = umma_desc(smem_u32(sm.a1)), b_desc = umma_desc(smem_u32(sm.b1t));
    const uint32_t idesc = umma_idesc(p.Ap);
    const float b2 = __ldg(p.b2);
    float* pool = reinterpret_cast<float*>(sm.a1);   // [128][32] floats, chunk-swizzled; A1 is free after the MMA
    uint32_t phase = 0;
    int buf = 0;
    const int c4 = D >> 2;
    int parts = 1, parts_sh = 0;                     // power of two, <= 8, parts * S * D/4 <= threads when possible
    while (parts < 8 && 2 * parts * p.S * c4 <= kAfmTcThreads) { parts <<= 1; ++parts_sh; }
    const int s_row = tid / P, pr_row = tid - s_row * P;        // this thread's (sample, pair) in every tile
    PROF(0);

    for (; tile < p.n_tiles; tile += gridDim.x, buf ^= 1) {
        const int64_t b0 = tile * p.S;
        const int n_s = (int)((p.B - b0) < p.S ? (p.B - b0) : p.S);
        const int n_rows = n_s * P;
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                             // rows copied by every thread are visible
        PROF(1); PROF_COUNT(12);
        // ---- this thread's pair row v = e_i * e_j, split into the A operand line
        const bool on = tid < n_rows;
        const int s = on ? s_row : 0, pr = on ? pr_row : 0;
        float v[KP];
#pragma unroll
        for (int d = 0; d < KP; ++d) v[d] = 0.f;
        if (on) {
            const float* ei = sm.e[buf] + (s * F + sm.pi[pr]) * p.estride;
            const float* ej = sm.e[buf] + (s * F + sm.pj[pr]) * p.estride;
#pragma unroll
            for (int c = 0; c < KP / 4; ++c)
                if (4 * c < D) {
                    const float4 x = *reinterpret_cast<const float4*>(ei + 4 * c);
                    const float4 y = *reinterpret_cast<const float4*>(ej + 4 * c);
                    v[4 * c] = x.x * y.x; v[4 * c + 1] = x.y * y.y; v[4 * c + 2] = x.z * y.z; v[4 * c + 3] = x.w * y.w;
                }
        }
        store_line_split<KP>(sm.a1, tid, v);
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (tid == 0) {
            fence_after();
            PROF(2);
#pragma unroll
            for (int term = 0; term < 3; ++term)         // hi.hi + lo.hi + hi.lo
#pragma unroll
                for (int kk = 0; kk < KP / 16; ++kk)
                    umma_bf16(tmem, a_desc + (term == 1 ? LO : 0) + 2 * kk, b_desc + (term == 2 ? LO : 0) + 2 * kk, idesc,
                              (term | kk) > 0);
            umma_commit(sm.bar);
        }
        // while the tensor core works: the next tile's rows (the other e buffer was last read two barriers ago)
        if (tile + gridDim.x < p.n_tiles) {
            afm_issue_rows(p, sm.e[buf ^ 1], sm.ix[buf ^ 1], tile + gridDim.x, tid, err_flag);
            if (tile + 2 * (int64_t)gridDim.x < p.n_tiles) afm_issue_idx(p, sm.ix[buf], tile + 2 * (int64_t)gridDim.x, tid);
            cp_async_commit();
        }
        mbar_wait(sm.bar, phase);
        phase ^= 1;
        fence_after();
        PROF(3);
        float sc = b2;
        for (int ch = 0; ch < p.Ap / 64; ++ch) {
            float h[64];
            tmem_ld64(my_tmem + 64 * ch, h);
#pragma unroll
            for (int c = 0; c < 16; ++c) {               // 16-byte broadcast loads of bias and w2
                const float4 bb = *reinterpret_cast<const float4*>(sm.bias + 64 * ch + 4 * c);
                const float4 ww = *reinterpret_cast<const float4*>(sm.w2 + 64 * ch + 4 * c);
                sc = fmaf(fmaxf(h[4 * c] + bb.x, 0.f), ww.x, sc);
                sc = fmaf(fmaxf(h[4 * c + 1] + bb.y, 0.f), ww.y, sc);
                sc = fmaf(fmaxf(h[4 * c + 2] + bb.z, 0.f), ww.z, sc);
                sc = fmaf(fmaxf(h[4 * c + 3] + bb.w, 0.f), ww.w, sc);
            }
        }
        if (p.Ap & 32) {
            float h[32];
            tmem_ld32(my_tmem + (p.Ap - 32), h);
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float4 bb = *reinterpret_cast<const float4*>(sm.bias + p.Ap - 32 + 4 * c);
                const float4 ww = *reinterpret_cast<const float4*>(sm.w2 + p.Ap - 32 + 4 * c);
                sc = fmaf(fmaxf(h[4 * c] + bb.x, 0.f), ww.x, sc);
                sc = fmaf(fmaxf(h[4 * c + 1] + bb.y, 0.f), ww.y, sc);
                sc = fmaf(fmaxf(h[4 * c + 2] + bb.z, 0.f), ww.z, sc);
                sc = fmaf(fmaxf(h[4 * c + 3] + bb.w, 0.f), ww.w, sc);
            }
        }
        sm.score[tid] = sc;
        fence_before();
        __syncthreads();
        PROF(4);
        // ---- softmax over the sample's P rows: one warp per sample
        for (int ss = warp; ss < n_s; ss += kAfmTcThreads / 32) {
            const int r0 = ss * P;
            float mx = -INFINITY;
            for (int q = lane; q < P; q += 32) mx = fmaxf(mx, sm.score[r0 + q]);
            mx = warp_max(mx);
            float ex[4], sum = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int q = lane + 32 * i;
                ex[i] = q < P ? expf(sm.score[r0 + q] - mx) : 0.f;
                sum += ex[i];
            }
            const float inv = 1.0f / warp_sum(sum);
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (lane + 32 * i < P) sm.attn[r0 + lane + 32 * i] = ex[i] * inv;
        }
        __syncthreads();
        PROF(5);
        // ---- out[s][:] = sum_p a_p v_p through the (now free) A tile
        {
            const float a = on ? sm.attn[tid] : 0.f;
#pragma unroll
            for (int c = 0; c < KP / 4; ++c)
                *reinterpret_cast<float4*>(pool + tid * 32 + 4 * ((c ^ tid) & 7)) =
                    make_float4(a * v[4 * c], a * v[4 * c + 1], a * v[4 * c + 2], a * v[4 * c + 3]);
        }
        __syncthreads();
        PROF(6);
        // `parts` adjacent lanes share one 16-byte output chunk: lane `part` adds pairs part, part + parts, ...
        // and the parts are folded by a fixed shuffle tree
        for (int it0 = 0; it0 < n_s * c4 * parts; it0 += kAfmTcThreads) {
            const int item = it0 + tid, o = item >> parts_sh, part = item & (parts - 1);
            const int ss = small_div(o, 1.0f / (float)c4), c = o - ss * c4;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            if (o < n_s * c4)
                for (int q = part; q < P; q += parts) {
                    const int r = ss * P + q;
                    const float4 x = *reinterpret_cast<const float4*>(pool + r * 32 + 4 * ((c ^ r) & 7));
                    acc.x += x.x; acc.y += x.y; acc.z += x.z; acc.w += x.w;
                }
            for (int w = parts >> 1; w > 0; w >>= 1) {
                acc.x += __shfl_xor_sync(kFull, acc.x, w); acc.y += __shfl_xor_sync(kFull, acc.y, w);
                acc.z += __shfl_xor_sync(kFull, acc.z, w); acc.w += __shfl_xor_sync(kFull, acc.w, w);
            }
            if (o < n_s * c4 && part == 0) *reinterpret_cast<float4*>(out + (b0 + ss) * D + 4 * c) = acc;
        }
        __syncthreads();                             // pool / score / attn are rewritten by the next tile
        PROF(7);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    fence_before();
    PROF_END;
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}


// ---- backward ------------------------------------------------------------------------------
// Per row r = (sample, pair):  pre = v W1^T + b1,  mask = [pre > 0],  s = w2 . relu(pre) + b2,
// a = softmax_pairs(s),  g_a = <g_out, v>,  g_s = a (g_a - sum_q a_q g_a_q).
// Everything that touches the hidden layer is written in terms of the 0/1 mask (exact in bf16):
//   g_v[r]  = a g_out + g_s[r] * (mask[r,:] . B2),        B2[d][a] = w2[a] W1[a][d]   (split hi | lo along N)
//   U[a][n] = sum_r mask[r][a] * X[r][n],                  X[r] = g_s[r] * [v_hi | v_lo | 1_hi, 1_lo]
// and the registered-weight gradients follow from U alone (exact identities, no division):
//   dW1[a][d] = w2[a] U[a][d],  db1[a] = w2[a] u0[a],  dw2[a] = sum_d W1[a][d] U[a][d] + b1[a] u0[a]
// (u0 = the "1" columns of U; U[a][d] = U_hi + U_lo).  mask is stored once (K-major for g_v) and read
// a second time as the MN-major (transposed) A operand of the U product, whose accumulator stays
// in TMEM for the whole life of the CTA.  db2 = sum_r g_s (mathematically 0) is summed on the side.
struct AfmTcBwdSmem {
    uint8_t *b3, *a1, *b1t, *a2, *b2t;   // b3 panel 0 and a1 are adjacent: a1 doubles as b3's second panel
    float   *e[2], *gout[2];
    int64_t *ix[2];
    float   *bias, *w2, *score, *attn, *ga, *gs, *dot, *red, *wmax;
    int     *pi, *pj, *pidx;
    uint64_t *bar, *bar_w;
    uint32_t* tmem_slot;
    __device__ AfmTcBwdSmem(uint8_t* base, const AfmTcParams& p) {
        uint8_t* q = base;
        b3 = q;   q += 128 * 128;
        a1 = q;   q += 128 * 128;
        b1t = q;  q += 128 * 128;
        a2 = q;   q += 2 * 128 * 128;
        b2t = q;  q += 2 * 64 * 128;
        const size_t eb = sizeof(float) * p.S * p.fs.F * p.estride;
        e[0] = (float*)q;  q += eb;
        e[1] = (float*)q;  q += eb;
        gout[0] = (float*)q;  q += sizeof(float) * p.S * 32;
        gout[1] = (float*)q;  q += sizeof(float) * p.S * 32;
        ix[0] = (int64_t*)q;  q += sizeof(int64_t) * kAfmTcMaxSF;
        ix[1] = (int64_t*)q;  q += sizeof(int64_t) * kAfmTcMaxSF;
        bias = (float*)q;  q += sizeof(float) * 128;
        w2 = (float*)q;    q += sizeof(float) * 128;
        score = (float*)q; q += sizeof(float) * kAfmTcRows;
        attn = (float*)q;  q += sizeof(float) * kAfmTcRows;
        ga = (float*)q;    q += sizeof(float) * kAfmTcRows;
        gs = (float*)q;    q += sizeof(float) * kAfmTcRows;
        dot = (float*)q;   q += sizeof(float) * kAfmTcMaxS;
        red = (float*)q;   q += sizeof(float) * kAfmTcThreads;
        wmax = (float*)q;  q += sizeof(float) * 4;
        pi = (int*)q;      q += sizeof(int) * 128;
        pj = (int*)q;      q += sizeof(int) * 128;
        pidx = (int*)q;    q += sizeof(int) * 256;
        bar = (uint64_t*)q; q += 8;
        bar_w = (uint64_t*)q; q += 8;
        tmem_slot = (uint32_t*)q;
    }
    static size_t bytes(const AfmTcParams& p) {
        return 1024 + 3 * 128 * 128 + 2 * 128 * 128 + 2 * 64 * 128 + 2 * sizeof(float) * p.S * p.fs.F * p.estride +
               2 * sizeof(float) * p.S * 32 + sizeof(float) * (2 * 128 + 4 * kAfmTcRows + kAfmTcMaxS + kAfmTcThreads) +
               sizeof(int) * 512 + 32 + 2 * sizeof(int64_t) * 64;
    }
};

__device__ __forceinline__ void afm_issue_gout(const AfmTcParams& p, float* dst, const float* g_out, int64_t tile, int tid) {
    const int c4 = p.D >> 2;
    const int64_t b0 = tile * p.S;
    const int n_s = (int)((p.B - b0) < p.S ? (p.B - b0) : p.S);
    for (int item = tid; item < n_s * c4; item += kAfmTcThreads) {
        const int s = small_div(item, 1.0f / (float)c4), c = item - s * c4;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                     ::"r"(smem_u32(dst + s * 32 + 4 * c)), "l"(g_out + (b0 + s) * p.D + 4 * c) : "memory");
    }
}

template <int KP>
__global__ void __launch_bounds__(kAfmTcThreads)
afm_bwd_tc_kernel(const __grid_constant__ AfmTcParams p, const float* __restrict__ g_out, float* __restrict__ g_rows,
                  float* __restrict__ partials, int32_t* err_flag) {
    extern __shared__ uint8_t afm_tc_raw[];
    uint8_t* base = afm_tc_raw + ((1024u - (smem_u32(afm_tc_raw) & 1023u)) & 1023u);
    AfmTcBwdSmem sm(base, p);
    PROF_DECL
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int F = p.fs.F, D = p.D, P = p.P, A = p.A, Ap = p.Ap, c4 = p.D >> 2;
    constexpr int LO = KP / 8;                       // 16-byte units from the hi half to the lo half of a line
    constexpr int N2 = 2 * KP;                       // g_v product: [hi | lo] along N
    constexpr int N3 = 2 * KP + 16;                  // U product:   [v_hi | v_lo | 1_hi, 1_lo, 0 ...]
    constexpr uint32_t kUOff = 128;                  // TMEM columns: [0,128) pre / g_v, [128, 128 + N3) U

    int64_t tile = blockIdx.x;
    if (tile < p.n_tiles) {
        afm_issue_gout(p, sm.gout[0], g_out, tile, tid);
        afm_issue_rows(p, sm.e[0], nullptr, tile, tid, err_flag);
        if (tile + gridDim.x < p.n_tiles) afm_issue_idx(p, sm.ix[1], tile + gridDim.x, tid);
        cp_async_commit();
    }
    if (tid == 0) {
        mbar_init(sm.bar, 1);
        mbar_init(sm.bar_w, 1);
        mbar_expect_tx(sm.bar_w, kAfmTileB1 + kAfmTileB2);        // B1 and B2 in two bulk (TMA) copies on one barrier
        bulk_copy_g2s(sm.b1t, p.tiles, kAfmTileB1, sm.bar_w);
        bulk_copy_g2s(sm.b2t, p.tiles + kAfmTileB1, kAfmTileB2, sm.bar_w);
        // max |W1|: scales the band around zero inside which a pre-activation is recomputed in fp32
        sm.wmax[0] = __ldg(reinterpret_cast<const float*>(p.tiles + kAfmTileB1 + kAfmTileB2));
    }
    if (warp == 0) tmem_alloc(sm.tmem_slot, 256);
    for (int n = tid; n < 128; n += kAfmTcThreads) {
        sm.bias[n] = n < A ? __ldg(p.b1 + n) : 0.f;
        sm.w2[n]   = n < A ? __ldg(p.w2 + n) : 0.f;
    }
    for (int i = tid; i < 2 * 128 * 128 / 16; i += kAfmTcThreads)       // mask columns >= Ap stay zero
        reinterpret_cast<uint4*>(sm.a2)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (tid == 0) {
        int q = 0;
        for (int i = 0; i < F; ++i)
            for (int j = i + 1; j < F; ++j) { sm.pi[q] = i; sm.pj[q] = j; ++q; }
        for (int f = 0; f < F; ++f) {                    // pidx[f][k] = k-th partner of f | its pair row << 8
            int k = 0;
            for (int g = 0; g < F; ++g) {
                if (g == f) continue;
                const int i = f < g ? f : g, j = f < g ? g : f;
                sm.pidx[f * 16 + k++] = g | ((i * (2 * F - i - 1) / 2 + (j - i - 1)) << 8);
            }
        }
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    mbar_wait(sm.bar_w, 0);
    const uint32_t tmem = *sm.tmem_slot;
    const uint32_t my_tmem = tmem + ((uint32_t)(warp * 32) << 16);
    const uint64_t a1_desc = umma_desc(smem_u32(sm.a1)), b1_desc = umma_desc(smem_u32(sm.b1t));
    const float b2 = __ldg(p.b2);
    float* stage = reinterpret_cast<float*>(sm.b3);  // [128][32] floats, chunk-swizzled; b3 is free after the U product
    uint32_t phase = 0;
    int buf = 0;
    bool first_tile = true;
    float gb2_acc = 0.f;
    const int s_row = tid / P, pr_row = tid - s_row * P;        // this thread's (sample, pair) in every tile
    PROF(0);

    for (; tile < p.n_tiles; tile += gridDim.x, buf ^= 1) {
        const int64_t b0 = tile * p.S;
        const int n_s = (int)((p.B - b0) < p.S ? (p.B - b0) : p.S);
        const int n_rows = n_s * P;
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();
        PROF(1); PROF_COUNT(12);
        const bool on = tid < n_rows;
        const int s = on ? s_row : 0, pr = on ? pr_row : 0;
        const float* esm = sm.e[buf];
        float v[KP];
        float ga = 0.f;
#pragma unroll
        for (int d = 0; d < KP; ++d) v[d] = 0.f;
        if (on) {
            const float* ei = esm + (s * F + sm.pi[pr]) * p.estride;
            const float* ej = esm + (s * F + sm.pj[pr]) * p.estride;
            const float* go = sm.gout[buf] + s * 32;
#pragma unroll
            for (int c = 0; c < KP / 4; ++c)
                if (4 * c < D) {
                    const float4 x = *reinterpret_cast<const float4*>(ei + 4 * c);
                    const float4 y = *reinterpret_cast<const float4*>(ej + 4 * c);
                    const float4 g = *reinterpret_cast<const float4*>(go + 4 * c);
                    v[4 * c] = x.x * y.x; v[4 * c + 1] = x.y * y.y; v[4 * c + 2] = x.z * y.z; v[4 * c + 3] = x.w * y.w;
                    ga = fmaf(g.x, v[4 * c], ga); ga = fmaf(g.y, v[4 * c + 1], ga);
                    ga = fmaf(g.z, v[4 * c + 2], ga); ga = fmaf(g.w, v[4 * c + 3], ga);
                }
        }
        sm.ga[tid] = ga;
        store_line_split<KP>(sm.a1, tid, v);
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (tid == 0) {                                  // pre = V W1^T
            fence_after();
            PROF(2);
#pragma unroll
            for (int term = 0; term < 3; ++term)
#pragma unroll
                for (int kk = 0; kk < KP / 16; ++kk)
                    umma_bf16(tmem, a1_desc + (term == 1 ? LO : 0) + 2 * kk, b1_desc + (term == 2 ? LO : 0) + 2 * kk,
                              umma_idesc(Ap), (term | kk) > 0);
            umma_commit(sm.bar);
        }
        if (tile + gridDim.x < p.n_tiles) {              // while the tensor core works: the next tile's inputs
            afm_issue_gout(p, sm.gout[buf ^ 1], g_out, tile + gridDim.x, tid);
            afm_issue_rows(p, sm.e[buf ^ 1], sm.ix[buf ^ 1], tile + gridDim.x, tid, err_flag);
            if (tile + 2 * (int64_t)gridDim.x < p.n_tiles) afm_issue_idx(p, sm.ix[buf], tile + 2 * (int64_t)gridDim.x, tid);
            cp_async_commit();
        }
        mbar_wait(sm.bar, phase);
        phase ^= 1;
        fence_after();
        PROF(3);
        // ---- score and the 0/1 mask line (bf16 1.0 = 0x3F80).  The ReLU decision is the one place where
        // a 1e-6 error of the split-bf16 product can change a gradient by a whole term, so any
        // pre-activation inside the error band around zero is recomputed in fp32 (about one element
        // in 10^4): the mask is then the fp32 kernel's mask.
        float band = 0.f;
#pragma unroll
        for (int d = 0; d < KP; ++d) band += fabsf(v[d]);
        // worst case of the three-term split is ~1.9e-5 * sum|v_d W_d|; errors add like a random walk
        // over the 32 terms, so a third of the worst case bounds them with a wide margin
        band *= 7e-6f * sm.wmax[0];
        // rare path: element a of this row was inside the band -> fp32 value decides the mask bit (the
        // score is left alone: |relu(x)| < band there, far below its own rounding)
        auto recheck = [&](int a) {
            if (a >= A) return;
            float t = 0.f;
#pragma unroll
            for (int d = 0; d < KP; ++d)
                if (d < D) t = fmaf(v[d], __ldg(p.w1 + a * D + d), t);
            const float x = t + sm.bias[a];
            uint8_t* line = sm.a2 + (a >> 6) * (128 * 128) + tid * 128;
            const int c = (a & 63) >> 3;
            *reinterpret_cast<uint16_t*>(line + ((c ^ (tid & 7)) << 4) + (a & 7) * 2) = x > 0.f ? 0x3F80 : 0;
        };
        float sc = b2;
        for (int ch = 0; ch < Ap / 64; ++ch) {           // one 64-column panel of the mask per TMEM load
            float h[64];
            tmem_ld64(my_tmem + 64 * ch, h);
            uint8_t* panel = sm.a2 + ch * (128 * 128);
            float closest = INFINITY;                    // min |pre-activation| of this row in the chunk
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                uint32_t w[4];
                float bb[8], ww[8];                      // 16-byte broadcast loads: bias and w2 of these 8 columns
                *reinterpret_cast<float4*>(bb)     = *reinterpret_cast<const float4*>(sm.bias + 64 * ch + 8 * c);
                *reinterpret_cast<float4*>(bb + 4) = *reinterpret_cast<const float4*>(sm.bias + 64 * ch + 8 * c + 4);
                *reinterpret_cast<float4*>(ww)     = *reinterpret_cast<const float4*>(sm.w2 + 64 * ch + 8 * c);
                *reinterpret_cast<float4*>(ww + 4) = *reinterpret_cast<const float4*>(sm.w2 + 64 * ch + 8 * c + 4);
#pragma unroll
                for (int j2 = 0; j2 < 4; ++j2) {
                    const int j = 8 * c + 2 * j2;
                    const float x0 = h[j] + bb[2 * j2], x1 = h[j + 1] + bb[2 * j2 + 1];
                    h[j] = x0; h[j + 1] = x1;            // kept for the rare path below
                    closest = fminf(closest, fminf(fabsf(x0), fabsf(x1)));
                    sc = fmaf(fmaxf(x0, 0.f), ww[2 * j2], sc);
                    sc = fmaf(fmaxf(x1, 0.f), ww[2 * j2 + 1], sc);
                    w[j2] = (x0 > 0.f ? 0x3F80u : 0u) | (x1 > 0.f ? 0x3F800000u : 0u);
                }
                *reinterpret_cast<uint4*>(panel + tid * 128 + ((c ^ (tid & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
            if (__any_sync(kFull, closest < band)) {     // rare, warp-uniform: which columns, from the registers
                uint32_t near0 = 0, near1 = 0;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    if (fabsf(h[j]) < band) near0 |= 1u << j;
                    if (fabsf(h[32 + j]) < band) near1 |= 1u << j;
                }
                uint64_t near = ((uint64_t)near1 << 32) | near0;
                while (near) { recheck(64 * ch + __ffsll((long long)near) - 1); near &= near - 1; }
            }
        }
        if (Ap & 32) {                                   // Ap = 32 or 96: the last 32 columns
            float h[32];
            tmem_ld32(my_tmem + (Ap - 32), h);
            uint8_t* panel = sm.a2 + ((Ap - 32) >> 6) * (128 * 128);
            float closest = INFINITY;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint32_t w[4];
                float bb[8], ww[8];
                *reinterpret_cast<float4*>(bb)     = *reinterpret_cast<const float4*>(sm.bias + Ap - 32 + 8 * c);
                *reinterpret_cast<float4*>(bb + 4) = *reinterpret_cast<const float4*>(sm.bias + Ap - 32 + 8 * c + 4);
                *reinterpret_cast<float4*>(ww)     = *reinterpret_cast<const float4*>(sm.w2 + Ap - 32 + 8 * c);
                *reinterpret_cast<float4*>(ww + 4) = *reinterpret_cast<const float4*>(sm.w2 + Ap - 32 + 8 * c + 4);
#pragma unroll
                for (int j2 = 0; j2 < 4; ++j2) {
                    const int j = 8 * c + 2 * j2;
                    const float x0 = h[j] + bb[2 * j2], x1 = h[j + 1] + bb[2 * j2 + 1];
                    h[j] = x0; h[j + 1] = x1;
                    closest = fminf(closest, fminf(fabsf(x0), fabsf(x1)));
                    sc = fmaf(fmaxf(x0, 0.f), ww[2 * j2], sc);
                    sc = fmaf(fmaxf(x1, 0.f), ww[2 * j2 + 1], sc);
                    w[j2] = (x0 > 0.f ? 0x3F80u : 0u) | (x1 > 0.f ? 0x3F800000u : 0u);
                }
                const int cc = (((Ap - 32) & 63) >> 3) + c;
                *reinterpret_cast<uint4*>(panel + tid * 128 + ((cc ^ (tid & 7)) << 4)) = make_uint4(w[0], w[1], w[2], w[3]);
            }
            if (__any_sync(kFull, closest < band)) {
                uint32_t near0 = 0;
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (fabsf(h[j]) < band) near0 |= 1u << j;
                while (near0) { recheck(Ap - 32 + __ffs(near0) - 1); near0 &= near0 - 1; }
            }
        }
        sm.score[tid] = sc;
        fence_before();
        __syncthreads();
        PROF(4);
        // ---- softmax over the sample's pairs and g_s: one warp per sample
        for (int ss = warp; ss < n_s; ss += kAfmTcThreads / 32) {
            const int r0 = ss * P;
            float mx = -INFINITY;
            for (int q = lane; q < P; q += 32) mx = fmaxf(mx, sm.score[r0 + q]);
            mx = warp_max(mx);
            float ex[4], gq[4], sum = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int q = lane + 32 * i;
                ex[i] = q < P ? expf(sm.score[r0 + q] - mx) : 0.f;
                gq[i] = q < P ? sm.ga[r0 + q] : 0.f;
                sum += ex[i];
            }
            const float inv = 1.0f / warp_sum(sum);
            float dsum = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                ex[i] *= inv;
                dsum = fmaf(ex[i], gq[i], dsum);
            }
            dsum = warp_sum(dsum);
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (lane + 32 * i < P) {
                    sm.attn[r0 + lane + 32 * i] = ex[i];
                    sm.gs[r0 + lane + 32 * i]   = ex[i] * (gq[i] - dsum);
                }
        }
        __syncthreads();
        PROF(5);
        // ---- X line: g_s * [v_hi | v_lo] in b3, [g_s hi, lo, 0...] in the second panel (the old A1 tile)
        const float gs = on ? sm.gs[tid] : 0.f;
        const float at = on ? sm.attn[tid] : 0.f;
        gb2_acc += gs;
        {
            float x[KP];
#pragma unroll
            for (int d = 0; d < KP; ++d) x[d] = gs * v[d];
            store_line_split<KP>(sm.b3, tid, x);
            float one[8] = {gs, gs - __bfloat162float(__float2bfloat16_rn(gs)), 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            one[0] = __bfloat162float(__float2bfloat16_rn(gs));
            const float zero[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (KP == 32) {                              // n = 64..79: chunks 0, 1 of the second panel
                store_chunk(sm.a1, tid, 0, one);
                store_chunk(sm.a1, tid, 1, zero);
            } else {                                     // n = 32..47: chunks 4, 5 of the first panel
                store_chunk(sm.b3, tid, 4, one);
                store_chunk(sm.b3, tid, 5, zero);
            }
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (tid == 0) {
            fence_after();
            PROF(6);
            // g_v part: mask (K-major, K = a) x B2 -> columns [0, N2)
            for (int kk = 0; kk < Ap / 16; ++kk)
                umma_bf16(tmem, umma_desc(smem_u32(sm.a2 + (kk >> 2) * (128 * 128))) + 2 * (kk & 3),
                          umma_desc(smem_u32(sm.b2t + (kk >> 2) * (64 * 128))) + 2 * (kk & 3), umma_idesc(N2), kk > 0);
            // U += mask^T X: both operands MN-major, K = the 128 rows of the tile (16 rows = 2048 B per step)
#pragma unroll
            for (int kk = 0; kk < 8; ++kk)
                umma_bf16(tmem + kUOff, umma_desc_mn(smem_u32(sm.a2 + kk * 2048), 128 * 128),
                          umma_desc_mn(smem_u32(sm.b3 + kk * 2048), 128 * 128),
                          umma_idesc(N3) | kUmmaAMn | kUmmaBMn, (!first_tile || kk > 0) ? 1u : 0u);
            umma_commit(sm.bar);
        }
        first_tile = false;
        mbar_wait(sm.bar, phase);
        phase ^= 1;
        fence_after();
        PROF(7);
        // ---- g_v = a g_out + g_s (mask . B2): staged for the per-field sums
        {
            float gv[KP];
            const float* go = sm.gout[buf] + s * 32;
            if (KP == 32) {
                float t0[32], t1[32];
                tmem_ld32(my_tmem, t0);
                tmem_ld32(my_tmem + 32, t1);
#pragma unroll
                for (int d = 0; d < KP; ++d) gv[d] = fmaf(gs, t0[d] + t1[d], at * (d < D ? go[d] : 0.f));
            } else {
                float t0[32];
                tmem_ld32(my_tmem, t0);
#pragma unroll
                for (int d = 0; d < KP; ++d) gv[d] = fmaf(gs, t0[d] + t0[(KP + d) & 31], at * (d < D ? go[d] : 0.f));
            }
#pragma unroll
            for (int c = 0; c < KP / 4; ++c)
                *reinterpret_cast<float4*>(stage + tid * 32 + 4 * ((c ^ tid) & 7)) =
                    on ? make_float4(gv[4 * c], gv[4 * c + 1], gv[4 * c + 2], gv[4 * c + 3]) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        fence_before();
        __syncthreads();
        PROF(8);
        // g_e[s][f][d] = sum_{g != f} g_v[pair(f,g)][d] * e[s][g][d]
        // one thread per (sample, field, 16-byte chunk); partners in ascending field order (ptab)
        for (int item = tid; item < n_s * F * c4; item += kAfmTcThreads) {
            const int sf = small_div(item, 1.0f / (float)c4), c = item - sf * c4;
            const int ss = small_div(sf, 1.0f / (float)F), f = sf - ss * F;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 3
            for (int k = 0; k < F - 1; ++k) {
                const int pt = sm.pidx[f * 16 + k];          // partner field | pair row << 8
                const int g = pt & 255, r = ss * P + (pt >> 8);
                const float4 x = *reinterpret_cast<const float4*>(stage + r * 32 + 4 * ((c ^ r) & 7));
                const float4 y = *reinterpret_cast<const float4*>(esm + (ss * F + g) * p.estride + 4 * c);
                acc.x = fmaf(x.x, y.x, acc.x); acc.y = fmaf(x.y, y.y, acc.y);
                acc.z = fmaf(x.z, y.z, acc.z); acc.w = fmaf(x.w, y.w, acc.w);
            }
            *reinterpret_cast<float4*>(g_rows + (b0 + ss) * F * D + f * D + 4 * c) = acc;
        }
        __syncthreads();                             // stage (b3), a1, score... are rewritten by the next tile
        PROF(9);
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");

    // ---- this CTA's share of the attention-weight gradients, from U (lane = a)
    float* outp = partials + (int64_t)blockIdx.x * (A * D + 2 * A + 1);
    {
        float u[KP];
        float u0 = 0.f;
#pragma unroll
        for (int d = 0; d < KP; ++d) u[d] = 0.f;
        if (!first_tile) {
            fence_after();
            if (KP == 32) {
                float t0[32], t1[32], t2[32];
                tmem_ld32(my_tmem + kUOff, t0);
                tmem_ld32(my_tmem + kUOff + 32, t1);
                tmem_ld32(my_tmem + kUOff + 64, t2);
#pragma unroll
                for (int d = 0; d < KP; ++d) u[d] = t0[d] + t1[d];
                u0 = t2[0] + t2[1];
            } else {
                float t0[32], t1[32];
                tmem_ld32(my_tmem + kUOff, t0);
                tmem_ld32(my_tmem + kUOff + 32, t1);
#pragma unroll
                for (int d = 0; d < KP; ++d) u[d] = t0[d] + t0[(KP + d) & 31];
                u0 = t1[0] + t1[1];
            }
        }
        if (tid < A) {
            const float w2a = sm.w2[tid];
            float gw2 = sm.bias[tid] * u0;
            float w1row[KP];
#pragma unroll
            for (int c = 0; c < KP / 4; ++c) {           // D is a multiple of 4: 16-byte loads, all in flight together
                const float4 w = 4 * c < D ? __ldg(reinterpret_cast<const float4*>(p.w1 + tid * D) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
                w1row[4 * c] = w.x; w1row[4 * c + 1] = w.y; w1row[4 * c + 2] = w.z; w1row[4 * c + 3] = w.w;
            }
#pragma unroll
            for (int d = 0; d < KP; ++d)
                if (d < D) {
                    outp[tid * D + d] = w2a * u[d];
                    gw2 = fmaf(w1row[d], u[d], gw2);
                }
            outp[A * D + tid]     = w2a * u0;
            outp[A * D + A + tid] = gw2;
        }
    }
    gb2_acc = warp_sum(gb2_acc);                      // fixed shuffle tree, then the four warp sums in order
    if (lane == 0) sm.red[warp] = gb2_acc;
    __syncthreads();
    if (tid == 0) outp[A * D + 2 * A] = (sm.red[0] + sm.red[1]) + (sm.red[2] + sm.red[3]);
    PROF(10);
    PROF_END;
    fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

}  // namespace tc

static int afm_tc_fill(const rk_field_t* fields, int F, const float* w1, const float* b1, const float* w2,
                       const float* b2, int A, int64_t B, const void* tiles, tc::AfmTcParams* p) {
    RK_CHECK_ARG(tiles, "afm: tiles is NULL (rk_afm_tile_bytes() bytes of scratch are required)");
    RK_CHECK_ARG(((uintptr_t)tiles % 128) == 0, "afm: tiles must be 128-byte aligned");
    p->tiles = (const uint8_t*)tiles;
    if (int rc = pack_fields(fields, F, &p->fs)) return rc;
    RK_CHECK_ARG(F >= 2 && F <= 16, "afm: %d fields (supported: 2..16, i.e. <= 120 pairs)", F);
    const int D = fields[0].dim;
    for (int f = 0; f < F; ++f) {
        RK_CHECK_ARG(fields[f].dim == D, "afm: field %d dim %d != %d", f, fields[f].dim, D);
        RK_CHECK_ARG(((uintptr_t)fields[f].weight % 16) == 0, "afm: table %d not 16-byte aligned", f);
    }
    RK_CHECK_ARG(D % 4 == 0 && D >= 4 && D <= 32, "afm: embedding_dim %d not in {4,8,..,32}", D);
    RK_CHECK_ARG(A >= 1 && A <= 128, "afm: attention_factor %d outside [1,128]", A);
    RK_CHECK_ARG(w1 && b1 && w2 && b2, "afm: NULL attention weight");
    p->w1 = w1; p->b1 = b1; p->w2 = w2; p->b2 = b2;
    p->D = D; p->Kp = (D + 15) / 16 * 16; p->A = A; p->Ap = (A + 31) / 32 * 32;
    p->P = F * (F - 1) / 2;
    int S = tc::kAfmTcRows / p->P;
    p->S = S > tc::kAfmTcMaxS ? tc::kAfmTcMaxS : S;
    p->estride = D + 4;                  // float4 reads of different rows land in different bank groups
    p->B = B;
    p->n_tiles = ceil_div(B, p->S);
    return 0;
}

}  // namespace rk

extern "C" {

int rk_afm_tc_fwd(const rk_field_t* fields, int F, const float* w1, const float* b1, const float* w2,
                  const float* b2, int A, int64_t B, float* out, void* tiles, int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    tc::AfmTcParams p;
    if (int rc = afm_tc_fill(fields, F, w1, b1, w2, b2, A, B, tiles, &p)) return rc;
    RK_CHECK_ARG(out, "afm_tc_fwd: out is NULL");
    if (B == 0) return 0;
    const size_t smem = tc::AfmTcFwdSmem::bytes(p);
    RK_CHECK_ARG(smem <= 227 * 1024, "afm_tc_fwd: %zu bytes of shared memory", smem);
    auto kernel = p.Kp == 16 ? tc::afm_fwd_tc_kernel<16> : tc::afm_fwd_tc_kernel<32>;
    RK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // Tiles are strided statically over the CTAs, so the grid must not exceed what is co-resident
    // (a second wave would redo the per-CTA set-up).  cudaOccupancyMaxActiveBlocksPerMultiprocessor
    // reports 1 for kernels that allocate TMEM, so the bound is stated here: 4 x 128 TMEM columns,
    // 4 x 128 threads x 128 registers, 4 x ~44 KB of shared memory per SM.
    constexpr int occ = 4;
    int64_t grid = p.n_tiles;
    const int64_t cap = (int64_t)sm_count() * occ;
    if (grid > cap) grid = cap;
    // both directions' weight tiles, once per forward
    if (p.Kp == 16) tc::afm_weight_tiles_kernel<16><<<2, 256, 0, (cudaStream_t)stream_>>>(w1, w2, A, p.D, (uint8_t*)tiles);
    else            tc::afm_weight_tiles_kernel<32><<<2, 256, 0, (cudaStream_t)stream_>>>(w1, w2, A, p.D, (uint8_t*)tiles);
    RK_LAUNCH_CHECK();
    kernel<<<(int)grid, tc::kAfmTcThreads, smem, (cudaStream_t)stream_>>>(p, out, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}

int rk_afm_tile_bytes(void) { return (int)rk::tc::kAfmTileBytes; }

int rk_afm_tc_bwd_ctas(int64_t B, int F) {
    if (F < 2 || F > 16 || B <= 0) return 1;
    int S = rk::tc::kAfmTcRows / (F * (F - 1) / 2);
    if (S > rk::tc::kAfmTcMaxS) S = rk::tc::kAfmTcMaxS;
    const int64_t tiles = rk::ceil_div(B, S);
    const int64_t cap = 2 * (int64_t)rk::sm_count();   // two CTAs per SM: 2 x 256 TMEM columns, ~107 KB of shared memory each
    return (int)(tiles < cap ? tiles : cap);
}

int rk_afm_tc_bwd(const rk_field_t* fields, int F, const float* w1, const float* b1, const float* w2,
                  const float* b2, int A, int64_t B, const float* g_out, float* g_rows, float* g_w1,
                  float* g_b1, float* g_w2, float* g_b2, float* partials, int n_ctas, const void* tiles,
                  int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    tc::AfmTcParams p;
    if (int rc = afm_tc_fill(fields, F, w1, b1, w2, b2, A, B, tiles, &p)) return rc;
    RK_CHECK_ARG(g_out && g_rows && g_w1 && g_b1 && g_w2 && g_b2 && partials, "afm_tc_bwd: NULL pointer");
    RK_CHECK_ARG(n_ctas == rk_afm_tc_bwd_ctas(B, F), "afm_tc_bwd: n_ctas %d != rk_afm_tc_bwd_ctas", n_ctas);
    RK_CHECK_ARG(g_b1 == g_w1 + (size_t)A * p.D && g_w2 == g_b1 + A && g_b2 == g_w2 + A,
                 "afm_tc_bwd: g_w1|g_b1|g_w2|g_b2 must be one contiguous buffer in that order");
    RK_CHECK_ARG(((uintptr_t)g_out % 16) == 0, "afm_tc_bwd: g_out must be 16-byte aligned");
    if (B == 0) return 0;
    const size_t smem = tc::AfmTcBwdSmem::bytes(p);
    RK_CHECK_ARG(smem <= 227 * 1024, "afm_tc_bwd: %zu bytes of shared memory", smem);
    auto kernel = p.Kp == 16 ? tc::afm_bwd_tc_kernel<16> : tc::afm_bwd_tc_kernel<32>;
    RK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaStream_t s = (cudaStream_t)stream_;
    kernel<<<n_ctas, tc::kAfmTcThreads, smem, s>>>(p, g_out, g_rows, partials, err_flag);
    RK_LAUNCH_CHECK();
    const int count = A * p.D + 2 * A + 1;
    return launch_reduce_partials(partials, n_ctas, count, g_w1, s);
}

}  // extern "C"
