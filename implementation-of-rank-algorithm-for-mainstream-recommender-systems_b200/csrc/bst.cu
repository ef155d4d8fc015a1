// bst.cu — BST behaviour-sequence transformer block (BSTTransformer.forward, BST/bst.py:66-91)
// with the sequence gather (BST/bst.py:224) and the pooling over all T positions (:238-241),
// forward and backward, fp32 SIMT, d_model = 16.
//
// One thread owns one (sample, position) row: its 16-wide activations live in registers, the
// six 16x16 weight matrices sit in shared memory in both orientations and are read with 16-byte
// broadcast loads (one load per four FMAs).  Keys/values of the CTA's samples are exchanged
// through shared memory; scores, the masked softmax (key padding mask t >= len -> -inf) and the
// context are computed per head in registers (d_head = 16/nhead is far too small for tensor
// cores).  The backward recomputes the forward in-kernel, keeps no [B,heads,T,T] tensor, and
// reduces the gradients of the REGISTERED block weights (w_q..w_o, ffn, both LayerNorms, the
// position table) per persistent CTA in registers; a second kernel adds the per-CTA partials in
// fixed order (no atomics).
#include <string.h>
#include "common.cuh"
#include "prof.cuh"
#include "bst.cuh"

namespace rk {

constexpr int kBstThreads = 128;



struct BstSmem {
    float *wt, *w, *vec, *pos;            // [6][256] k-major, [6][256] registered, [10][16], [T][16]
    float *ks, *vs, *qs, *dc, *gs, *as, *xs, *qks, *cs;   // [rows][20] each
    float *mrow, *lrow, *delta;           // [rows][H]
    double* vsum;                         // [8][32] column-sum accumulators (bias / LayerNorm gradients)
    __device__ BstSmem(float* base, int T, int H, bool bwd) {
        float* p = base;
        wt = p;  p += 6 * 256;
        w = p;   p += bwd ? 6 * 256 : 0;
        vec = p; p += 160;
        pos = p; p += T * 16;
        ks = p;  p += kBstRows * kBstLd;
        vs = p;  p += kBstRows * kBstLd;
        gs = p;  p += kBstRows * kBstLd;     // forward: the block output rows (for pooling)
        if (bwd) {
            qs = p;  p += kBstRows * kBstLd;
            dc = p;  p += kBstRows * kBstLd;
            as = p;  p += kBstRows * kBstLd;
            xs = p;  p += kBstRows * kBstLd;
            qks = p; p += kBstRows * kBstLd;
            cs = p;  p += kBstRows * kBstLd;
            mrow = p;  p += kBstRows * H;
            lrow = p;  p += kBstRows * H;
            delta = p; p += kBstRows * H;
            vsum = reinterpret_cast<double*>(p); p += 2 * 8 * 32;
        }
    }
    static size_t bytes(int T, int H, bool bwd) {
        size_t n = 6 * 256 + (bwd ? 6 * 256 : 0) + 160 + (size_t)T * 16 + (size_t)(bwd ? 9 : 3) * kBstRows * kBstLd +
                   (bwd ? (size_t)3 * kBstRows * H + 2 * 8 * 32 : 0);
        return n * sizeof(float);
    }
};

__device__ __forceinline__ void bst_stage_weights(const BstParams& p, const BstSmem& sm, bool bwd) {
    for (int i = threadIdx.x; i < 6 * 256; i += kBstThreads) {
        const int m = i >> 8, e = i & 255, k = e >> 4, n = e & 15;
        sm.wt[i] = __ldg(p.w[m] + n * 16 + k);          // wt[k][n] = W[n][k]
        if (bwd) sm.w[i] = __ldg(p.w[m] + e);
    }
    for (int i = threadIdx.x; i < 160; i += kBstThreads) sm.vec[i] = __ldg(p.vec[i >> 4] + (i & 15));
    for (int i = threadIdx.x; i < p.T * 16; i += kBstThreads) sm.pos[i] = __ldg(p.pos + i);
}

template <int H>
__global__ void __launch_bounds__(kBstThreads)
bst_fwd_kernel(const __grid_constant__ BstParams p, float* __restrict__ y_out, float* __restrict__ pool_out,
               int pool_ld, int32_t* err_flag) {
    extern __shared__ __align__(16) float smem_raw[];
    BstSmem sm(smem_raw, p.T, H, false);
    bst_stage_weights(p, sm, false);
    __syncthreads();
    const int r = threadIdx.x, T = p.T;
    for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const int64_t b0 = tile * p.S;
        const int ns = (int)((p.B - b0) < p.S ? (p.B - b0) : p.S);
        const int rows = ns * T;
        const bool on = r < rows;
        const int s = on ? r / T : 0, t = on ? r - s * T : 0;
        const int64_t b = b0 + s;
        float x[16], qk[16], q[16];
        int L = 0;
        if (on) {
            L = bst_len(p, b);
            bst_load_x(p, b, t, x, err_flag);
            float k[16], v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) qk[i] = x[i] + sm.pos[t * 16 + i];
            set_vec(q, sm.vec + VBQ * 16); set_vec(k, sm.vec + VBK * 16); set_vec(v, sm.vec + VBV * 16);
            matvec16(sm.wt + MQ * 256, qk, q);
            matvec16(sm.wt + MK * 256, qk, k);
            matvec16(sm.wt + MV * 256, x, v);
            store_row(sm.ks + r * kBstLd, k);
            store_row(sm.vs + r * kBstLd, v);
        }
        __syncthreads();
        if (on) {
            float ctx[16], mh[H], lh[H];
            bst_attend<H>(q, sm.ks, sm.vs, s * T, L, ctx, mh, lh);
            const BstDrop drop = bst_drop_masks(p, b * T + t);
            float z[16], zh[16], o1[16], hp[16], f[16], y[16];
            set_vec(z, sm.vec + VBO * 16);
            matvec16(sm.wt + MO * 256, ctx, z);
            bst_drop(drop, 0, z);
#pragma unroll
            for (int i = 0; i < 16; ++i) z[i] += qk[i];
            layer_norm16(z, sm.vec + VG1 * 16, sm.vec + VBE1 * 16, zh, o1);
            set_vec(hp, sm.vec + VB1 * 16);
            matvec16(sm.wt + M1 * 256, o1, hp);
#pragma unroll
            for (int i = 0; i < 16; ++i) hp[i] = hp[i] > 0.f ? hp[i] : 0.01f * hp[i];
            bst_drop(drop, 1, hp);
            set_vec(f, sm.vec + VB2 * 16);
            matvec16(sm.wt + M2 * 256, hp, f);
            bst_drop(drop, 2, f);
#pragma unroll
            for (int i = 0; i < 16; ++i) z[i] = o1[i] + f[i];
            layer_norm16(z, sm.vec + VG2 * 16, sm.vec + VBE2 * 16, zh, y);
            if (y_out) store_row(y_out + (b * T + t) * 16, y);
            store_row(sm.gs + r * kBstLd, y);
        }
        __syncthreads();
        if (pool_out) {
            for (int item = r; item < ns * 16; item += kBstThreads) {
                const int ss = item >> 4, n = item & 15;
                float a = 0.f;
                for (int tt = 0; tt < T; ++tt) a += sm.gs[(ss * T + tt) * kBstLd + n];
                if (p.pool_mean) a /= (float)__ldg(p.seq_len + b0 + ss);
                pool_out[(b0 + ss) * pool_ld + n] = a;
            }
        }
        __syncthreads();
    }
}

// dW[n][k] += sum_rows G[row][n] * A[row][k]: thread owns (n, k), (n, k+1)
__device__ __forceinline__ void bst_outer(const float* __restrict__ gs, const float* __restrict__ as, int rows,
                                          float (&acc)[2]) {
    const int e = threadIdx.x * 2, n = e >> 4, k = e & 15;
    float a0 = acc[0], a1 = acc[1];
    for (int row = 0; row < rows; ++row) {
        const float g = gs[row * kBstLd + n];
        const float2 a = *reinterpret_cast<const float2*>(as + row * kBstLd + k);
        a0 = fmaf(g, a.x, a0);
        a1 = fmaf(g, a.y, a1);
    }
    acc[0] = a0; acc[1] = a1;
}
// column sums of one or two staged arrays: threads 0..15 -> gs, 16..31 -> as (if used)
__device__ __forceinline__ void bst_colsum(const float* __restrict__ gs, const float* __restrict__ as, int rows,
                                           double& acc) {
    const int tid = threadIdx.x;
    if (tid < 16 || (as != nullptr && tid < 32)) {
        const float* src = (tid < 16 ? gs : as) + (tid & 15);
        float a = 0.f;
        for (int row = 0; row < rows; ++row) a += src[row * kBstLd];
        acc += (double)a;     // across tiles in double: these sums run over every row of the batch
    }
}

// partial layout (floats): [pos T*16][wq 256][bq 16][wk][bk][wv][bv][wo][bo][g1][be1][w1][b1][w2][b2][g2][be2]
template <int H>
__global__ void __launch_bounds__(kBstThreads)
bst_bwd_kernel(const __grid_constant__ BstParams p, const float* __restrict__ g_y, const float* __restrict__ g_pool,
               int g_pool_ld, float* __restrict__ g_x, float* __restrict__ partials, int32_t* err_flag) {
    constexpr int DH = 16 / H;
    extern __shared__ __align__(16) float smem_raw[];
    BstSmem sm(smem_raw, p.T, H, true);
    PROF_DECL
    bst_stage_weights(p, sm, true);
    __syncthreads();
    const int r = threadIdx.x, T = p.T;
    const float scale = 1.0f / sqrtf((float)DH);
    float macc[6][2];
#pragma unroll
    for (int m = 0; m < 6; ++m) { macc[m][0] = 0.f; macc[m][1] = 0.f; }
    if (r < 32) {
#pragma unroll
        for (int i = 0; i < 8; ++i) sm.vsum[i * 32 + r] = 0.0;
    }
    float pacc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) pacc[i] = 0.f;
    PROF(0);

    for (int64_t tile = blockIdx.x; tile < p.n_tiles; tile += gridDim.x) {
        const int64_t b0 = tile * p.S;
        const int ns = (int)((p.B - b0) < p.S ? (p.B - b0) : p.S);
        const int rows = ns * T;
        const bool on = r < rows;
        const int s = on ? r / T : 0, t = on ? r - s * T : 0;
        const int64_t b = b0 + s;
        const int row0 = s * T;
        int L = 0;
        float zh1[16], zh2[16], act[16], rstd1 = 0.f, rstd2 = 0.f;
        unsigned hmask = 0;
        BstDrop drop;
        drop.active = false; drop.scale = 1.f; drop.k[0] = drop.k[1] = drop.k[2] = 0xffffu;
        float zero16[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) zero16[i] = 0.f;
        // ---- A. recompute the forward, parking what other rows / later phases need in smem
        if (on) {
            L = bst_len(p, b);
            float x[16], qk[16], q[16], k[16], v[16];
            bst_load_x(p, b, t, x, err_flag);
#pragma unroll
            for (int i = 0; i < 16; ++i) qk[i] = x[i] + sm.pos[t * 16 + i];
            set_vec(q, sm.vec + VBQ * 16); set_vec(k, sm.vec + VBK * 16); set_vec(v, sm.vec + VBV * 16);
            matvec16(sm.wt + MQ * 256, qk, q);
            matvec16(sm.wt + MK * 256, qk, k);
            matvec16(sm.wt + MV * 256, x, v);
            store_row(sm.xs + r * kBstLd, x);
            store_row(sm.qks + r * kBstLd, qk);
            store_row(sm.qs + r * kBstLd, q);
            store_row(sm.ks + r * kBstLd, k);
            store_row(sm.vs + r * kBstLd, v);
        } else {
            store_row(sm.xs + r * kBstLd, zero16);
            store_row(sm.qks + r * kBstLd, zero16);
        }
        __syncthreads();
        PROF(1); PROF_COUNT(12);
        if (on) {
            float q[16], qk[16], ctx[16], mh[H], lh[H];
            load_row(sm.qs + r * kBstLd, q);
            load_row(sm.qks + r * kBstLd, qk);
            bst_attend<H>(q, sm.ks, sm.vs, row0, L, ctx, mh, lh);
#pragma unroll
            for (int h = 0; h < H; ++h) { sm.mrow[r * H + h] = mh[h]; sm.lrow[r * H + h] = 1.0f / lh[h]; }   // lrow holds 1 / sum
            store_row(sm.cs + r * kBstLd, ctx);
            drop = bst_drop_masks(p, b * T + t);
            float z[16], o1[16], hp[16], f[16], y[16];
            set_vec(z, sm.vec + VBO * 16);
            matvec16(sm.wt + MO * 256, ctx, z);
            bst_drop(drop, 0, z);
#pragma unroll
            for (int i = 0; i < 16; ++i) z[i] += qk[i];
            rstd1 = layer_norm16(z, sm.vec + VG1 * 16, sm.vec + VBE1 * 16, zh1, o1);
            set_vec(hp, sm.vec + VB1 * 16);
            matvec16(sm.wt + M1 * 256, o1, hp);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                if (hp[i] > 0.f) hmask |= 1u << i;
                act[i] = hp[i] > 0.f ? hp[i] : 0.01f * hp[i];
            }
            bst_drop(drop, 1, act);
            set_vec(f, sm.vec + VB2 * 16);
            matvec16(sm.wt + M2 * 256, act, f);
            bst_drop(drop, 2, f);
#pragma unroll
            for (int i = 0; i < 16; ++i) z[i] = o1[i] + f[i];
            rstd2 = layer_norm16(z, sm.vec + VG2 * 16, sm.vec + VBE2 * 16, zh2, y);
        } else {
            store_row(sm.cs + r * kBstLd, zero16);
        }
        // ---- B. upstream gradient of this row, LayerNorm 2 backward
        PROF(2);
        float dy[16], dz[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) dy[i] = 0.f;
        if (on) {
            if (g_y) load_row(g_y + (b * T + t) * 16, dy);
            if (g_pool) {
                const float inv = p.pool_mean ? 1.0f / (float)__ldg(p.seq_len + b) : 1.0f;
#pragma unroll
                for (int i = 0; i < 16; ++i) dy[i] = fmaf(g_pool[b * g_pool_ld + i], inv, dy[i]);
            }
        }
        {
            float t0[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) t0[i] = on ? dy[i] * zh2[i] : 0.f;
            store_row(sm.gs + r * kBstLd, t0);
            store_row(sm.as + r * kBstLd, dy);
        }
        __syncthreads();
        bst_colsum(sm.gs, sm.as, rows, sm.vsum[0 * 32 + (r & 31)]);                 // d ln2_g | d ln2_b
        __syncthreads();
        if (on) layer_norm16_bwd(dy, sm.vec + VG2 * 16, zh2, rstd2, dz);
        else {
#pragma unroll
            for (int i = 0; i < 16; ++i) { dz[i] = 0.f; act[i] = 0.f; }
        }
        // ---- C. FFN backward  (df = gradient of the FFN output before its dropout)
        PROF(3);
        float df[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) df[i] = dz[i];
        bst_drop(drop, 2, df);
        store_row(sm.gs + r * kBstLd, df);
        store_row(sm.as + r * kBstLd, act);
        __syncthreads();
        bst_outer(sm.gs, sm.as, rows, macc[M2]);
        bst_colsum(sm.gs, nullptr, rows, sm.vsum[1 * 32 + (r & 31)]);               // d b2
        __syncthreads();
        float dh[16], o1[16], do1[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) { dh[i] = 0.f; o1[i] = 0.f; }
        if (on) {
            matvec16(sm.w + M2 * 256, df, dh);                       // W2^T df
            bst_drop(drop, 1, dh);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                dh[i] *= ((hmask >> i) & 1u) ? 1.0f : 0.01f;
                o1[i] = fmaf(zh1[i], sm.vec[VG1 * 16 + i], sm.vec[VBE1 * 16 + i]);
            }
        }
        store_row(sm.gs + r * kBstLd, dh);
        store_row(sm.as + r * kBstLd, o1);
        __syncthreads();
        bst_outer(sm.gs, sm.as, rows, macc[M1]);
        bst_colsum(sm.gs, nullptr, rows, sm.vsum[2 * 32 + (r & 31)]);               // d b1
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 16; ++i) do1[i] = dz[i];
        if (on) matvec16(sm.w + M1 * 256, dh, do1);                  // + W1^T dh
        // ---- D. LayerNorm 1 backward, output projection backward
        PROF(4);
        {
            float t0[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) t0[i] = on ? do1[i] * zh1[i] : 0.f;
            store_row(sm.gs + r * kBstLd, t0);
            store_row(sm.as + r * kBstLd, do1);
        }
        __syncthreads();
        bst_colsum(sm.gs, sm.as, rows, sm.vsum[3 * 32 + (r & 31)]);                 // d ln1_g | d ln1_b
        __syncthreads();
        float dz1[16], dctx[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) { dz1[i] = 0.f; dctx[i] = 0.f; }
        if (on) layer_norm16_bwd(do1, sm.vec + VG1 * 16, zh1, rstd1, dz1);
        float dwo[16];                                               // gradient of w_o(ctx) before its dropout
#pragma unroll
        for (int i = 0; i < 16; ++i) dwo[i] = dz1[i];
        bst_drop(drop, 0, dwo);
        store_row(sm.gs + r * kBstLd, dwo);
        __syncthreads();
        bst_outer(sm.gs, sm.cs, rows, macc[MO]);                 // d w_o = dwo (x) ctx
        bst_colsum(sm.gs, nullptr, rows, sm.vsum[4 * 32 + (r & 31)]);               // d b_o
        if (on) {
            matvec16(sm.w + MO * 256, dwo, dctx);                    // W_o^T dwo
            float ctx[16];
            load_row(sm.cs + r * kBstLd, ctx);
#pragma unroll
            for (int h = 0; h < H; ++h) {
                float d = 0.f;
#pragma unroll
                for (int j = 0; j < DH; ++j) d = fmaf(dctx[h * DH + j], ctx[h * DH + j], d);
                sm.delta[r * H + h] = d;
            }
        }
        store_row(sm.dc + r * kBstLd, dctx);
        __syncthreads();
        // ---- E. attention backward: as a query (dq) and as a key (dk, dv)
        PROF(5);
        float dq[16], dk[16], dv[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) { dq[i] = 0.f; dk[i] = 0.f; dv[i] = 0.f; }
        if (on) {
            float q[16], kme[16], vme[16];
            load_row(sm.qs + r * kBstLd, q);
            load_row(sm.ks + r * kBstLd, kme);
            load_row(sm.vs + r * kBstLd, vme);
            // as a query: one pass over the L live keys, the H heads side by side (independent exp chains)
            float mq[H], ilq[H], dlq[H];
#pragma unroll
            for (int h = 0; h < H; ++h) { mq[h] = sm.mrow[r * H + h]; ilq[h] = sm.lrow[r * H + h]; dlq[h] = sm.delta[r * H + h]; }
            for (int u = 0; u < L; ++u) {
                float kr[16], vr[16];
                load_row(sm.ks + (row0 + u) * kBstLd, kr);
                load_row(sm.vs + (row0 + u) * kBstLd, vr);
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    float sc = 0.f, dA = 0.f;
#pragma unroll
                    for (int j = 0; j < DH; ++j) {
                        sc = fmaf(q[h * DH + j], kr[h * DH + j], sc);
                        dA = fmaf(dctx[h * DH + j], vr[h * DH + j], dA);
                    }
                    const float a  = expf(sc * scale - mq[h]) * ilq[h];
                    const float dS = a * (dA - dlq[h]) * scale;
#pragma unroll
                    for (int j = 0; j < DH; ++j) dq[h * DH + j] = fmaf(dS, kr[h * DH + j], dq[h * DH + j]);
                }
            }
            if (t < L) {   // this row is a live key: every position of the sample queries it
                for (int tq = 0; tq < T; ++tq) {
                    const int rq = row0 + tq;
                    float qr[16], dr[16];
                    load_row(sm.qs + rq * kBstLd, qr);
                    load_row(sm.dc + rq * kBstLd, dr);
#pragma unroll
                    for (int h = 0; h < H; ++h) {
                        float sc = 0.f, dA = 0.f;
#pragma unroll
                        for (int j = 0; j < DH; ++j) {
                            sc = fmaf(qr[h * DH + j], kme[h * DH + j], sc);
                            dA = fmaf(dr[h * DH + j], vme[h * DH + j], dA);
                        }
                        const float a  = expf(sc * scale - sm.mrow[rq * H + h]) * sm.lrow[rq * H + h];
                        const float dS = a * (dA - sm.delta[rq * H + h]) * scale;
#pragma unroll
                        for (int j = 0; j < DH; ++j) {
                            dv[h * DH + j] = fmaf(a, dr[h * DH + j], dv[h * DH + j]);
                            dk[h * DH + j] = fmaf(dS, qr[h * DH + j], dk[h * DH + j]);
                        }
                    }
                }
            }
        }
        __syncthreads();
        // ---- F. projection backward, input gradient, position-table gradient
        PROF(6);
        store_row(sm.gs + r * kBstLd, dq);
        __syncthreads();
        bst_outer(sm.gs, sm.qks, rows, macc[MQ]);
        bst_colsum(sm.gs, nullptr, rows, sm.vsum[5 * 32 + (r & 31)]);               // d b_q
        __syncthreads();
        store_row(sm.gs + r * kBstLd, dk);
        __syncthreads();
        bst_outer(sm.gs, sm.qks, rows, macc[MK]);
        bst_colsum(sm.gs, nullptr, rows, sm.vsum[6 * 32 + (r & 31)]);               // d b_k
        __syncthreads();
        store_row(sm.gs + r * kBstLd, dv);
        __syncthreads();
        bst_outer(sm.gs, sm.xs, rows, macc[MV]);
        bst_colsum(sm.gs, nullptr, rows, sm.vsum[7 * 32 + (r & 31)]);               // d b_v
        __syncthreads();
        float dqk[16];
        PROF(7);
#pragma unroll
        for (int i = 0; i < 16; ++i) dqk[i] = dz1[i];                // residual path of LayerNorm 1
        if (on) {
            matvec16(sm.w + MQ * 256, dq, dqk);
            matvec16(sm.w + MK * 256, dk, dqk);
            float dx[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) dx[i] = dqk[i];
            matvec16(sm.w + MV * 256, dv, dx);
            store_row(g_x + (b * T + t) * 16, dx);
        }
        store_row(sm.gs + r * kBstLd, dqk);
        __syncthreads();
        PROF(8);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int e = r + i * kBstThreads;
            if (e < T * 16) {
                const int tt = e >> 4, n = e & 15;
                float a = pacc[i];
                for (int ss = 0; ss < ns; ++ss) a += sm.gs[(ss * T + tt) * kBstLd + n];
                pacc[i] = a;
            }
        }
        __syncthreads();
        PROF(9);
    }

    // ---- per-CTA partials of the registered parameters
    PROF(10);
    PROF_END;
    float* out = partials + (int64_t)blockIdx.x * (T * 16 + 6 * 256 + 160);
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const int e = r + i * kBstThreads;
        if (e < T * 16) out[e] = pacc[i];
    }
    float* o = out + T * 16;
    const int e2 = r * 2;
    // order: wq bq wk bk wv bv wo bo g1 be1 w1 b1 w2 b2 g2 be2
    const int mat_off[6] = {0, 272, 544, 816, 1120, 1392};   // wq wk wv wo w1 w2
    o[mat_off[MQ] + e2] = macc[MQ][0]; o[mat_off[MQ] + e2 + 1] = macc[MQ][1];
    o[mat_off[MK] + e2] = macc[MK][0]; o[mat_off[MK] + e2 + 1] = macc[MK][1];
    o[mat_off[MV] + e2] = macc[MV][0]; o[mat_off[MV] + e2 + 1] = macc[MV][1];
    o[mat_off[MO] + e2] = macc[MO][0]; o[mat_off[MO] + e2 + 1] = macc[MO][1];
    o[mat_off[M1] + e2] = macc[M1][0]; o[mat_off[M1] + e2 + 1] = macc[M1][1];
    o[mat_off[M2] + e2] = macc[M2][0]; o[mat_off[M2] + e2 + 1] = macc[M2][1];
    if (r < 16) {
        o[256 + r]  = (float)sm.vsum[5 * 32 + r];    // bq
        o[528 + r]  = (float)sm.vsum[6 * 32 + r];    // bk
        o[800 + r]  = (float)sm.vsum[7 * 32 + r];    // bv
        o[1072 + r] = (float)sm.vsum[4 * 32 + r];    // bo
        o[1088 + r] = (float)sm.vsum[3 * 32 + r];    // ln1_g
        o[1376 + r] = (float)sm.vsum[2 * 32 + r];    // b1
        o[1648 + r] = (float)sm.vsum[1 * 32 + r];    // b2
        o[1664 + r] = (float)sm.vsum[0 * 32 + r];    // ln2_g
    } else if (r < 32) {
        o[1104 + r - 16] = (float)sm.vsum[3 * 32 + r];   // ln1_b
        o[1680 + r - 16] = (float)sm.vsum[0 * 32 + r];   // ln2_b
    }
}

// ---- sequences longer than one 128-row tile (fp32) ------------------------------------------------
// A CTA owns one sample at a time, samples strided statically over the grid (sample = blockIdx.x +
// k * gridDim.x), so the backward's per-CTA partials are reproducible.  The T query rows are cut into
// chunks of 128 (thread = row in the chunk) and the L = min(len, T) live keys into key chunks of 128,
// whose k / v rows are recomputed (gather + matvec16) per (query chunk, key chunk) pair.  The softmax
// runs online over the key chunks: the chunk's max, one rescale of the running sum and context, then
// bst_attend's second pass.  With one key chunk this is bst_attend exactly.  The position table is read
// row by row from global memory: T x 16 floats need not fit in shared memory.
struct BstLongSmem {
    float *wt, *w, *vec;                  // [6][256] k-major, [6][256] registered, [10][16]
    float *ks, *vs, *gs;                  // key chunk k / v rows, staging      [128][20] each
    float *qs, *qks, *dc, *cs, *as;       // backward: query chunk q / qk / dctx / ctx, staging
    float *mrow, *lrow, *delta;           // [128][H]
    double* vsum;                         // [8][32]
    __device__ BstLongSmem(float* base, int H, bool bwd) {
        float* p = base;
        wt = p;  p += 6 * 256;
        w = p;   p += bwd ? 6 * 256 : 0;
        vec = p; p += 160;
        ks = p;  p += kBstRows * kBstLd;
        vs = p;  p += kBstRows * kBstLd;
        gs = p;  p += kBstRows * kBstLd;
        if (bwd) {
            qs = p;  p += kBstRows * kBstLd;
            qks = p; p += kBstRows * kBstLd;
            dc = p;  p += kBstRows * kBstLd;
            cs = p;  p += kBstRows * kBstLd;
            as = p;  p += kBstRows * kBstLd;
            mrow = p;  p += kBstRows * H;
            lrow = p;  p += kBstRows * H;
            delta = p; p += kBstRows * H;
            vsum = reinterpret_cast<double*>(p); p += 2 * 8 * 32;
        }
    }
    static size_t bytes(int H, bool bwd) {
        size_t n = 6 * 256 + (bwd ? 6 * 256 : 0) + 160 + (size_t)(bwd ? 8 : 3) * kBstRows * kBstLd +
                   (bwd ? (size_t)3 * kBstRows * H + 2 * 8 * 32 : 0);
        return n * sizeof(float);
    }
};

__device__ __forceinline__ void bst_stage_weights_long(const BstParams& p, const BstLongSmem& sm, bool bwd) {
    for (int i = threadIdx.x; i < 6 * 256; i += kBstThreads) {
        const int m = i >> 8, e = i & 255, k = e >> 4, n = e & 15;
        sm.wt[i] = __ldg(p.w[m] + n * 16 + k);
        if (bwd) sm.w[i] = __ldg(p.w[m] + e);
    }
    for (int i = threadIdx.x; i < 160; i += kBstThreads) sm.vec[i] = __ldg(p.vec[i >> 4] + (i & 15));
}

// x and qk = x + pos[t] of position t of sample b
__device__ __forceinline__ void bst_long_input(const BstParams& p, int64_t b, int t, float (&x)[16], float (&qk)[16],
                                               int32_t* err_flag) {
    bst_load_x(p, b, t, x, err_flag);
    const float* pr = p.pos + (int64_t)t * 16;
#pragma unroll
    for (int i = 0; i < 16; ++i) qk[i] = x[i] + __ldg(pr + i);
}

// k / v of key position u into this thread's row of ks / vs; the backward also parks qk and x (kqk, kx)
__device__ __forceinline__ void bst_long_key_row(const BstParams& p, const BstLongSmem& sm, int64_t b, int u,
                                                 float* kqk, float* kx, int32_t* err_flag) {
    const int r = threadIdx.x;
    float x[16], qk[16], k[16], v[16];
    bst_long_input(p, b, u, x, qk, err_flag);
    set_vec(k, sm.vec + VBK * 16); set_vec(v, sm.vec + VBV * 16);
    matvec16(sm.wt + MK * 256, qk, k);
    matvec16(sm.wt + MV * 256, x, v);
    store_row(sm.ks + r * kBstLd, k);
    store_row(sm.vs + r * kBstLd, v);
    if (kqk) { store_row(kqk + r * kBstLd, qk); store_row(kx + r * kBstLd, x); }
}

// One key chunk of n rows into the running max m, sum l and (unnormalised) context of one query row.
template <int H>
__device__ __forceinline__ void bst_attend_chunk(const float (&q)[16], const float* __restrict__ ks,
                                                 const float* __restrict__ vs, int n, float (&ctx)[16],
                                                 float (&m)[H], float (&l)[H]) {
    constexpr int DH = 16 / H;
    const float scale = 1.0f / sqrtf((float)DH);
    float mc[H];
#pragma unroll
    for (int h = 0; h < H; ++h) mc[h] = m[h];
    for (int u = 0; u < n; ++u) {
        float kr[16];
        load_row(ks + u * kBstLd, kr);
#pragma unroll
        for (int h = 0; h < H; ++h) {
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < DH; ++j) s = fmaf(q[h * DH + j], kr[h * DH + j], s);
            mc[h] = fmaxf(mc[h], s * scale);
        }
    }
    // the chunk's sum and context start from 0 and are added to the rescaled running ones (blocked summation:
    // a long sequence is not one float chain of L terms); with one chunk, l = lc and ctx = cc exactly
    float lc[H], cc[16];
#pragma unroll
    for (int h = 0; h < H; ++h) lc[h] = 0.f;
#pragma unroll
    for (int i = 0; i < 16; ++i) cc[i] = 0.f;
    for (int u = 0; u < n; ++u) {
        float kr[16], vr[16];
        load_row(ks + u * kBstLd, kr);
        load_row(vs + u * kBstLd, vr);
#pragma unroll
        for (int h = 0; h < H; ++h) {
            float s = 0.f;
#pragma unroll
            for (int j = 0; j < DH; ++j) s = fmaf(q[h * DH + j], kr[h * DH + j], s);
            const float pr = expf(s * scale - mc[h]);
            lc[h] += pr;
#pragma unroll
            for (int j = 0; j < DH; ++j) cc[h * DH + j] = fmaf(pr, vr[h * DH + j], cc[h * DH + j]);
        }
    }
#pragma unroll
    for (int h = 0; h < H; ++h) {
        const float alpha = expf(m[h] - mc[h]);      // 0 on the first chunk (m = -inf)
        l[h] = fmaf(l[h], alpha, lc[h]);
#pragma unroll
        for (int j = 0; j < DH; ++j) ctx[h * DH + j] = fmaf(ctx[h * DH + j], alpha, cc[h * DH + j]);
        m[h] = mc[h];
    }
}

// bst_colsum added row by row straight into the double accumulator: the sums run over every row of the batch
// and cancel heavily, and a chunk can hold a single row
__device__ __forceinline__ void bst_colsum_d(const float* __restrict__ gs, const float* __restrict__ as, int rows,
                                             double& acc) {
    const int tid = threadIdx.x;
    if (tid < 16 || (as != nullptr && tid < 32)) {
        const float* src = (tid < 16 ? gs : as) + (tid & 15);
        double a = acc;
        for (int row = 0; row < rows; ++row) a += (double)src[row * kBstLd];
        acc = a;
    }
}

template <int H>
__device__ __forceinline__ void bst_attend_init(float (&ctx)[16], float (&m)[H], float (&l)[H]) {
#pragma unroll
    for (int h = 0; h < H; ++h) { m[h] = -INFINITY; l[h] = 0.f; }
#pragma unroll
    for (int i = 0; i < 16; ++i) ctx[i] = 0.f;
}
// L == 0: every key masked -> 0/0 = NaN, exactly as softmax over all -inf in the reference
template <int H>
__device__ __forceinline__ void bst_attend_finish(float (&ctx)[16], const float (&l)[H]) {
    constexpr int DH = 16 / H;
#pragma unroll
    for (int h = 0; h < H; ++h)
#pragma unroll
        for (int j = 0; j < DH; ++j) ctx[h * DH + j] = ctx[h * DH + j] / l[h];
}

template <int H>
__global__ void __launch_bounds__(kBstThreads)
bst_fwd_long_kernel(const __grid_constant__ BstParams p, float* __restrict__ y_out, float* __restrict__ pool_out,
                    int pool_ld, int32_t* err_flag) {
    extern __shared__ __align__(16) float smem_raw[];
    BstLongSmem sm(smem_raw, H, false);
    bst_stage_weights_long(p, sm, false);
    __syncthreads();
    const int r = threadIdx.x, T = p.T;
    for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x) {
        const int L = bst_len(p, b);
        int loaded = -1;                  // key chunk held in ks / vs: with one key chunk it is built once
        double pool = 0.0;                // threads 0..15: column r of the pooled row, summed t = 0, 1, .. in double
        for (int t0 = 0; t0 < T; t0 += kBstRows) {
            const int t = t0 + r, rows = min(kBstRows, T - t0);
            const bool on = t < T;
            float x[16], qk[16], q[16];
            if (on) {
                bst_long_input(p, b, t, x, qk, err_flag);
                set_vec(q, sm.vec + VBQ * 16);
                matvec16(sm.wt + MQ * 256, qk, q);
            }
            float ctx[16], mh[H], lh[H];
            bst_attend_init<H>(ctx, mh, lh);
            for (int u0 = 0; u0 < L; u0 += kBstRows) {
                const int n = min(kBstRows, L - u0);
                if (u0 / kBstRows != loaded) {
                    __syncthreads();
                    if (r < n) bst_long_key_row(p, sm, b, u0 + r, nullptr, nullptr, err_flag);
                    __syncthreads();
                    loaded = u0 / kBstRows;
                }
                if (on) bst_attend_chunk<H>(q, sm.ks, sm.vs, n, ctx, mh, lh);
            }
            if (on) {
                bst_attend_finish<H>(ctx, lh);
                const BstDrop drop = bst_drop_masks(p, b * T + t);
                float z[16], zh[16], o1[16], hp[16], f[16], y[16];
                set_vec(z, sm.vec + VBO * 16);
                matvec16(sm.wt + MO * 256, ctx, z);
                bst_drop(drop, 0, z);
#pragma unroll
                for (int i = 0; i < 16; ++i) z[i] += qk[i];
                layer_norm16(z, sm.vec + VG1 * 16, sm.vec + VBE1 * 16, zh, o1);
                set_vec(hp, sm.vec + VB1 * 16);
                matvec16(sm.wt + M1 * 256, o1, hp);
#pragma unroll
                for (int i = 0; i < 16; ++i) hp[i] = hp[i] > 0.f ? hp[i] : 0.01f * hp[i];
                bst_drop(drop, 1, hp);
                set_vec(f, sm.vec + VB2 * 16);
                matvec16(sm.wt + M2 * 256, hp, f);
                bst_drop(drop, 2, f);
#pragma unroll
                for (int i = 0; i < 16; ++i) z[i] = o1[i] + f[i];
                layer_norm16(z, sm.vec + VG2 * 16, sm.vec + VBE2 * 16, zh, y);
                if (y_out) store_row(y_out + (b * T + t) * 16, y);
                store_row(sm.gs + r * kBstLd, y);
            }
            __syncthreads();
            if (pool_out && r < 16)
                for (int row = 0; row < rows; ++row) pool += (double)sm.gs[row * kBstLd + r];
            __syncthreads();
        }
        if (pool_out && r < 16) {
            float a = (float)pool;
            if (p.pool_mean) a /= (float)__ldg(p.seq_len + b);
            pool_out[b * pool_ld + r] = a;
        }
    }
}

// The backward works through the query chunks in order.  Per chunk: the chunk's forward (m and 1/l over
// every key chunk), phases B-D of bst_bwd_kernel down to dctx and delta, then the key chunks again:
// query-row threads accumulate dq, key-row threads this query chunk's dk / dv of their rows.  Everything
// downstream of dk / dv is linear, so each contribution is added where it lands, in this fixed loop
// order: W_k^T dk + W_v^T dv into the sample's g_x row (the first contribution writes), W_k^T dk into the
// CTA's own position-table rows of `partials`, dk (x) qk and dv (x) x into macc, dk and dv into vsum.
// Position u is owned as a query and as a key by thread u mod 128, so every g_x row and position-table
// row is read and written by one thread.
template <int H>
__global__ void __launch_bounds__(kBstThreads)
bst_bwd_long_kernel(const __grid_constant__ BstParams p, const float* __restrict__ g_y,
                    const float* __restrict__ g_pool, int g_pool_ld, float* __restrict__ g_x,
                    float* __restrict__ partials, int32_t* err_flag) {
    constexpr int DH = 16 / H;
    extern __shared__ __align__(16) float smem_raw[];
    BstLongSmem sm(smem_raw, H, true);
    bst_stage_weights_long(p, sm, true);
    const int r = threadIdx.x, T = p.T;
    const float scale = 1.0f / sqrtf((float)DH);
    float* kqk = sm.cs;       // the key chunk's qk and x rows: ctx and the staging array are free in phase E
    float* kx = sm.as;
    float macc[6][2];
#pragma unroll
    for (int m = 0; m < 6; ++m) { macc[m][0] = 0.f; macc[m][1] = 0.f; }
    if (r < 32) {
#pragma unroll
        for (int i = 0; i < 8; ++i) sm.vsum[i * 32 + r] = 0.0;
    }
    float* out = partials + (int64_t)blockIdx.x * (T * 16 + 6 * 256 + 160);
    for (int t = r; t < T; t += kBstRows)          // position-table rows of this CTA, accumulated in place
        for (int i = 0; i < 16; ++i) out[t * 16 + i] = 0.f;
    float zero16[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) zero16[i] = 0.f;
    __syncthreads();

    for (int64_t b = blockIdx.x; b < p.B; b += gridDim.x) {
        const int L = bst_len(p, b);
        for (int t0 = 0; t0 < T; t0 += kBstRows) {
            const int t = t0 + r, rows = min(kBstRows, T - t0);
            const bool on = t < T;
            // ---- A. the chunk's forward: q / qk parked for the key rows, m and 1/l over every key chunk
            float q[16], qk[16], ctx[16], mh[H], lh[H];
            if (on) {
                float x[16];
                bst_long_input(p, b, t, x, qk, err_flag);
                set_vec(q, sm.vec + VBQ * 16);
                matvec16(sm.wt + MQ * 256, qk, q);
                store_row(sm.qs + r * kBstLd, q);
                store_row(sm.qks + r * kBstLd, qk);
            }
            bst_attend_init<H>(ctx, mh, lh);
            for (int u0 = 0; u0 < L; u0 += kBstRows) {
                const int n = min(kBstRows, L - u0);
                __syncthreads();
                if (r < n) bst_long_key_row(p, sm, b, u0 + r, nullptr, nullptr, err_flag);
                __syncthreads();
                if (on) bst_attend_chunk<H>(q, sm.ks, sm.vs, n, ctx, mh, lh);
            }
            float zh1[16], zh2[16], act[16], rstd1 = 0.f, rstd2 = 0.f;
            unsigned hmask = 0;
            BstDrop drop;
            drop.active = false; drop.scale = 1.f; drop.k[0] = drop.k[1] = drop.k[2] = 0xffffu;
            if (on) {
                bst_attend_finish<H>(ctx, lh);
#pragma unroll
                for (int h = 0; h < H; ++h) { sm.mrow[r * H + h] = mh[h]; sm.lrow[r * H + h] = 1.0f / lh[h]; }
                store_row(sm.cs + r * kBstLd, ctx);
                drop = bst_drop_masks(p, b * T + t);
                float z[16], o1[16], hp[16], f[16], y[16];
                set_vec(z, sm.vec + VBO * 16);
                matvec16(sm.wt + MO * 256, ctx, z);
                bst_drop(drop, 0, z);
#pragma unroll
                for (int i = 0; i < 16; ++i) z[i] += qk[i];
                rstd1 = layer_norm16(z, sm.vec + VG1 * 16, sm.vec + VBE1 * 16, zh1, o1);
                set_vec(hp, sm.vec + VB1 * 16);
                matvec16(sm.wt + M1 * 256, o1, hp);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    if (hp[i] > 0.f) hmask |= 1u << i;
                    act[i] = hp[i] > 0.f ? hp[i] : 0.01f * hp[i];
                }
                bst_drop(drop, 1, act);
                set_vec(f, sm.vec + VB2 * 16);
                matvec16(sm.wt + M2 * 256, act, f);
                bst_drop(drop, 2, f);
#pragma unroll
                for (int i = 0; i < 16; ++i) z[i] = o1[i] + f[i];
                rstd2 = layer_norm16(z, sm.vec + VG2 * 16, sm.vec + VBE2 * 16, zh2, y);
            }
            // ---- B. upstream gradient of this row, LayerNorm 2 backward
            float dy[16], dz[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) dy[i] = 0.f;
            if (on) {
                if (g_y) load_row(g_y + (b * T + t) * 16, dy);
                if (g_pool) {
                    const float inv = p.pool_mean ? 1.0f / (float)__ldg(p.seq_len + b) : 1.0f;
#pragma unroll
                    for (int i = 0; i < 16; ++i) dy[i] = fmaf(g_pool[b * g_pool_ld + i], inv, dy[i]);
                }
            }
            {
                float t0v[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) t0v[i] = on ? dy[i] * zh2[i] : 0.f;
                store_row(sm.gs + r * kBstLd, t0v);
                store_row(sm.as + r * kBstLd, dy);
            }
            __syncthreads();
            bst_colsum_d(sm.gs, sm.as, rows, sm.vsum[0 * 32 + (r & 31)]);                 // d ln2_g | d ln2_b
            __syncthreads();
            if (on) layer_norm16_bwd(dy, sm.vec + VG2 * 16, zh2, rstd2, dz);
            else {
#pragma unroll
                for (int i = 0; i < 16; ++i) { dz[i] = 0.f; act[i] = 0.f; }
            }
            // ---- C. FFN backward
            float df[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) df[i] = dz[i];
            bst_drop(drop, 2, df);
            store_row(sm.gs + r * kBstLd, df);
            store_row(sm.as + r * kBstLd, act);
            __syncthreads();
            bst_outer(sm.gs, sm.as, rows, macc[M2]);
            bst_colsum_d(sm.gs, nullptr, rows, sm.vsum[1 * 32 + (r & 31)]);               // d b2
            __syncthreads();
            float dh[16], o1[16], do1[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) { dh[i] = 0.f; o1[i] = 0.f; }
            if (on) {
                matvec16(sm.w + M2 * 256, df, dh);
                bst_drop(drop, 1, dh);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    dh[i] *= ((hmask >> i) & 1u) ? 1.0f : 0.01f;
                    o1[i] = fmaf(zh1[i], sm.vec[VG1 * 16 + i], sm.vec[VBE1 * 16 + i]);
                }
            }
            store_row(sm.gs + r * kBstLd, dh);
            store_row(sm.as + r * kBstLd, o1);
            __syncthreads();
            bst_outer(sm.gs, sm.as, rows, macc[M1]);
            bst_colsum_d(sm.gs, nullptr, rows, sm.vsum[2 * 32 + (r & 31)]);               // d b1
            __syncthreads();
#pragma unroll
            for (int i = 0; i < 16; ++i) do1[i] = dz[i];
            if (on) matvec16(sm.w + M1 * 256, dh, do1);
            // ---- D. LayerNorm 1 backward, output projection backward
            {
                float t0v[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) t0v[i] = on ? do1[i] * zh1[i] : 0.f;
                store_row(sm.gs + r * kBstLd, t0v);
                store_row(sm.as + r * kBstLd, do1);
            }
            __syncthreads();
            bst_colsum_d(sm.gs, sm.as, rows, sm.vsum[3 * 32 + (r & 31)]);                 // d ln1_g | d ln1_b
            __syncthreads();
            float dz1[16], dctx[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) { dz1[i] = 0.f; dctx[i] = 0.f; }
            if (on) layer_norm16_bwd(do1, sm.vec + VG1 * 16, zh1, rstd1, dz1);
            float dwo[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) dwo[i] = dz1[i];
            bst_drop(drop, 0, dwo);
            store_row(sm.gs + r * kBstLd, dwo);
            __syncthreads();
            bst_outer(sm.gs, sm.cs, rows, macc[MO]);                                    // d w_o = dwo (x) ctx
            bst_colsum_d(sm.gs, nullptr, rows, sm.vsum[4 * 32 + (r & 31)]);               // d b_o
            if (on) {
                matvec16(sm.w + MO * 256, dwo, dctx);
#pragma unroll
                for (int h = 0; h < H; ++h) {
                    float d = 0.f;
#pragma unroll
                    for (int j = 0; j < DH; ++j) d = fmaf(dctx[h * DH + j], ctx[h * DH + j], d);
                    sm.delta[r * H + h] = d;
                }
            }
            store_row(sm.dc + r * kBstLd, dctx);
            // ---- E. attention backward, key chunk after key chunk
            float dq[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) dq[i] = 0.f;
            for (int u0 = 0; u0 < L; u0 += kBstRows) {
                const int n = min(kBstRows, L - u0), u = u0 + r;
                const bool key = r < n;
                __syncthreads();
                if (key) bst_long_key_row(p, sm, b, u, kqk, kx, err_flag);
                __syncthreads();
                if (on) {        // as a query: the n keys of this chunk, summed from 0 and then added to dq
                    float dqc[16], mq[H], ilq[H], dlq[H];
#pragma unroll
                    for (int i = 0; i < 16; ++i) dqc[i] = 0.f;
#pragma unroll
                    for (int h = 0; h < H; ++h) { mq[h] = sm.mrow[r * H + h]; ilq[h] = sm.lrow[r * H + h]; dlq[h] = sm.delta[r * H + h]; }
                    for (int uu = 0; uu < n; ++uu) {
                        float kr[16], vr[16];
                        load_row(sm.ks + uu * kBstLd, kr);
                        load_row(sm.vs + uu * kBstLd, vr);
#pragma unroll
                        for (int h = 0; h < H; ++h) {
                            float sc = 0.f, dA = 0.f;
#pragma unroll
                            for (int j = 0; j < DH; ++j) {
                                sc = fmaf(q[h * DH + j], kr[h * DH + j], sc);
                                dA = fmaf(dctx[h * DH + j], vr[h * DH + j], dA);
                            }
                            const float a  = expf(sc * scale - mq[h]) * ilq[h];
                            const float dS = a * (dA - dlq[h]) * scale;
#pragma unroll
                            for (int j = 0; j < DH; ++j) dqc[h * DH + j] = fmaf(dS, kr[h * DH + j], dqc[h * DH + j]);
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 16; ++i) dq[i] += dqc[i];
                }
                float dk[16], dv[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) { dk[i] = 0.f; dv[i] = 0.f; }
                if (key) {       // as a live key: the rows of this query chunk
                    float kme[16], vme[16];
                    load_row(sm.ks + r * kBstLd, kme);
                    load_row(sm.vs + r * kBstLd, vme);
                    for (int tq = 0; tq < rows; ++tq) {
                        float qr[16], dr[16];
                        load_row(sm.qs + tq * kBstLd, qr);
                        load_row(sm.dc + tq * kBstLd, dr);
#pragma unroll
                        for (int h = 0; h < H; ++h) {
                            float sc = 0.f, dA = 0.f;
#pragma unroll
                            for (int j = 0; j < DH; ++j) {
                                sc = fmaf(qr[h * DH + j], kme[h * DH + j], sc);
                                dA = fmaf(dr[h * DH + j], vme[h * DH + j], dA);
                            }
                            const float a  = expf(sc * scale - sm.mrow[tq * H + h]) * sm.lrow[tq * H + h];
                            const float dS = a * (dA - sm.delta[tq * H + h]) * scale;
#pragma unroll
                            for (int j = 0; j < DH; ++j) {
                                dv[h * DH + j] = fmaf(a, dr[h * DH + j], dv[h * DH + j]);
                                dk[h * DH + j] = fmaf(dS, qr[h * DH + j], dk[h * DH + j]);
                            }
                        }
                    }
                }
                __syncthreads();
                store_row(sm.gs + r * kBstLd, dk);
                __syncthreads();
                bst_outer(sm.gs, kqk, n, macc[MK]);
                bst_colsum_d(sm.gs, nullptr, n, sm.vsum[6 * 32 + (r & 31)]);              // d b_k
                __syncthreads();
                store_row(sm.gs + r * kBstLd, dv);
                __syncthreads();
                bst_outer(sm.gs, kx, n, macc[MV]);
                bst_colsum_d(sm.gs, nullptr, n, sm.vsum[7 * 32 + (r & 31)]);              // d b_v
                if (key) {
                    float dpos[16], dx[16];
#pragma unroll
                    for (int i = 0; i < 16; ++i) dpos[i] = 0.f;
                    matvec16(sm.w + MK * 256, dk, dpos);
                    float* pr = out + u * 16;
#pragma unroll
                    for (int i = 0; i < 16; ++i) { pr[i] += dpos[i]; dx[i] = dpos[i]; }
                    matvec16(sm.w + MV * 256, dv, dx);
                    float* gx = g_x + (b * T + u) * 16;
                    if (t0 > 0) {
                        float prev[16];
                        load_row(gx, prev);
#pragma unroll
                        for (int i = 0; i < 16; ++i) dx[i] += prev[i];
                    }
                    store_row(gx, dx);
                }
            }
            // ---- F. the query side: dq (x) qk, W_q^T dq + dz1 into g_x and the position table
            __syncthreads();
            store_row(sm.gs + r * kBstLd, dq);
            __syncthreads();
            bst_outer(sm.gs, sm.qks, rows, macc[MQ]);
            bst_colsum_d(sm.gs, nullptr, rows, sm.vsum[5 * 32 + (r & 31)]);               // d b_q
            if (on) {
                float dqk[16];
#pragma unroll
                for (int i = 0; i < 16; ++i) dqk[i] = dz1[i];                // residual path of LayerNorm 1
                matvec16(sm.w + MQ * 256, dq, dqk);
                float* pr = out + t * 16;
#pragma unroll
                for (int i = 0; i < 16; ++i) pr[i] += dqk[i];
                float* gx = g_x + (b * T + t) * 16;
                if (t < L) {                                                // a live key: its key side wrote first
                    float prev[16];
                    load_row(gx, prev);
#pragma unroll
                    for (int i = 0; i < 16; ++i) dqk[i] += prev[i];
                }
                store_row(gx, dqk);
            }
            __syncthreads();
        }
    }

    float* o = out + T * 16;
    const int e2 = r * 2;
    const int mat_off[6] = {0, 272, 544, 816, 1120, 1392};   // wq wk wv wo w1 w2
#pragma unroll
    for (int m = 0; m < 6; ++m) { o[mat_off[m] + e2] = macc[m][0]; o[mat_off[m] + e2 + 1] = macc[m][1]; }
    if (r < 16) {
        o[256 + r]  = (float)sm.vsum[5 * 32 + r];    // bq
        o[528 + r]  = (float)sm.vsum[6 * 32 + r];    // bk
        o[800 + r]  = (float)sm.vsum[7 * 32 + r];    // bv
        o[1072 + r] = (float)sm.vsum[4 * 32 + r];    // bo
        o[1088 + r] = (float)sm.vsum[3 * 32 + r];    // ln1_g
        o[1376 + r] = (float)sm.vsum[2 * 32 + r];    // b1
        o[1648 + r] = (float)sm.vsum[1 * 32 + r];    // b2
        o[1664 + r] = (float)sm.vsum[0 * 32 + r];    // ln2_g
    } else if (r < 32) {
        o[1104 + r - 16] = (float)sm.vsum[3 * 32 + r];   // ln1_b
        o[1680 + r - 16] = (float)sm.vsum[0 * 32 + r];   // ln2_b
    }
}

static int bst_fill(const rk_bst_block_t* blk, const float* table, const int64_t* idx, int64_t table_rows,
                    const float* x_in, const int64_t* seq_len, int64_t B, int T, int pool_mean, BstParams* p) {
    RK_CHECK_ARG(blk, "bst: block is NULL");
    const float* w[6]  = {blk->wq, blk->wk, blk->wv, blk->wo, blk->w1, blk->w2};
    const float* v[10] = {blk->bq, blk->bk, blk->bv, blk->bo, blk->ln1_g, blk->ln1_b, blk->b1, blk->b2,
                          blk->ln2_g, blk->ln2_b};
    for (int i = 0; i < 6; ++i) { RK_CHECK_ARG(w[i], "bst: weight matrix %d is NULL", i); p->w[i] = w[i]; }
    for (int i = 0; i < 10; ++i) { RK_CHECK_ARG(v[i], "bst: vector %d is NULL", i); p->vec[i] = v[i]; }
    RK_CHECK_ARG(blk->pos && seq_len, "bst: NULL pos or seq_len");
    RK_CHECK_ARG((x_in != nullptr) != (table != nullptr && idx != nullptr),
                 "bst: pass either x_in or (table, idx)");
    RK_CHECK_ARG(T >= 1, "bst: sequence length %d is below 1", T);
    RK_CHECK_ARG(blk->precision != RK_BST_BF16_TENSOR || T <= kBstRows,
                 "bst: the tensor-core block takes sequences of at most %d positions (got %d); "
                 "use RK_BST_FP32 for longer ones", kBstRows, T);
    RK_CHECK_ARG(B >= 0, "bst: B=%lld", (long long)B);
    const void* src = x_in ? (const void*)x_in : (const void*)table;
    RK_CHECK_ARG(((uintptr_t)src % 16) == 0, "bst: input rows must be 16-byte aligned");
    p->pos = blk->pos;
    p->table = table; p->idx = idx; p->table_rows = table_rows; p->x_in = x_in;
    p->seq_len = seq_len;
    p->B = B; p->T = T; p->S = T <= kBstRows ? kBstRows / T : 1; p->pool_mean = pool_mean;
    RK_CHECK_ARG(blk->dropout_p >= 0.f && blk->dropout_p < 1.f, "bst: dropout_p %g outside [0,1)", (double)blk->dropout_p);
    p->drop_thr = (uint32_t)lrintf(blk->dropout_p * 65536.f);
    p->drop_scale = 1.0f / (1.0f - blk->dropout_p);
    p->rng = (const unsigned long long*)blk->rng;
    RK_CHECK_ARG(p->drop_thr == 0 || p->rng, "bst: dropout_p > 0 needs rng (device [seed, offset])");
    p->n_tiles = ceil_div(B, p->S);
    return 0;
}

template <int H>
static int bst_launch_fwd(const BstParams& p, float* y_out, float* pool_out, int pool_ld, int32_t* err_flag,
                          cudaStream_t s) {
    const size_t smem = BstSmem::bytes(p.T, H, false);
    RK_CUDA(cudaFuncSetAttribute(bst_fwd_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t grid = p.n_tiles;
    const int64_t cap = (int64_t)sm_count() * 4;
    if (grid > cap) grid = cap;
    bst_fwd_kernel<H><<<(int)grid, kBstThreads, smem, s>>>(p, y_out, pool_out, pool_ld, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}
template <int H>
static int bst_launch_fwd_long(const BstParams& p, float* y_out, float* pool_out, int pool_ld, int32_t* err_flag,
                               cudaStream_t s) {
    const size_t smem = BstLongSmem::bytes(H, false);
    RK_CUDA(cudaFuncSetAttribute(bst_fwd_long_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t grid = p.B;
    const int64_t cap = (int64_t)sm_count() * 32;
    if (grid > cap) grid = cap;
    bst_fwd_long_kernel<H><<<(int)grid, kBstThreads, smem, s>>>(p, y_out, pool_out, pool_ld, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}
template <int H>
static int bst_launch_bwd_long(const BstParams& p, const float* g_y, const float* g_pool, int g_pool_ld, float* g_x,
                               float* partials, int n_ctas, int32_t* err_flag, cudaStream_t s) {
    const size_t smem = BstLongSmem::bytes(H, true);
    RK_CUDA(cudaFuncSetAttribute(bst_bwd_long_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bst_bwd_long_kernel<H><<<n_ctas, kBstThreads, smem, s>>>(p, g_y, g_pool, g_pool_ld, g_x, partials, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}
template <int H>
static int bst_launch_bwd(const BstParams& p, const float* g_y, const float* g_pool, int g_pool_ld, float* g_x,
                          float* partials, int n_ctas, int32_t* err_flag, cudaStream_t s) {
    const size_t smem = BstSmem::bytes(p.T, H, true);
    RK_CHECK_ARG(smem <= 227 * 1024, "bst_bwd: %zu bytes of shared memory", smem);
    RK_CUDA(cudaFuncSetAttribute(bst_bwd_kernel<H>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bst_bwd_kernel<H><<<n_ctas, kBstThreads, smem, s>>>(p, g_y, g_pool, g_pool_ld, g_x, partials, err_flag);
    RK_LAUNCH_CHECK();
    return 0;
}

}  // namespace rk

extern "C" {

int rk_bst_grad_floats(int T) { return T * 16 + 6 * 256 + 160; }

// Above 128 positions (fp32) a CTA owns whole samples: at most two CTAs per SM, and at most 2^26 floats of
// partials (T*16 + 1696 per CTA) in all.
int rk_bst_bwd_ctas(int64_t B, int T, int precision) {
    if (T < 1 || B <= 0) return 1;
    if (T > rk::kBstRows) {
        if (precision != RK_BST_FP32) return 1;
        int64_t cap = (int64_t)rk::sm_count() * 2;
        const int64_t fit = ((int64_t)1 << 26) / rk_bst_grad_floats(T);
        if (cap > fit) cap = fit > 1 ? fit : 1;
        return (int)(B < cap ? B : cap);
    }
    if (precision == RK_BST_BF16_TENSOR) return rk::bst_tc_bwd_ctas(B, T);
    const int64_t tiles = rk::ceil_div(B, rk::kBstRows / T);
    const int64_t cap = (int64_t)rk::sm_count() * 2;
    return (int)(tiles < cap ? tiles : cap);
}

int rk_bst_block_fwd(const rk_bst_block_t* blk, int nhead, const float* table, const int64_t* idx,
                     int64_t table_rows, const float* x_in, const int64_t* seq_len, int64_t B, int T,
                     float* y_out, float* pool_out, int pool_ld, int pool_mean, int32_t* err_flag,
                     rk_stream_t stream_) {
    using namespace rk;
    BstParams p;
    memset(&p, 0, sizeof(p));
    if (int rc = bst_fill(blk, table, idx, table_rows, x_in, seq_len, B, T, pool_mean, &p)) return rc;
    RK_CHECK_ARG(y_out || pool_out, "bst_fwd: no output requested");
    if (B == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream_;
    if (blk->precision == RK_BST_BF16_TENSOR) return bst_tc_fwd(p, nhead, y_out, pool_out, pool_ld, err_flag, s);
    RK_CHECK_ARG(blk->precision == RK_BST_FP32, "bst_fwd: unknown precision %d", blk->precision);
    if (T > kBstRows) {
        switch (nhead) {
            case 1:  return bst_launch_fwd_long<1>(p, y_out, pool_out, pool_ld, err_flag, s);
            case 2:  return bst_launch_fwd_long<2>(p, y_out, pool_out, pool_ld, err_flag, s);
            case 4:  return bst_launch_fwd_long<4>(p, y_out, pool_out, pool_ld, err_flag, s);
            case 8:  return bst_launch_fwd_long<8>(p, y_out, pool_out, pool_ld, err_flag, s);
            case 16: return bst_launch_fwd_long<16>(p, y_out, pool_out, pool_ld, err_flag, s);
        }
        RK_CHECK_ARG(false, "bst: nhead %d does not divide d_model 16 (the reference's view() fails too)", nhead);
    }
    switch (nhead) {
        case 1:  return bst_launch_fwd<1>(p, y_out, pool_out, pool_ld, err_flag, s);
        case 2:  return bst_launch_fwd<2>(p, y_out, pool_out, pool_ld, err_flag, s);
        case 4:  return bst_launch_fwd<4>(p, y_out, pool_out, pool_ld, err_flag, s);
        case 8:  return bst_launch_fwd<8>(p, y_out, pool_out, pool_ld, err_flag, s);
        case 16: return bst_launch_fwd<16>(p, y_out, pool_out, pool_ld, err_flag, s);
    }
    RK_CHECK_ARG(false, "bst: nhead %d does not divide d_model 16 (the reference's view() fails too)", nhead);
    return -1;
}

int rk_bst_block_bwd(const rk_bst_block_t* blk, int nhead, const float* table, const int64_t* idx,
                     int64_t table_rows, const float* x_in, const int64_t* seq_len, int64_t B, int T,
                     const float* g_y, const float* g_pool, int g_pool_ld, int pool_mean, float* g_x,
                     float* g_params, float* partials, int n_ctas, int32_t* err_flag, rk_stream_t stream_) {
    using namespace rk;
    BstParams p;
    memset(&p, 0, sizeof(p));
    if (int rc = bst_fill(blk, table, idx, table_rows, x_in, seq_len, B, T, pool_mean, &p)) return rc;
    RK_CHECK_ARG((g_y || g_pool) && g_x && g_params && partials, "bst_bwd: NULL pointer");
    RK_CHECK_ARG(n_ctas == rk_bst_bwd_ctas(B, T, blk->precision), "bst_bwd: n_ctas %d != rk_bst_bwd_ctas", n_ctas);
    if (B == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream_;
    if (blk->precision == RK_BST_BF16_TENSOR) {
        if (int rc2 = bst_tc_bwd(p, nhead, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s)) return rc2;
        return launch_reduce_partials(partials, n_ctas, rk_bst_grad_floats(T), g_params, s);
    }
    RK_CHECK_ARG(blk->precision == RK_BST_FP32, "bst_bwd: unknown precision %d", blk->precision);
    int rc = -1;
    if (T > kBstRows) {
        switch (nhead) {
            case 1:  rc = bst_launch_bwd_long<1>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
            case 2:  rc = bst_launch_bwd_long<2>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
            case 4:  rc = bst_launch_bwd_long<4>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
            case 8:  rc = bst_launch_bwd_long<8>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
            case 16: rc = bst_launch_bwd_long<16>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
            default: RK_CHECK_ARG(false, "bst: nhead %d does not divide d_model 16", nhead);
        }
        if (rc) return rc;
        return launch_reduce_partials(partials, n_ctas, rk_bst_grad_floats(T), g_params, s);
    }
    switch (nhead) {
        case 1:  rc = bst_launch_bwd<1>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
        case 2:  rc = bst_launch_bwd<2>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
        case 4:  rc = bst_launch_bwd<4>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
        case 8:  rc = bst_launch_bwd<8>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
        case 16: rc = bst_launch_bwd<16>(p, g_y, g_pool, g_pool_ld, g_x, partials, n_ctas, err_flag, s); break;
        default: RK_CHECK_ARG(false, "bst: nhead %d does not divide d_model 16", nhead);
    }
    if (rc) return rc;
    const int count = rk_bst_grad_floats(T);
    return launch_reduce_partials(partials, n_ctas, count, g_params, s);
}

}  // extern "C"
