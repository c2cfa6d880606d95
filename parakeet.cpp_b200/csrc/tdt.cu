// tdt.cu -- K10: batched TDT greedy decode as ONE persistent cooperative kernel.
//
// Replaces tdt_greedy_decode / tdt_greedy_decode_with_timestamps (reference
// src/tdt.cpp:36-110, :122-201) and what they call per step: RNNTPrediction::step
// (src/rnnt.cpp:22-28) -> Embedding -> LSTM::step (src/lstm.cpp:40-49) -> LSTMCell::forward
// (:11-29, gate order i,f,g,o, one merged bias) and TDTJoint::forward (src/tdt.cpp:15-24,
// pred_proj_ without bias, two log_softmax heads), argmax label (first maximum) / duration.
//
// The reference decodes utterances one after another with a host round trip per symbol.
// Here all utterances of the batch advance in lock step inside one kernel; the serial
// chain per utterance is unchanged:
//     saved = state; pred = LSTM(embed(token)); (label, dur) = joint(enc[t], pred)
//     blank  -> state = saved, t += max(skip, 1)
//     symbol -> emit (start = t, end = min(t + max(skip,1) - 1, T-1), conf = exp(lp)),
//               token = symbol, t += skip (skip = 0 stays on the frame)
// max_symbols_per_step has no observable effect in the reference (after 10 zero-duration
// symbols the inner loop is simply re-entered on the same frame with the same state), so it
// is not modelled; a token capacity bounds the loop instead (reference would livelock).
//
// RNNT mode (p.max_symbols > 0, D = 0: rnnt_greedy_decode(_with_timestamps), src/rnnt.cpp:56-177) reuses every phase;
// only the state update differs: blank -> state = saved, t += 1; symbol -> emit (start = end = t), token = symbol,
// stay on the frame; the max_symbols-th symbol on one frame moves to the next frame with state and token KEPT.  The
// per-utterance symbol count is replicated in shared memory like the frame position.  The engine sizes the token
// capacity as Tmax * max_symbols, the most the rule can emit, so an RNNT decode is never truncated.
//
// Design (weights-stationary, 2-D decomposition): the grid is one CTA per SM, grouped in thread-block
// CLUSTERS of CL = 4 (or 2) CTAs.  A cluster owns a block of weight ROWS (LSTM units, joint-hidden
// rows, label/duration rows); inside the cluster, CTA rank q owns the K-SLICE [q K/CL, (q+1) K/CL) of
// those rows, resident in shared memory for the whole decode.  Per phase a CTA therefore streams only
// its k-slice of the per-utterance vectors (h, z) from L2 -- 1/CL of the bytes a row-only split needs
// (that stream, LSU-bound at ~20 B/clk/SM, was the largest part of a step) -- multiplies it with its
// weight slice on tensor cores, and the CL partial sums of a row meet through distributed shared
// memory: after one cluster barrier each CTA adds the partials of the rows it finalises, reading its
// peers' buffers with ld.shared::cluster in a fixed order (deterministic).
//   P1 LSTM gates + cell (per layer) | P2 joint hidden | P3 logits -> per-CTA (max, sum-exp)
//   partials + atomicMax of packed (value, index) keys | P4 state update, replicated in every
//   CTA from the keys (no barrier before the next P1; confidences are finalised one phase later
//   from the partials, in a fixed order, by the CTA that owns the utterance, while it waits at a
//   grid barrier).
// Three monotonic-counter grid barriers per step (cooperative launch guarantees co-residency);
// they also order the reuse of the partial-sum buffers between phases.
// enc_proj(enc)+bias for all frames and the layer-0 input table W_ih.E[token]+b for all
// tokens are precomputed by GEMMs (engine.cu).
//
// Every product runs on mma.sync.m16n8k16 with the bf16 hi/lo operand split of the encoder GEMMs
// (x_hi.W_hi + x_hi.W_lo + x_lo.W_hi, fp32 accumulate: ~16 mantissa bits): weights are split once
// at load (engine.cu: row = [hi: K][lo: K] bf16); the PRODUCER of a vector (LSTM cell, joint hidden)
// stores it already split, as bf16 hi / lo planes [utterance][k], so consumers only copy (cp.async)
// and read A fragments with ldmatrix.  Operands of the phase epilogues (G0[token], EP[t], biases)
// are fetched BEFORE the product so their L2 latency overlaps it; the LSTM cell state never leaves
// shared memory.
#include <cstdlib>

#include "kernels.h"

namespace pk {
namespace {

constexpr int NWARP = 8;
constexpr int NTHR = NWARP * 32;
constexpr int BCH = 64;         // utterances per pass (4 MMA m-blocks)
constexpr int RG = 80;          // weight rows per pass of a cluster (10 MMA n-blocks = 20 LSTM units)
constexpr int RLD = BCH + 4;    // row stride of the partial-sum buffer (floats): conflict-free fragment stores
constexpr int MYMAX = 40;       // rows one CTA finalises per pass (RG / CL, whole LSTM units: 10 units at CL = 2)
constexpr int NPV = MYMAX * BCH / NTHR;   // epilogue items per thread

__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async8(uint32_t dst, const void *gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
    asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void mma_bf16(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
// 32-bit weight fragment word (two consecutive k of one row); weights never change during the kernel
template <bool WS>
__device__ __forceinline__ uint32_t ldw32(const bf16 *p) {
    uint32_t v;
    if (WS) asm("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(smem_addr(p)));
    else asm("ld.global.nc.b32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void store_split(bf16 *hi, bf16 *lo, size_t idx, float v) {
    const bf16 h = __float2bfloat16_rn(v);
    hi[idx] = h;
    lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
}
// ---- thread-block cluster primitives
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t smem_a, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_a), "r"(rank));
    return r;
}
__device__ __forceinline__ float ld_cluster_f32(uint32_t a) {
    float v;
    asm volatile("ld.shared::cluster.f32 %0, [%1];" : "=f"(v) : "r"(a) : "memory");
    return v;
}

// Stage this CTA's k-slice of the 64 utterance vectors: xs[plane][utterance][KS + 8] bf16.
//   xsrc(b) -> pointer to the first element of the slice of utterance b's hi row; lo = hi + lo_off
template <typename XSrc>
__device__ __forceinline__ void stage_x(XSrc xsrc, size_t lo_off, int KS, int Bpad, int bc, bf16 *xs) {
    const int XLD = KS + 8, pieces = KS / 8;          // 16-byte pieces per row
    const int xrows = min(BCH, Bpad);                 // rows per plane of the staging buffer (see tdt_smem_bytes)
    const uint32_t xs_s = smem_addr(xs);
    for (int idx = threadIdx.x; idx < BCH * pieces; idx += NTHR) {
        const int row = idx / pieces, pc = idx - row * pieces;
        if (bc + row >= Bpad) continue;               // rows past the batch: stale data, results discarded
        const bf16 *s = xsrc(bc + row) + pc * 8;
        const uint32_t dst = xs_s + (uint32_t)(row * XLD + pc * 8) * 2u;
        cp_async16(dst, s);
        cp_async16(dst + (uint32_t)(xrows * XLD) * 2u, s + lo_off);
    }
    cp_async_commit_wait_all();
    __syncthreads();
}

// acc[nb] += W[rows of n-block nb][k-slice] . xs   for the NBH n-blocks of this warp
//   W: row r at W + r * RS (bf16 elements): [hi ...][lo ...] with lo at +LO; k index 0 = first k of the slice
//   warp w: utterance block (w & 3), n-blocks [ (w >> 2) * NBH, +NBH )
template <int NBH, bool WS>
__device__ __forceinline__ void mma_slice(float (&acc)[NBH][4], const bf16 *W, int RS, int LO, int R, int KS, const bf16 *xs, int xrows) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, cq = lane & 3;
    const int mb = warp & 3, nh = warp >> 2;
    const int XLD = KS + 8;
    const uint32_t a_base = smem_addr(xs) + (uint32_t)((mb * 16 + (lane & 7) + ((lane >> 3) & 1) * 8) * XLD + ((lane >> 4) & 1) * 8) * 2u;
    const uint32_t lo_plane = (uint32_t)(xrows * XLD) * 2u;   // (m-blocks past xrows read stale shared memory: results discarded)
    const bf16 *wrow[NBH];
#pragma unroll
    for (int nb = 0; nb < NBH; ++nb)
        wrow[nb] = W + (size_t)min((nh * NBH + nb) * 8 + g, R - 1) * RS + 2 * cq;   // rows >= R: clamped, discarded
    for (int ks = 0; ks < KS / 16; ++ks) {
        uint32_t ah[4], al[4];
        ldsm_x4(ah, a_base + ks * 32u);
        ldsm_x4(al, a_base + lo_plane + ks * 32u);
#pragma unroll
        for (int nb = 0; nb < NBH; ++nb) {
            const bf16 *wp = wrow[nb] + ks * 16;
            const uint32_t b0h = ldw32<WS>(wp), b1h = ldw32<WS>(wp + 8), b0l = ldw32<WS>(wp + LO), b1l = ldw32<WS>(wp + LO + 8);
            mma_bf16(acc[nb], ah, b0h, b1h);
            mma_bf16(acc[nb], ah, b0l, b1l);
            mma_bf16(acc[nb], al, b0h, b1h);
        }
    }
}
template <int NBH>
__device__ __forceinline__ void store_partials(const float (&acc)[NBH][4], float *red) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, cq = lane & 3;
    const int mb = warp & 3, nh = warp >> 2;
#pragma unroll
    for (int nb = 0; nb < NBH; ++nb) {
        const int n = (nh * NBH + nb) * 8 + 2 * cq, u = mb * 16 + g;
        red[n * RLD + u] = acc[nb][0];
        red[(n + 1) * RLD + u] = acc[nb][1];
        red[n * RLD + u + 8] = acc[nb][2];
        red[(n + 1) * RLD + u + 8] = acc[nb][3];
    }
}

// measurement aid: cycles thread 0 of CTA 0 spent in the sections of cluster_pass, summed over a decode:
// [0] x staging + operand prefetch until the staged slice is visible, [1] products, [2] partial store + cluster barrier,
// [3] DSMEM gather + finalisation, [4] number of passes
__device__ long long g_pass_clk[8];

// One pass over R <= RG weight rows of the cluster: up to two products accumulated together
// (W1 . x1 [+ W2 . x2]), partial sums exchanged through DSMEM, rows finalised by their owner CTA.
//   myrow(i) -> row (0..R-1) of the i-th row this CTA finalises, i < nmy (nmy <= MYMAX)
//   pre(r, b) -> float operand of the epilogue, fetched before the products;  fin(i, r, b, sum, pre)
//   post() runs right after the last product has read its weights (e.g. to start the asynchronous copy of the next
//   weight tile into the staging buffer while the partial sums are exchanged and finalised)
template <int CL, int NBH, bool WS1, bool WS2, typename X1, typename X2, typename MyRow, typename Pre, typename Fin, typename Post>
__device__ __forceinline__ void cluster_pass(const bf16 *W1, int RS1, int LO1, X1 x1, const bf16 *W2, int RS2, int LO2, X2 x2,
                                             size_t lo_off, int R, int KS, int Bpad, int bc, bf16 *xs, float *red, int nmy,
                                             MyRow myrow, Pre pre, Fin fin, Post post, bool stage_x1 = true) {
    const int xrows = min(BCH, Bpad);
    const bool prof = blockIdx.x == 0 && threadIdx.x == 0;
    long long pt0 = 0, pt1 = 0, pt2 = 0, pt3 = 0;
    if (prof) pt0 = clock64();
    float acc[NBH][4];
#pragma unroll
    for (int nb = 0; nb < NBH; ++nb) acc[nb][0] = acc[nb][1] = acc[nb][2] = acc[nb][3] = 0.f;
    // stage x1 (async) and fetch the epilogue operands while it is in flight
    float pv[NPV];
    {
        const int XLD = KS + 8, pieces = KS / 8;
        const uint32_t xs_s = smem_addr(xs);
        if (stage_x1)               // (false: xs still holds this slice from the previous pass of the same phase)
        for (int idx = threadIdx.x; idx < BCH * pieces; idx += NTHR) {
            const int row = idx / pieces, pc = idx - row * pieces;
            if (bc + row >= Bpad) continue;
            const bf16 *s = x1(bc + row) + pc * 8;
            const uint32_t dst = xs_s + (uint32_t)(row * XLD + pc * 8) * 2u;
            cp_async16(dst, s);
            cp_async16(dst + (uint32_t)(xrows * XLD) * 2u, s + lo_off);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    }
#pragma unroll
    for (int j = 0; j < NPV; ++j) {
        const int idx = threadIdx.x + j * NTHR, i = idx / BCH, b2 = idx % BCH;
        pv[j] = (i < nmy && bc + b2 < Bpad) ? pre(myrow(i), bc + b2) : 0.f;
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
    if (prof) pt1 = clock64();
    mma_slice<NBH, WS1>(acc, W1, RS1, LO1, R, KS, xs, xrows);
    if (W2 != nullptr) {
        __syncthreads();                              // everyone is done reading x1
        stage_x(x2, lo_off, KS, Bpad, bc, xs);
        mma_slice<NBH, WS2>(acc, W2, RS2, LO2, R, KS, xs, xrows);
    }
    post();
    if (prof) pt2 = clock64();
    store_partials<NBH>(acc, red);
    cluster_sync_all();                               // all CL partial buffers complete and visible
    if (prof) pt3 = clock64();
    uint32_t peer[CL];
#pragma unroll
    for (int q = 0; q < CL; ++q) peer[q] = mapa_rank(smem_addr(red), (uint32_t)q);
#pragma unroll
    for (int j = 0; j < NPV; ++j) {
        const int idx = threadIdx.x + j * NTHR, i = idx / BCH, b2 = idx % BCH;
        if (i < nmy && bc + b2 < Bpad) {
            const int r = myrow(i);
            const uint32_t off = (uint32_t)(r * RLD + b2) * 4u;
            float s = 0.f;
#pragma unroll
            for (int q = 0; q < CL; ++q) s += ld_cluster_f32(peer[q] + off);
            fin(i, r, bc + b2, s, pv[j]);
        }
    }
    __syncthreads();
    if (prof) {
        const long long pt4 = clock64();
        g_pass_clk[0] += pt1 - pt0;
        g_pass_clk[1] += pt2 - pt1;
        g_pass_clk[2] += pt3 - pt2;
        g_pass_clk[3] += pt4 - pt3;
        g_pass_clk[4] += 1;
    }
}

struct NoPost {
    __device__ __forceinline__ void operator()() const {}
};
template <int CL, bool WS1, bool WS2, typename X1, typename X2, typename MyRow, typename Pre, typename Fin, typename Post = NoPost>
__device__ __forceinline__ void cluster_pass_n(const bf16 *W1, int RS1, int LO1, X1 x1, const bf16 *W2, int RS2, int LO2, X2 x2,
                                               size_t lo_off, int R, int KS, int Bpad, int bc, bf16 *xs, float *red, int nmy,
                                               MyRow myrow, Pre pre, Fin fin, Post post = Post(), bool stage_x1 = true) {
    if (R <= 16) cluster_pass<CL, 1, WS1, WS2>(W1, RS1, LO1, x1, W2, RS2, LO2, x2, lo_off, R, KS, Bpad, bc, xs, red, nmy, myrow, pre, fin, post, stage_x1);
    else if (R <= 32) cluster_pass<CL, 2, WS1, WS2>(W1, RS1, LO1, x1, W2, RS2, LO2, x2, lo_off, R, KS, Bpad, bc, xs, red, nmy, myrow, pre, fin, post, stage_x1);
    else if (R <= 48) cluster_pass<CL, 3, WS1, WS2>(W1, RS1, LO1, x1, W2, RS2, LO2, x2, lo_off, R, KS, Bpad, bc, xs, red, nmy, myrow, pre, fin, post, stage_x1);
    else cluster_pass<CL, 5, WS1, WS2>(W1, RS1, LO1, x1, W2, RS2, LO2, x2, lo_off, R, KS, Bpad, bc, xs, red, nmy, myrow, pre, fin, post, stage_x1);
}

// Monotonic-counter grid barrier (all CTAs are co-resident: cooperative launch), split into
// arrive / wait so that work which does not depend on the other CTAs can sit in between.
// Cheaper than cooperative_groups' grid.sync() and traps instead of hanging if a CTA never arrives.
// (A hierarchical variant -- hardware cluster barrier, one atomic per cluster, second cluster barrier -- was measured
// SLOWER: 5.4-6.1k cycles per use against 3.2-5.1k; two barrier.cluster round trips cost more than the 111 atomics saved.)
// Same-address atomics serialise in the L2 (~27 cycles each: 148 of them made a barrier 3.2-5.1k cycles), so the arrivals
// are spread over GBAR counters on different 128-byte lines (CTA c -> counter c % GBAR) and lanes 0..GBAR-1 of warp 0
// poll one counter each.
constexpr int GBAR = 8, GBAR_STRIDE = 32;      // counters, uints between them
__device__ __forceinline__ void grid_arrive(unsigned int *counter) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter + (blockIdx.x % GBAR) * GBAR_STRIDE, 1u);
    }
}
__device__ __forceinline__ void grid_wait(unsigned int *counter, unsigned int round /* 1, 2, ... */) {
    if (threadIdx.x < 32) {
        const int l = threadIdx.x;
        if (l < GBAR) {
            const unsigned int members = (gridDim.x - l + GBAR - 1) / GBAR;     // CTAs that arrive on counter l
            const unsigned int target = members * round;
            unsigned int v, spin = 0;
            do {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter + l * GBAR_STRIDE) : "memory");
                if (++spin > (1u << 28)) __trap();
            } while (v < target);
        }
        __syncwarp();
        if (threadIdx.x == 0) __threadfence();
    }
    __syncthreads();
}

// (value, index) packed so that atomicMax picks the larger value and, on ties, the SMALLER index
// (the reference's strict '>' scans keep the first maximum).
__device__ __forceinline__ unsigned long long pack_key(float v, int idx) {
    unsigned int u = __float_as_uint(v);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned int)idx);
}
__device__ __forceinline__ void unpack_key(unsigned long long k, float &v, int &idx) {
    unsigned int u = (unsigned int)(k >> 32);
    u = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
    v = __uint_as_float(u);
    idx = (int)(0xFFFFFFFFu - (unsigned int)(k & 0xFFFFFFFFu));
}

struct TdtGeom {            // per-cluster row blocks and per-CTA shared-memory sizes (host and device agree)
    int UPC, JPC, OPC;      // LSTM units / joint rows / output rows per CLUSTER
    int KSP, KSJ;           // k-slice widths for K = P and K = J
    int MU;                 // LSTM units one CTA finalises (ceil(UPC / CL))
};
__host__ __device__ inline TdtGeom tdt_geom(int P, int J, int NO, int n_clusters, int CL) {
    TdtGeom q;
    q.UPC = (P + n_clusters - 1) / n_clusters;
    q.JPC = (J + n_clusters - 1) / n_clusters;
    q.OPC = (NO + n_clusters - 1) / n_clusters;
    q.KSP = P / CL;
    q.KSJ = J / CL;
    q.MU = (q.UPC + CL - 1) / CL;
    return q;
}

template <int CL>
__global__ void __launch_bounds__(NTHR, 1) tdt_decode_kernel(TdtParams p) {
    extern __shared__ __align__(16) float sm[];
    const int G = gridDim.x, g = blockIdx.x, tid = threadIdx.x;
    const int NC = G / CL;                                   // clusters
    const int cid = (int)cluster_id_x(), rank = (int)cluster_ctarank();
    const int P = p.P, J = p.J, V = p.V, D = p.D, L = p.L, Bpad = p.Bpad;
    const int NO = V + D;
    const TdtGeom ge = tdt_geom(P, J, NO, NC, CL);
    const int u0 = min(cid * ge.UPC, P), u1 = min(u0 + ge.UPC, P), nU = u1 - u0;        // this cluster's LSTM units
    const int j0 = min(cid * ge.JPC, J), j1 = min(j0 + ge.JPC, J);
    const int o0 = min(cid * ge.OPC, NO), o1 = min(o0 + ge.OPC, NO);
    const int KSP = ge.KSP, KSJ = ge.KSJ;
    const int kP0 = rank * KSP, kJ0 = rank * KSJ;                                       // this CTA's k-slices
    const int RSP = 2 * (KSP + 4), RSJ = 2 * (KSJ + 4);      // smem weight row strides (bf16): [hi KS+4][lo KS+4]

    // ---- shared memory carve-up: [partials][gates][x slice][cell state][decode state][weights...]
    float *red = sm;                                          // [RG][RLD] this CTA's k-slice partial sums
    float *gsm = red + RG * RLD;                              // [MYMAX][BCH] gate pre-activations / logits of my rows
    bf16 *xs = reinterpret_cast<bf16 *>(gsm + MYMAX * BCH);   // [2][BCH][KSmax + 8]
    const int KSmax = max(KSP, KSJ);
    float *csm = reinterpret_cast<float *>(xs + (size_t)2 * min(BCH, Bpad) * (KSmax + 8));  // [L][2][MU][Bpad] LSTM cell state
    int *s_cur = reinterpret_cast<int *>(csm + (size_t)L * 2 * ge.MU * Bpad);    // replicated decode state, [Bpad] each
    int *s_token = s_cur + Bpad, *s_tpos = s_token + Bpad, *s_active = s_tpos + Bpad, *s_ntok = s_active + Bpad;
    int *s_pend = s_ntok + Bpad;                   // slot of a token whose confidence is still pending (-1: none)
    float *s_vraw = reinterpret_cast<float *>(s_pend + Bpad);   // raw (unboosted) logit of that token (phrase boosting)
    int *s_nsym = reinterpret_cast<int *>(s_vraw + Bpad);       // RNNT: symbols emitted on the current frame
    bf16 *wbf = reinterpret_cast<bf16 *>(s_nsym + (p.max_symbols > 0 ? Bpad : 0));
    // Weight rows in global memory are [hi: K][lo: K]; a CTA keeps columns [k0, k0 + KS) of its cluster's rows.
    auto stage_rows = [&](bf16 *dst, const bf16 *src, int rows, int K, int k0, int KS) {
        const int RS = 2 * (KS + 4), n8 = KS / 4;            // 8-byte pieces per half row
        for (int i = tid; i < rows * n8; i += blockDim.x) {
            const int r = i / n8, pc = i - r * n8;
            const uint2 *s = reinterpret_cast<const uint2 *>(src + (size_t)r * 2 * K + k0) + pc;
            uint2 *d = reinterpret_cast<uint2 *>(dst + (size_t)r * RS) + pc;
            *d = *s;
            *reinterpret_cast<uint2 *>(reinterpret_cast<bf16 *>(d) + KS + 4) = *reinterpret_cast<const uint2 *>(reinterpret_cast<const bf16 *>(s) + K);
        }
    };
    // LSTM weights arrive "unit-major" (row = unit*4 + gate, engine.cu), so the cluster's rows
    // [u0*4, u1*4) are one contiguous block: W_hh always lives in shared memory, W_ih of the
    // upper layers too when it fits (else its fragments are read from L2).
    const bf16 *w_hh[PK_MAX_LSTM], *w_ih[PK_MAX_LSTM];
    {
        bf16 *cur = wbf;
        for (int l = 0; l < L; ++l) {
            stage_rows(cur, p.Whh[l] + (size_t)u0 * 4 * 2 * P, nU * 4, P, kP0, KSP);
            w_hh[l] = cur;
            cur += (size_t)ge.UPC * 4 * RSP;
            w_ih[l] = nullptr;
            if (l > 0) {
                if (p.wih_in_smem) {
                    stage_rows(cur, p.Wih[l] + (size_t)u0 * 4 * 2 * P, nU * 4, P, kP0, KSP);
                    w_ih[l] = cur;
                    cur += (size_t)ge.UPC * 4 * RSP;
                } else {
                    w_ih[l] = p.Wih[l] + (size_t)u0 * 4 * 2 * P + kP0;     // global: row stride 2P, lo at +P
                }
            }
        }
    }
    bf16 *w_p = wbf + 2 * (size_t)p.smem_lstm_floats;        // [JPC] rows, K-slice of P
    stage_rows(w_p, p.Wp + (size_t)j0 * 2 * P, j1 - j0, P, kP0, KSP);
    const bf16 *w_o;                                         // [OPC] rows, K-slice of J: shared if it fits
    if (p.out_in_smem) {
        bf16 *w_os = w_p + (size_t)ge.JPC * RSP;
        stage_rows(w_os, p.Wout + (size_t)o0 * 2 * J, o1 - o0, J, kJ0, KSJ);
        w_o = w_os;
    } else {
        w_o = p.Wout + (size_t)o0 * 2 * J + kJ0;              // global: row stride 2J, lo at +J
    }
    const int RSO = p.out_in_smem ? RSJ : 2 * J, LOO = p.out_in_smem ? KSJ + 4 : J;
    // (48-80 rows per pass)  Weights that do not fit in shared memory (tdt-600m: the 8198-row output matrix) are streamed per pass through a
    // staging tile by 8-byte cp.async in the layout of the resident weights, so that their products read shared memory
    // like everyone else (the previous per-fragment ld.global made P3 57 % of a 600m decode step); the copy of pass i+1
    // is started as soon as the products of pass i have read the tile and overlaps the partial-sum exchange.
    bf16 *wstage = w_p + (size_t)ge.JPC * RSP + (p.out_in_smem ? (size_t)ge.OPC * RSJ : 0);
    auto stage_rows_async = [&](bf16 *dst, const bf16 *src, int rows, int K, int k0, int KS) {
        const int RS = 2 * (KS + 4), n8 = KS / 4;
        const uint32_t d0 = smem_addr(dst);
        for (int i = tid; i < rows * n8; i += blockDim.x) {
            const int r = i / n8, pc = i - r * n8;
            const bf16 *sp = src + (size_t)r * 2 * K + k0 + pc * 4;
            const uint32_t dd = d0 + (uint32_t)(r * RS + pc * 4) * 2u;
            cp_async8(dd, sp);
            cp_async8(dd + (uint32_t)(KS + 4) * 2u, sp + K);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    for (int i = tid; i < L * 2 * ge.MU * Bpad; i += blockDim.x) csm[i] = 0.f;   // zero cell state (tdt.cpp:49-59)
    for (int b = tid; b < Bpad; b += blockDim.x) {                               // initial decode state
        s_cur[b] = 0;
        s_token[b] = (p.carry && b < p.n_utt) ? p.tok_state[b] : V - 1;
        s_tpos[b] = 0;
        s_active[b] = (b < p.n_utt && p.row_off[b + 1] > p.row_off[b]) ? 1 : 0;
        s_ntok[b] = 0;
        s_pend[b] = -1;
        if (p.max_symbols > 0) s_nsym[b] = 0;
    }
    __syncthreads();
    // Units this CTA finalises (same enumeration as the cell update in P1): pass ug, slot mi -> unit u, state slot cslot.
    auto for_my_units = [&](auto fn) {
        for (int ug = 0; ug < nU; ug += RG / 4) {
            const int nu = min(RG / 4, nU - ug), myu = (nu - rank + CL - 1) / CL;
            for (int mi = 0; mi < myu; ++mi) fn(u0 + ug + rank + CL * mi, ug / CL + mi);
        }
    };
    if (p.carry) {   // committed cell state of the previous chunk -> plane 0 (eou.cpp:22-33 initialises it to zero once)
        for (int l = 0; l < L; ++l)
            for_my_units([&](int u, int cslot) {
                for (int b = tid; b < Bpad; b += blockDim.x)
                    csm[((size_t)(l * 2 + 0) * ge.MU + cslot) * Bpad + b] = p.c_state[((size_t)l * Bpad + b) * P + u];
            });
        __syncthreads();
    }

    // h: bf16 planes [hi|lo][L][2][Bpad][P] (two state planes per utterance); z: [hi|lo][Bpad][J]
    const size_t HS = (size_t)P * Bpad;
    bf16 *hb = reinterpret_cast<bf16 *>(p.hbuf), *zb = reinterpret_cast<bf16 *>(p.z);
    const size_t h_lo = (size_t)L * 2 * HS, z_lo = (size_t)J * Bpad;
    const size_t KB = (size_t)Bpad;      // one key buffer
    const size_t PB = (size_t)G * Bpad;  // one partial buffer
    unsigned int nbar = 0;
    // deferred confidence: 1 / sum_q lsum_q * exp(lmax_q - gmax) over the per-CTA partials of `buf`
    auto finalize_conf = [&](int buf) {
        const int warp = tid >> 5, lane = tid & 31;
        for (int b = g + warp * G; b < p.n_utt; b += G * NWARP) {   // utterances owned by this CTA (b % G == g)
            const int slot = s_pend[b];
            if (slot < 0) continue;
            // all partials of this lane first (one L2 round trip), then max and sum (fixed order: q ascending per lane)
            constexpr int QMAX = 8;                                  // grids up to 256 CTAs
            float m[QMAX], sv[QMAX];
#pragma unroll
            for (int i = 0; i < QMAX; ++i) {
                const int q = lane + 32 * i;
                m[i] = q < G ? p.pl_max[buf * PB + (size_t)q * Bpad + b] : -INFINITY;
                sv[i] = q < G ? p.pl_sum[buf * PB + (size_t)q * Bpad + b] : 0.f;
            }
            float gmax = -INFINITY;
#pragma unroll
            for (int i = 0; i < QMAX; ++i) gmax = fmaxf(gmax, m[i]);
            gmax = warp_max(gmax);
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < QMAX; ++i)
                if (m[i] > -INFINITY) s += sv[i] * expf(m[i] - gmax);
            s = warp_sum(s);
            // exp(log-prob of the emitted token); without boosting the token IS the maximum: exp(0) / s
            if (lane == 0) p.t_conf[(size_t)b * p.cap + slot] = p.boost_on ? expf(s_vraw[b] - gmax) / s : 1.0f / s;
        }
    };
    auto nox = [&](int) { return static_cast<const bf16 *>(nullptr); };

    long long tacc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tprev = clock64();
    auto tick = [&](int slot) {   // phase timing of CTA 0 (debug aid, p.dbg may be null)
        const long long now = clock64();
        tacc[slot] += now - tprev;
        tprev = now;
    };
    int step = 0;
    for (;; ++step) {
        const int kb = step % 3;
        if (g == 0)   // reset the key buffer of the NEXT step (last read two barriers ago)
            for (int b = tid; b < Bpad; b += blockDim.x) {
                p.key_lab[((step + 1) % 3) * KB + b] = 0ull;
                p.key_dur[((step + 1) % 3) * KB + b] = 0ull;
            }
        // ================= P1: LSTM layers =================
        // W_ih of an upper layer that is not resident is streamed through the staging tile (free until P3): with two
        // layers its copy starts here and lands under layer 0's products; deeper stacks stage right before use.
        const bool staged_ih = !p.wih_in_smem && L > 1 && p.wstage_rows >= nU * 4 && nU <= RG / 4 && KSP == KSJ;
        if (staged_ih && L == 2) stage_rows_async(wstage, p.Wih[1] + (size_t)u0 * 4 * 2 * P, nU * 4, P, kP0, KSP);
        for (int l = 0; l < L; ++l) {
            if (staged_ih && L > 2 && l >= 1) stage_rows_async(wstage, p.Wih[l] + (size_t)u0 * 4 * 2 * P, nU * 4, P, kP0, KSP);
            for (int bc = 0; bc < Bpad; bc += BCH)
                for (int ug = 0; ug < nU; ug += RG / 4) {               // passes of <= 20 units (one for the 110m)
                    const int nu = min(RG / 4, nU - ug), R = nu * 4;
                    const int myu = (nu - rank + CL - 1) / CL;          // units ug + rank, ug + rank + CL, ...
                    // rows I finalise: unit-local index ul = rank + CL * (i >> 2), gate i & 3
                    auto myrow = [&](int i) { return ((rank + CL * (i >> 2)) << 2) | (i & 3); };
                    auto pre_g = [&](int r, int b) {
                        const int u = u0 + ug + (r >> 2), gt = r & 3;
                        return (l == 0) ? p.G0[(size_t)s_token[b] * 4 * P + gt * P + u] : p.bih[l][gt * P + u];
                    };
                    auto fin_g = [&](int i, int, int b, float v, float e) { gsm[i * BCH + (b - bc)] = v + e; };
                    auto xprev = [&](int b) { return hb + ((size_t)(l * 2 + s_cur[b])) * HS + (size_t)b * P + kP0; };
                    const bf16 *W1 = w_hh[l] + (size_t)ug * 4 * RSP;
                    if (l == 0) {
                        cluster_pass_n<CL, true, true>(W1, RSP, KSP + 4, xprev, nullptr, 0, 0, nox, h_lo, R, KSP, Bpad, bc, xs, red,
                                                       myu * 4, myrow, pre_g, fin_g);
                    } else {   // + input part W_ih . h'_{l-1}(new), accumulated into the same partial sums
                        auto xh = [&](int b) { return hb + ((size_t)((l - 1) * 2 + (1 - s_cur[b]))) * HS + (size_t)b * P + kP0; };
                        if (p.wih_in_smem)
                            cluster_pass_n<CL, true, true>(W1, RSP, KSP + 4, xprev, w_ih[l] + (size_t)ug * 4 * RSP, RSP, KSP + 4, xh, h_lo, R,
                                                           KSP, Bpad, bc, xs, red, myu * 4, myrow, pre_g, fin_g);
                        else if (staged_ih)          // (one pass: nU <= 20 units; the tile holds rows [u0*4, u1*4) of W_ih[l])
                            cluster_pass_n<CL, true, true>(W1, RSP, KSP + 4, xprev, wstage, RSP, KSP + 4, xh, h_lo, R,
                                                           KSP, Bpad, bc, xs, red, myu * 4, myrow, pre_g, fin_g);
                        else
                            cluster_pass_n<CL, true, false>(W1, RSP, KSP + 4, xprev, w_ih[l] + (size_t)ug * 4 * 2 * P, 2 * P, P, xh, h_lo, R,
                                                            KSP, Bpad, bc, xs, red, myu * 4, myrow, pre_g, fin_g);
                    }
                    // cell update of my units (tdt/lstm.cpp:11-29); state index = (pass, my unit slot)
                    for (int idx = tid; idx < myu * BCH; idx += blockDim.x) {
                        const int mi = idx / BCH, bb = idx % BCH, b = bc + bb;
                        if (b >= Bpad) continue;
                        const int u = u0 + ug + rank + CL * mi;
                        const int cslot = ug / CL + mi;                // < MU
                        const float gi = gsm[(mi * 4 + 0) * BCH + bb], gf = gsm[(mi * 4 + 1) * BCH + bb];
                        const float gg = gsm[(mi * 4 + 2) * BCH + bb], go = gsm[(mi * 4 + 3) * BCH + bb];
                        const int cu = s_cur[b];
                        const float c_old = csm[((size_t)(l * 2 + cu) * ge.MU + cslot) * Bpad + b];
                        const float c_new = sigmoidf_(gf) * c_old + sigmoidf_(gi) * tanhf(gg);
                        const float h_new = sigmoidf_(go) * tanhf(c_new);
                        csm[((size_t)(l * 2 + 1 - cu) * ge.MU + cslot) * Bpad + b] = c_new;
                        store_split(hb, hb + h_lo, ((size_t)(l * 2 + 1 - cu)) * HS + (size_t)b * P + u, h_new);
                    }
                    if (ug + RG / 4 < nU || bc + BCH < Bpad) cluster_sync_all();   // partial buffers are reused by the next pass
                }
            tick(0);
            grid_arrive(p.bar);
            if (l == L - 1) {
                // confidences of the tokens emitted in the previous step: their partials were complete at
                // that step's last barrier, so this sits in the shadow of the barrier wait
                if (step > 0) finalize_conf((step - 1) % 3);
                __syncthreads();
                for (int b = tid; b < Bpad; b += blockDim.x) s_pend[b] = -1;
            }
            grid_wait(p.bar, ++nbar);
            tick(1);
        }
        // ================= P2: joint hidden z = relu(EP[t] + Wp . h') =================
        for (int bc = 0; bc < Bpad; bc += BCH)
            for (int rg = j0; rg < j1; rg += RG) {
                const int R = min(RG, j1 - rg);
                const int nmy = (R - rank + CL - 1) / CL;               // rows rank, rank + CL, ...
                cluster_pass_n<CL, true, true>(
                    w_p + (size_t)(rg - j0) * RSP, RSP, KSP + 4,
                    [&](int b) { return hb + ((size_t)((L - 1) * 2 + (1 - s_cur[b]))) * HS + (size_t)b * P + kP0; }, nullptr, 0, 0, nox,
                    h_lo, R, KSP, Bpad, bc, xs, red, nmy, [&](int i) { return rank + CL * i; },
                    [&](int r, int b) {
                        if (b >= p.n_utt) return 0.f;
                        const int T = p.row_off[b + 1] - p.row_off[b];
                        if (T <= 0) return 0.f;           // (carried decode: a stream without frames this chunk)
                        const int t = min(s_tpos[b], T - 1);
                        return p.EP[(size_t)(p.row_off[b] + t) * J + rg + r];
                    },
                    [&](int, int r, int b, float v, float e) { store_split(zb, zb + z_lo, (size_t)b * J + rg + r, fmaxf(v + e, 0.f)); });
                if (rg + RG < j1 || bc + BCH < Bpad) cluster_sync_all();
            }
        tick(2);
        grid_arrive(p.bar);
        grid_wait(p.bar, ++nbar);
        tick(3);
        // ================= P3: logits -> per-CTA partials + global arg-max keys =================
        const bool staged_out = !p.out_in_smem && p.wstage_rows >= 16;
        const int RGo = staged_out ? p.wstage_rows : RG;                 // rows per pass of the output matrix
        for (int bc = 0; bc < Bpad; bc += BCH) {
            float lmax = -INFINITY, lsum = 0.f, dmax = -INFINITY;
            int lidx = 0x7fffffff, didx = 0x7fffffff;
            float kmax = -INFINITY;                       // phrase boosting: arg-max key on the BOOSTED logits,
            int kidx = 0x7fffffff;                        // (lmax, lsum) stay raw for the softmax denominator
            const int BW = (V + 31) >> 5;
            if (staged_out && o1 > o0) stage_rows_async(wstage, p.Wout + (size_t)o0 * 2 * J, min(RGo, o1 - o0), J, kJ0, KSJ);
            for (int rg = o0; rg < o1; rg += RGo) {
                const int R = min(RGo, o1 - rg);
                const int nmy = (R - rank + CL - 1) / CL;
                auto xz = [&](int b) { return zb + (size_t)b * J + kJ0; };
                auto myrow = [&](int i) { return rank + CL * i; };
                auto pb = [&](int r, int) { return p.bout[rg + r]; };
                auto fl = [&](int i, int, int b, float v, float e) { gsm[i * BCH + (b - bc)] = v + e; };
                const bool first_pass = rg == o0;          // z is staged once per (phase, utterance chunk): no pass overwrites xs in P3
                if (p.out_in_smem) {
                    cluster_pass_n<CL, true, true>(w_o + (size_t)(rg - o0) * RSO, RSO, LOO, xz, nullptr, 0, 0, nox, z_lo, R, KSJ, Bpad, bc, xs,
                                                   red, nmy, myrow, pb, fl, NoPost(), first_pass);
                } else if (staged_out) {
                    // (the x staging inside the pass waits for ALL outstanding cp.async groups: this tile included)
                    auto next_tile = [&]() {
                        const int rn = rg + RGo;
                        __syncthreads();                  // every warp has finished reading the tile
                        if (rn < o1) stage_rows_async(wstage, p.Wout + (size_t)rn * 2 * J, min(RGo, o1 - rn), J, kJ0, KSJ);
                    };
                    cluster_pass_n<CL, true, true>(wstage, RSJ, KSJ + 4, xz, nullptr, 0, 0, nox, z_lo, R, KSJ, Bpad, bc, xs, red, nmy, myrow, pb, fl,
                                                   next_tile, first_pass);
                } else {
                    cluster_pass_n<CL, false, true>(w_o + (size_t)(rg - o0) * RSO, RSO, LOO, xz, nullptr, 0, 0, nox, z_lo, R, KSJ, Bpad, bc, xs,
                                                    red, nmy, myrow, pb, fl);
                }
                if (tid < BCH) {
                    for (int i = 0; i < nmy; ++i) {
                        const float v = gsm[i * BCH + tid];
                        const int n = rg + rank + CL * i;
                        if (n < V) {
                            if (v > lmax) {
                                lsum = lsum * expf(lmax - v) + 1.f;
                                lmax = v;
                                lidx = n;
                            } else {
                                lsum += expf(v - lmax);
                            }
                            if (p.boost_on && bc + tid < Bpad) {
                                const float vb = v + (((p.boost_bits[(size_t)(bc + tid) * BW + (n >> 5)] >> (n & 31)) & 1u) ? p.boost : 0.0f);
                                if (vb > kmax) {         // rows ascend within a CTA: strict '>' keeps the first maximum
                                    kmax = vb;
                                    kidx = n;
                                }
                            }
                        } else if (v > dmax) {
                            dmax = v;
                            didx = n - V;
                        }
                    }
                }
                __syncthreads();
                if (rg + RGo < o1 || bc + BCH < Bpad) cluster_sync_all();
            }
            if (tid < BCH && bc + tid < Bpad) {
                const int b = bc + tid;
                p.pl_max[kb * PB + (size_t)g * Bpad + b] = lmax;
                p.pl_sum[kb * PB + (size_t)g * Bpad + b] = lsum;
                if (b < p.n_utt && s_active[b]) {
                    if (p.boost_on) {
                        if (kmax > -INFINITY) atomicMax(&p.key_lab[kb * KB + b], pack_key(kmax, kidx));
                    } else if (lmax > -INFINITY) {
                        atomicMax(&p.key_lab[kb * KB + b], pack_key(lmax, lidx));
                    }
                    if (dmax > -INFINITY) atomicMax(&p.key_dur[kb * KB + b], pack_key(dmax, didx));
                }
            }
        }
        tick(4);
        grid_arrive(p.bar);
        grid_wait(p.bar, ++nbar);
        tick(5);
        // ================= P4 (replicated in every CTA): state update =================
        int any = 0;
        for (int b = tid; b < p.n_utt; b += blockDim.x) {
            if (!s_active[b]) continue;
            float lmax, dmax;
            int lidx, didx;
            unpack_key(p.key_lab[kb * KB + b], lmax, lidx);
            unpack_key(p.key_dur[kb * KB + b], dmax, didx);
            const int T = p.row_off[b + 1] - p.row_off[b];
            // (RNNT: no duration key; skip = 0 gives its rule below: blank t += 1, symbol end = start = t, stay)
            const bool rnnt = p.max_symbols > 0;   // (read from the parameter here: no register held across the step)
            const int skip = rnnt ? 0 : (didx < p.n_dur) ? p.durations[didx] : 1;
            int t = s_tpos[b];
            bool act = true;
            if (lidx == V - 1) {                 // blank: LSTM state reverts (cur unchanged)
                t += max(skip, 1);
                if (rnnt) s_nsym[b] = 0;
            } else {
                const int n = s_ntok[b];
                if (n < p.cap && (b % G) == g) { // the owner CTA writes the token; confidence follows
                    int32_t *row = p.tok + (size_t)b * (1 + p.cap);
                    row[1 + n] = lidx;
                    const int base = p.carry ? p.frame_base[b] : 0;
                    p.t_start[(size_t)b * p.cap + n] = base + t;
                    p.t_end[(size_t)b * p.cap + n] = p.carry ? base + t + max(skip, 1) - 1 : min(t + max(skip, 1) - 1, T - 1);
                    row[0] = n + 1;
                }
                if (n < p.cap) s_pend[b] = n;
                if (p.boost_on && (b % G) == g) {
                    // raw logit of the emitted token (its key carries the boosted value), then ContextTrie::advance
                    // (phrase_boost.cpp:53-66) and the bitmap of the next step's boosted tokens (:40-51)
                    const int BW = (V + 31) >> 5;
                    uint32_t *bits = p.boost_bits + (size_t)b * BW;
                    s_vraw[b] = ((bits[lidx >> 5] >> (lidx & 31)) & 1u) ? lmax - p.boost : lmax;
                    int32_t *act = p.trie_active + (size_t)b * 64;
                    const int na = p.trie_nact[b];
                    int32_t nxt[64];
                    int nn = 1;
                    nxt[0] = 0;
                    for (int a = 0; a < na; ++a) {
                        const int node = act[a];
                        for (int e2 = p.trie.first[node]; e2 < p.trie.first[node + 1]; ++e2)
                            if (p.trie.tok[e2] == lidx) {
                                const int ch = p.trie.child[e2];
                                bool dup = false;
                                for (int q = 0; q < nn; ++q) dup |= nxt[q] == ch;
                                if (!dup && nn < 64) nxt[nn++] = ch;
                            }
                    }
                    for (int w = 0; w < BW; ++w) bits[w] = 0u;
                    for (int q = 0; q < nn; ++q) {
                        act[q] = nxt[q];
                        for (int e2 = p.trie.first[nxt[q]]; e2 < p.trie.first[nxt[q] + 1]; ++e2) {
                            const int tk = p.trie.tok[e2];
                            if (tk >= 0 && tk < V) bits[tk >> 5] |= 1u << (tk & 31);
                        }
                    }
                    p.trie_nact[b] = nn;
                }
                s_ntok[b] = n + 1;
                s_token[b] = lidx;
                s_cur[b] = 1 - s_cur[b];         // commit the new LSTM state
                t += skip;
                if (rnnt) {                      // rnnt.cpp:82-106: the loop over max_symbols ends, the frame loop moves on
                    const int ns = s_nsym[b] + 1;
                    if (ns >= p.max_symbols) t += 1;
                    s_nsym[b] = ns >= p.max_symbols ? 0 : ns;
                }
                if (n + 1 >= p.cap && !(rnnt && t >= T)) {   // (RNNT: a full buffer at the last frame is not a truncation)
                    act = false;
                    if ((b % G) == g) p.overflow[b] = 1;
                }
            }
            s_tpos[b] = t;
            if (t >= T) act = false;
            s_active[b] = act ? 1 : 0;
            any |= act ? 1 : 0;
        }
        any = __syncthreads_or(any);
        tick(6);
        if (!any || step + 1 >= p.max_steps) break;
    }
    if (p.dbg && g == 0 && tid == 0) {
        for (int i = 0; i < 7; ++i) p.dbg[i] = tacc[i];
        p.dbg[7] = step + 1;
    }
    // confidences of the last step's tokens (all partials were visible at that step's last barrier)
    finalize_conf(step % 3);
    if (p.carry) {
        // Hand the committed state to the next chunk: cell state of my units, h of my units into plane 0, last token.
        // (Every CTA left the loop at the same step, after the step's last grid barrier: nobody reads h any more.)
        for (int l = 0; l < L; ++l)
            for_my_units([&](int u, int cslot) {
                for (int b = tid; b < Bpad; b += blockDim.x) {
                    const int cu = s_cur[b];
                    p.c_state[((size_t)l * Bpad + b) * P + u] = csm[((size_t)(l * 2 + cu) * ge.MU + cslot) * Bpad + b];
                    if (cu == 1) {
                        const size_t src = ((size_t)(l * 2 + 1)) * HS + (size_t)b * P + u, dst = ((size_t)(l * 2 + 0)) * HS + (size_t)b * P + u;
                        hb[dst] = hb[src];
                        hb[h_lo + dst] = hb[h_lo + src];
                    }
                }
            });
        for (int b = g + tid * G; b < p.n_utt; b += G * blockDim.x) p.tok_state[b] = s_token[b];
    }
    cluster_sync_all();              // nobody leaves while a peer may still read its partial sums
}

__global__ void tdt_init_kernel(TdtParams p) {
    pdl_wait();
    pdl_trigger();
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < GBAR * GBAR_STRIDE) p.bar[b] = 0u;
    if (b < 3 * p.Bpad) {
        p.key_lab[b] = 0ull;
        p.key_dur[b] = 0ull;
    }
    if (b < p.n_utt) {
        p.tok[(size_t)b * (1 + p.cap)] = 0;
        p.overflow[b] = 0;
        if (p.boost_on) {     // ContextTrie: only the root is active; its children are the boosted tokens of the first step
            const int BW = (p.V + 31) >> 5;
            uint32_t *bits = p.boost_bits + (size_t)b * BW;
            for (int w = 0; w < BW; ++w) bits[w] = 0u;
            for (int e = p.trie.first[0]; e < p.trie.first[1]; ++e) {
                const int tk = p.trie.tok[e];
                if (tk >= 0 && tk < p.V) bits[tk >> 5] |= 1u << (tk & 31);
            }
            p.trie_active[(size_t)b * 64] = 0;
            p.trie_nact[b] = 1;
        }
    }
}

// fp32 rows [rows][K] -> pre-split rows [rows][2 K] = [hi: K][lo: K] bf16
__global__ void tdt_split_rows_kernel(const float *__restrict__ src, int rows, int K, bf16 *__restrict__ dst) {
    pdl_wait();
    pdl_trigger();
    const size_t n = (size_t)rows * K;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / K;
        const int k = (int)(i - r * K);
        const float v = src[i];
        const bf16 h = __float2bfloat16_rn(v);
        dst[r * 2 * K + k] = h;
        dst[r * 2 * K + K + k] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
}

// Shared memory of one CTA (bytes) for `n_clusters` clusters of CL; decides what stays in shared memory.
size_t tdt_smem_bytes(const TdtParams &p, int n_clusters, int CL, bool *out_in_smem, bool *wih_in_smem, int *lstm_floats, int *wstage_rows) {
    const TdtGeom ge = tdt_geom(p.P, p.J, p.V + p.D, n_clusters, CL);
    const size_t budget = 225 * 1024 / sizeof(float);
    const int KSmax = ge.KSP > ge.KSJ ? ge.KSP : ge.KSJ;
    const int xrows = p.Bpad < BCH ? p.Bpad : BCH;      // the x staging planes hold min(64, Bpad) utterance rows
    size_t fixed = (size_t)RG * RLD + (size_t)MYMAX * BCH + (size_t)2 * xrows * (KSmax + 8) / 2 + (size_t)p.L * 2 * ge.MU * p.Bpad +
                   (p.max_symbols > 0 ? 8 : 7) * (size_t)p.Bpad;
    // a staged weight row = [hi KS+4][lo KS+4] bf16 = KS + 4 floats
    const size_t hh = (size_t)p.L * ge.UPC * 4 * (ge.KSP + 4), ih = (size_t)(p.L - 1) * ge.UPC * 4 * (ge.KSP + 4);
    const size_t wp = (size_t)ge.JPC * (ge.KSP + 4), wo = (size_t)ge.OPC * (ge.KSJ + 4);
    size_t total = fixed + hh + wp;                 // always resident
    *wih_in_smem = (ih == 0) || (total + ih <= budget);
    *lstm_floats = (int)(hh + (*wih_in_smem ? ih : 0));
    *out_in_smem = total + (*wih_in_smem ? ih : 0) + wo <= budget;
    *wstage_rows = 0;
    if (*out_in_smem) {
        total += (*wih_in_smem ? ih : 0) + wo;
    } else {
        // Large vocabulary (tdt-600m: 8198 output rows): the output matrix is streamed every step, so the staging tile
        // comes first -- 80 rows per pass cost a third of the passes that 16 rows do, and each pass has a fixed cost of
        // ~9k cycles (x staging, cluster barrier, DSMEM exchange).  W_ih of the upper layers stays resident only if it still
        // fits; otherwise it is streamed through the same tile (P1 uses the tile before P3 needs it).
        const size_t left = budget > total ? budget - total : 0;
        int rows = (int)(left / (size_t)(ge.KSJ + 4));
        rows = rows >= 80 ? 80 : (rows >= 64 ? 64 : (rows >= 48 ? 48 : (rows >= 32 ? 32 : (rows >= 16 ? 16 : 0))));
        *wstage_rows = rows;
        total += (size_t)rows * (ge.KSJ + 4);
        *wih_in_smem = (ih == 0) || (total + ih <= budget);
        *lstm_floats = (int)(hh + (*wih_in_smem ? ih : 0));
        if (*wih_in_smem) total += ih;
    }
    return total * sizeof(float);
}

template <int CL>
cudaError_t launch_cl(TdtParams p, int num_sms, cudaStream_t st, bool *fits) {
    *fits = false;
    if (p.P % (16 * CL) || p.J % (16 * CL)) return cudaSuccess;
    // upper bound on clusters; the occupancy query below says how many can be co-resident
    int nc = num_sms / CL;
    if (nc * CL > 256) nc = 256 / CL;                // finalize_conf reads <= 8 partials per lane
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeCooperative;
    attr[1].val.cooperative = 1;
    cfg.blockDim = dim3(NTHR);
    cfg.stream = st;
    cfg.attrs = attr;
    cfg.numAttrs = 2;
    cudaError_t err;
    for (int iter = 0; iter < 2; ++iter) {
        bool out_in_smem, wih_in_smem;
        int lstm_floats, wstage_rows;
        const size_t smem = tdt_smem_bytes(p, nc, CL, &out_in_smem, &wih_in_smem, &lstm_floats, &wstage_rows);
        if (smem > 227 * 1024) return cudaSuccess;
        err = cudaFuncSetAttribute(tdt_decode_kernel<CL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) { cudaGetLastError(); return cudaSuccess; }
        cfg.gridDim = dim3(nc * CL);
        cfg.dynamicSmemBytes = smem;
        int max_clusters = 0;
        err = cudaOccupancyMaxActiveClusters(&max_clusters, tdt_decode_kernel<CL>, &cfg);
        if (err != cudaSuccess) { cudaGetLastError(); return cudaSuccess; }
        if (max_clusters >= nc) {
            p.out_in_smem = out_in_smem ? 1 : 0;
            p.wih_in_smem = wih_in_smem ? 1 : 0;
            p.smem_lstm_floats = lstm_floats;
            p.wstage_rows = getenv("PK_TDT_NO_STAGE") ? 0 : wstage_rows;
            *fits = true;
            tdt_init_kernel<<<((3 * p.Bpad > GBAR * GBAR_STRIDE ? 3 * p.Bpad : GBAR * GBAR_STRIDE) + 127) / 128, 128, 0, st>>>(p);
            return cudaLaunchKernelEx(&cfg, tdt_decode_kernel<CL>, p);
        }
        if (max_clusters < 1) return cudaSuccess;
        nc = max_clusters;                           // retry with what fits (geometry and smem change with nc)
    }
    return cudaSuccess;
}

// Co-resident cluster counts are a property of the device and the kernel's footprint: decide once
// which cluster size to use (prefer 4 when it keeps >= 3/4 of the SMs busy).
int g_tdt_cl = 0;

}  // namespace

void tdt_pass_profile(long long *out8, bool reset) {
    if (out8) cudaMemcpyFromSymbol(out8, g_pass_clk, 8 * sizeof(long long));
    if (reset) {
        long long z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        cudaMemcpyToSymbol(g_pass_clk, z, sizeof(z));
    }
}

void launch_tdt_split_rows(const float *src, int rows, int K, bf16 *dst, cudaStream_t st) {
    tdt_split_rows_kernel<<<256, 256, 0, st>>>(src, rows, K, dst);
}

cudaError_t launch_tdt_decode(TdtParams p, int num_sms, cudaStream_t st) {
    bool fits = false;
    cudaError_t err;
    if (g_tdt_cl == 0) {
        g_tdt_cl = 4;
        if (const char *ev = getenv("PK_TDT_CLUSTER")) g_tdt_cl = atoi(ev) == 2 ? 2 : 4;
    }
    if (g_tdt_cl == 4) {
        err = launch_cl<4>(p, num_sms, st, &fits);
        if (fits) return err;
        g_tdt_cl = 2;
    }
    err = launch_cl<2>(p, num_sms, st, &fits);
    if (fits) return err;
    return cudaErrorLaunchOutOfResources;
}

}  // namespace pk
