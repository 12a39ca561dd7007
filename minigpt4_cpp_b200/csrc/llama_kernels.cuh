// llama_kernels.cuh — sm_100a kernels of the LLaMA step (decode matvec family, attention, embedding gather).
//
// Numerics mirror ggml@master-31cfbb1 (SURVEY.md §A.3): activations are quantised to the weight type's
// vec_dot type (Q8_0 / Q8_1 / Q8_K / F16) and the block dot products are integer (dp4a) with F32 scaling —
// the same formulation the reference's CPU path uses, which is also the bandwidth-optimal one.  Only float
// summation order differs from the CPU path.
//
// BIT-EXACT PARITY: every float reduction here follows the canonical order the CPU oracle fixes (oracle/oracle.cpp
// "FLOAT REDUCTION ORDER"): lane l accumulates blocks l, l+32, ... in increasing order, lanes are combined with an
// xor-butterfly (16,8,4,2,1); FMAs only where written (fmaf); the file is compiled with -fmad=false.  Changing a loop
// order or a reduction here REQUIRES the same change in the oracle.
//
// The decode matvec is HBM-bound: weights are read exactly once with 128-bit non-allocating loads from the
// repacked planes; activations live in shared memory; reductions use warp shuffles.  Tensor cores are NOT
// used for N=1 on purpose (north_star).
#pragma once
#include "llama.h"

namespace mg4 {
namespace k {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

enum Epi : int { EPI_PLAIN = 0, EPI_QKV = 1, EPI_RESID = 2, EPI_SWIGLU = 3, EPI_LOGITS = 4 };
enum Act : int { ACT_Q8_0 = 0, ACT_Q8_1 = 1, ACT_Q8_K = 2, ACT_F16 = 3 };

__host__ __device__ constexpr int act_of(int wt) {
    return (wt == GG_Q4_0 || wt == GG_Q5_0 || wt == GG_Q8_0) ? ACT_Q8_0 : (wt == GG_Q4_1 || wt == GG_Q5_1) ? ACT_Q8_1
         : (wt == GG_Q4_K || wt == GG_Q5_K || wt == GG_Q6_K) ? ACT_Q8_K : ACT_F16;
}
// bytes of one staged activation vector in shared memory (16-byte aligned)
__host__ __device__ inline size_t act_bytes(int act, int cols) {
    size_t b = act == ACT_F16 ? (size_t)cols * 2
             : act == ACT_Q8_K ? (size_t)cols + (size_t)cols / 256 * 4 + (size_t)cols / 16 * 2
                               : (size_t)cols + (size_t)cols / 32 * 8;
    return (b + 15) & ~(size_t)15;
}

struct MatvecArgs {
    QMat w;
    const float *x; int x_stride;     // F32 input rows [ntok][x_stride]
    const float *norm_w;              // fused RMSNorm weight (nullable)
    unsigned char *staged;            // global scratch [ntok][act_bytes]: activations quantised ONCE per op by stage_kernel
    int ntok; int rows_per_warp; int epi; int n_valid;  // n_valid: real row count (rows may be padded to even)
    float *out; int out_stride; const float *resid;
    // EPI_QKV
    float *q_out; __half *kcache; __half *vcache; const float2 *rope; int e_local; int half_dim; int part;
    DeviceState *state;
    const __half *tab_silu;
};

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg_stream(const uint2 *p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ unsigned ldg_stream(const unsigned *p) {
    unsigned r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// CTA-wide sync of 256 threads: the stand-alone kernels below use the whole CTA (__syncthreads); the persistent decode megakernel
// (llama_mega6.cuh) syncs its first eight warps on named barrier 1 while the other warps keep streaming.
template <bool MEGA> __device__ __forceinline__ void cta_sync() {
    if (MEGA) asm volatile("bar.sync 1, 256;" ::: "memory"); else __syncthreads();
}
__device__ __forceinline__ double block_sum(double v, double *red) {  // red: >= 33 doubles of shared memory; 256 threads
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    cta_sync<false>();
    if (lane == 0) red[warp] = v;
    cta_sync<false>();
    if (warp == 0) { double t = lane < 8 ? red[lane] : 0.0; t = warp_sum(t); if (lane == 0) red[32] = t; }
    cta_sync<false>();
    return red[32];
}
__device__ __forceinline__ float block_max(float v, float *red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_max(v);
    cta_sync<false>();
    if (lane == 0) red[warp] = v;
    cta_sync<false>();
    if (warp == 0) { float t = lane < 8 ? red[lane] : -INFINITY; t = warp_max(t); if (lane == 0) red[32] = t; }
    cta_sync<false>();
    return red[32];
}
__device__ __forceinline__ float lut_f16(const __half *tab, float x) {  // ggml fp16 LUT op: in rounded to F16, out F16
    return __half2float(tab[__half_as_ushort(__float2half_rn(x))]);
}

// ---------------------------------------------------------------------------------------------
// activation staging: F32 row (optionally RMS-normalised, eps 1e-6, double accumulation like ggml_rms_norm)
// -> shared memory in the weight type's vec_dot format (quantize_row_q8_0 / q8_1 AVX2 semantics, q8_K)
// ---------------------------------------------------------------------------------------------
template <int ACT>
__device__ void stage_act(const float *__restrict__ x, const float *__restrict__ nw, int cols, unsigned char *sm, double *red) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5; constexpr int nwarps = 8, nthreads = 256;
    float scale = 1.0f;
    if (nw) {
        // canonical RMS order (oracle.cpp): 512 partials, partial p owns elements 2048k + 4p + e; 16 warp butterflies + a top
        // butterfly.  This 256-thread kernel computes partials p = tid and p = tid + 256.
        double ssa = 0.0, ssb = 0.0;
        for (int k = 0; 2048 * k < cols; ++k) {
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int ia = 2048 * k + 4 * tid + e, ib = ia + 1024;
                if (ia < cols) { const float v = x[ia]; ssa += (double)(v * v); }
                if (ib < cols) { const float v = x[ib]; ssb += (double)(v * v); }
            }
        }
        ssa = warp_sum(ssa); ssb = warp_sum(ssb);
        cta_sync<false>();
        if (lane == 0) { red[warp] = ssa; red[warp + 8] = ssb; }
        cta_sync<false>();
        if (warp == 0) { double t = lane < 16 ? red[lane] : 0.0; t = warp_sum(t); if (lane == 0) red[32] = t; }
        cta_sync<false>();
        const double tot = red[32];
        const float mean = (float)(tot / (double)cols);
        scale = 1.0f / sqrtf(mean + 1e-6f);
    }
    if (ACT == ACT_F16) {
        __half *h = (__half *)sm;
        for (int i = tid; i < cols; i += nthreads) { float v = x[i]; if (nw) v = (v * scale) * nw[i]; h[i] = __float2half_rn(v); }
    } else if (ACT == ACT_Q8_K) {
        int8_t *qs = (int8_t *)sm; float *d = (float *)(sm + cols); int16_t *bs = (int16_t *)(sm + cols + cols / 256 * 4);
        for (int sb = warp; sb < cols / 256; sb += nwarps) {
            float v[8]; float amax = 0.f, mx = 0.f; int mi = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int i = sb * 256 + lane * 8 + j; float t = x[i]; if (nw) t = (t * scale) * nw[i]; v[j] = t;
                const float a = fabsf(t); if (a > amax) { amax = a; mx = t; mi = lane * 8 + j; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {  // first-index arg-max of |x| (strict > in the sequential reference)
                const float oa = __shfl_xor_sync(0xffffffffu, amax, o), om = __shfl_xor_sync(0xffffffffu, mx, o);
                const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
                if (oa > amax || (oa == amax && oi < mi)) { amax = oa; mx = om; mi = oi; }
            }
            int q[8]; int s = 0;
            const float iscale = amax != 0.f ? -128.f / mx : 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j) { int t = __float2int_rn(iscale * v[j]); t = t < 127 ? t : 127; q[j] = t; s += t; }
            if (amax == 0.f) { s = 0; }
            unsigned w0 = (q[0] & 0xff) | ((q[1] & 0xff) << 8) | ((q[2] & 0xff) << 16) | ((unsigned)(q[3] & 0xff) << 24);
            unsigned w1 = (q[4] & 0xff) | ((q[5] & 0xff) << 8) | ((q[6] & 0xff) << 16) | ((unsigned)(q[7] & 0xff) << 24);
            *(uint2 *)(qs + sb * 256 + lane * 8) = make_uint2(w0, w1);
            const int s2 = s + __shfl_xor_sync(0xffffffffu, s, 1);
            if ((lane & 1) == 0) bs[sb * 16 + (lane >> 1)] = (int16_t)s2;
            if (lane == 0) d[sb] = amax != 0.f ? 1.0f / iscale : 0.f;
        }
    } else {
        int8_t *qs = (int8_t *)sm; float *d = (float *)(sm + cols); float *s = d + cols / 32;
        for (int b = warp; b < cols / 32; b += nwarps) {
            const int i = b * 32 + lane;
            float v = x[i]; if (nw) v = (v * scale) * nw[i];
            const float amax = warp_max(fabsf(v));
            const float dd = amax / 127.f;
            const float id = amax != 0.0f ? 127.f / amax : 0.0f;
            const int q = __float2int_rn(v * id);
            qs[(lane < 16 ? 0 : cols / 2) + b * 16 + (lane & 15)] = (int8_t)q;  // split planes: first/second 16 of each block
            const int sum = warp_sum(q);
            if (lane == 0) {
                if (ACT == ACT_Q8_0) { d[b] = __half2float(__float2half_rn(dd)); s[b] = 0.f; }
                else { d[b] = dd; s[b] = dd * (float)sum; }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// per-codec partial dot products of TWO adjacent rows against NT staged activation vectors.
// Each returns lane-partial sums; the caller finishes with warp_sum.
// ---------------------------------------------------------------------------------------------
// Q4_0 / Q4_1, row-packed layout: row = [nb x 16 B nibbles][nb x {half d | half2 d,m}]; row0/row1 may point to global
// memory (stand-alone kernels) or to a shared-memory ring slot filled by cp.async.bulk (megakernel).
template <int NT, bool SMEM>
__device__ __forceinline__ void dot2_q4(const unsigned char *row0, const unsigned char *row1, int nb, int cols, bool q41, const unsigned char *act, size_t astride, int lane, float (&res)[2][NT]) {
    const uint4 *qs0 = (const uint4 *)row0, *qs1 = (const uint4 *)row1;
    const unsigned char *sc0 = row0 + (size_t)nb * 16, *sc1 = row1 + (size_t)nb * 16;
    float accd[2][NT], accm[2][NT];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) { accd[r][t] = 0.f; accm[r][t] = 0.f; }
    for (int b0 = 0; b0 < nb; b0 += 128) {
        uint4 q[2][4]; float dv[2][4], mv[2][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int b = b0 + i * 32 + lane;
            if (b < nb) {
                if (SMEM) { q[0][i] = qs0[b]; q[1][i] = qs1[b]; } else { q[0][i] = ldg_stream(qs0 + b); q[1][i] = ldg_stream(qs1 + b); }
                if (q41) {
                    const unsigned a0 = SMEM ? ((const unsigned *)sc0)[b] : ldg_stream((const unsigned *)sc0 + b), a1 = SMEM ? ((const unsigned *)sc1)[b] : ldg_stream((const unsigned *)sc1 + b);
                    const float2 f0 = __half22float2(*(const __half2 *)&a0), f1 = __half22float2(*(const __half2 *)&a1);
                    dv[0][i] = f0.x; mv[0][i] = f0.y; dv[1][i] = f1.x; mv[1][i] = f1.y;
                } else {
                    dv[0][i] = __half2float(((const __half *)sc0)[b]); dv[1][i] = __half2float(((const __half *)sc1)[b]);
                    mv[0][i] = 0.f; mv[1][i] = 0.f;
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int b = b0 + i * 32 + lane;
            if (b < nb) {
                int lo[2][4], hi[2][4];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    const unsigned wv[4] = {q[r][i].x, q[r][i].y, q[r][i].z, q[r][i].w};
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        lo[r][j] = (int)(wv[j] & 0x0F0F0F0Fu); hi[r][j] = (int)((wv[j] >> 4) & 0x0F0F0F0Fu);
                        if (!q41) { lo[r][j] = (int)__vsub4((unsigned)lo[r][j], 0x08080808u); hi[r][j] = (int)__vsub4((unsigned)hi[r][j], 0x08080808u); }
                    }
                }
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const unsigned char *at = act + t * astride;
                    const int4 a0 = *(const int4 *)(at + b * 16), a1 = *(const int4 *)(at + cols / 2 + b * 16);
                    const float ad = ((const float *)(at + cols))[b];
                    const float as = ((const float *)(at + cols))[nb + b];
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        int sdot = __dp4a(lo[r][0], a0.x, 0); sdot = __dp4a(lo[r][1], a0.y, sdot); sdot = __dp4a(lo[r][2], a0.z, sdot); sdot = __dp4a(lo[r][3], a0.w, sdot);
                        sdot = __dp4a(hi[r][0], a1.x, sdot); sdot = __dp4a(hi[r][1], a1.y, sdot); sdot = __dp4a(hi[r][2], a1.z, sdot); sdot = __dp4a(hi[r][3], a1.w, sdot);
                        if (q41) { accd[r][t] = fmaf(dv[r][i] * ad, (float)sdot, accd[r][t]); accm[r][t] = fmaf(mv[r][i], as, accm[r][t]); }
                        else { accd[r][t] += ((float)sdot * dv[r][i]) * ad; }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) res[r][t] = warp_sum(accd[r][t]) + warp_sum(accm[r][t]);
}

__device__ __forceinline__ void scale_min_k4(const unsigned char *q, int j, int &sc, int &mn) {
    if (j < 4) { sc = q[j] & 63; mn = q[j + 4] & 63; }
    else { sc = (q[j + 4] & 0xF) | ((q[j - 4] >> 6) << 4); mn = (q[j + 4] >> 4) | ((q[j] >> 6) << 4); }
}

template <int NT>
__device__ __forceinline__ void dot2_q5k(const QMat &w, int r0, const unsigned char *act, size_t astride, int lane, float (&res)[2][NT]) {
    const int nsb = w.cols / 256;
    const int sub = lane >> 3, j = (lane & 7) >> 1, hf = lane & 1;  // 8 lanes per super-block: (j, half)
    float accd[2][NT], accm[2][NT];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) { accd[r][t] = 0.f; accm[r][t] = 0.f; }
    for (int sb0 = 0; sb0 < nsb; sb0 += 4) {
        const int sb = sb0 + sub;
        if (sb < nsb) {
            uint4 qs[2], qh[2], sc[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {   // row-packed: [nsb x 128 B qs][nsb x 32 B qh][nsb x 16 B {scales[12], d, dmin}]
                const unsigned char *row = (const unsigned char *)w.p0 + (size_t)(r0 + r) * (size_t)w.row_bytes;
                qs[r] = ldg_stream((const uint4 *)row + sb * 8 + j * 2 + hf);
                qh[r] = ldg_stream((const uint4 *)(row + (size_t)nsb * 128) + sb * 2 + hf);
                sc[r] = ldg_stream((const uint4 *)(row + (size_t)nsb * 160) + sb);
            }
            int lo[2][4], hi[2][4]; float dd[2], dmin[2]; int sca[2], scb[2], mna[2], mnb[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const unsigned qv[4] = {qs[r].x, qs[r].y, qs[r].z, qs[r].w}, hv[4] = {qh[r].x, qh[r].y, qh[r].z, qh[r].w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    lo[r][i] = (int)((qv[i] & 0x0F0F0F0Fu) | (((hv[i] >> (2 * j)) & 0x01010101u) << 4));
                    hi[r][i] = (int)(((qv[i] >> 4) & 0x0F0F0F0Fu) | (((hv[i] >> (2 * j + 1)) & 0x01010101u) << 4));
                }
                const unsigned char *sp = (const unsigned char *)&sc[r];
                scale_min_k4(sp, 2 * j, sca[r], mna[r]); scale_min_k4(sp, 2 * j + 1, scb[r], mnb[r]);
                const float2 f = __half22float2(*(const __half2 *)&sc[r].w);
                dd[r] = f.x; dmin[r] = f.y;
            }
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const unsigned char *at = act + t * astride;
                const int4 a0 = *(const int4 *)(at + sb * 256 + 64 * j + 16 * hf);
                const int4 a1 = *(const int4 *)(at + sb * 256 + 64 * j + 32 + 16 * hf);
                const float d8 = ((const float *)(at + w.cols))[sb];
                const int16_t *bs = (const int16_t *)(at + w.cols + nsb * 4) + sb * 16;
                const int b0 = bs[4 * j + hf], b1 = bs[4 * j + 2 + hf];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    int s0 = __dp4a(lo[r][0], a0.x, 0); s0 = __dp4a(lo[r][1], a0.y, s0); s0 = __dp4a(lo[r][2], a0.z, s0); s0 = __dp4a(lo[r][3], a0.w, s0);
                    int s1 = __dp4a(hi[r][0], a1.x, 0); s1 = __dp4a(hi[r][1], a1.y, s1); s1 = __dp4a(hi[r][2], a1.z, s1); s1 = __dp4a(hi[r][3], a1.w, s1);
                    accd[r][t] += (dd[r] * d8) * (float)(sca[r] * s0 + scb[r] * s1);
                    accm[r][t] += (dmin[r] * d8) * (float)(mna[r] * b0 + mnb[r] * b1);
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) res[r][t] = warp_sum(accd[r][t]) - warp_sum(accm[r][t]);
}

// Q5_0 / Q5_1 / Q8_0 (reached by loading a ggjt file that holds such tensors; tests/test_block_types_gpu.py).  Device layout
// (planes, [row][block]): p0 = payload (Q8_0: 32 int8; Q5_x: 16 B of nibbles), p1 = Q5_x fifth bits (32-bit qh), p2 = half d (Q5_0, Q8_0) or
// half2 {d, m} (Q5_1).  Canonical order = oracle.cpp dot_canon_q5_0 / q5_1 / q8_0: lane l owns blocks l, l+32, ...; xor butterflies.
__device__ __forceinline__ unsigned spread4_to_bit4(unsigned n) { return ((n * 0x00204081u) & 0x01010101u) << 4; }  // bit i of n (< 16) -> bit 4 of byte i
template <int WT, int NT>
__device__ __forceinline__ void dot2_b32(const QMat &w, int r0, const unsigned char *act, size_t astride, int lane, float (&res)[2][NT]) {
    constexpr bool Q8 = WT == GG_Q8_0, Q51 = WT == GG_Q5_1;
    const int nb = w.cols / 32, cols = w.cols;
    float accd[2][NT], accm[2][NT];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) { accd[r][t] = 0.f; accm[r][t] = 0.f; }
    for (int b = lane; b < nb; b += 32) {
        int lo[2][4], hi[2][4]; float dv[2], mv[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const size_t o = (size_t)(r0 + r) * nb + b;
            if (Q8) {
                const uint4 q0 = ldg_stream((const uint4 *)w.p0 + o * 2), q1 = ldg_stream((const uint4 *)w.p0 + o * 2 + 1);
                lo[r][0] = (int)q0.x; lo[r][1] = (int)q0.y; lo[r][2] = (int)q0.z; lo[r][3] = (int)q0.w;
                hi[r][0] = (int)q1.x; hi[r][1] = (int)q1.y; hi[r][2] = (int)q1.z; hi[r][3] = (int)q1.w;
            } else {
                const uint4 q = ldg_stream((const uint4 *)w.p0 + o);
                const unsigned qh = ldg_stream((const unsigned *)w.p1 + o);
                const unsigned wv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    unsigned l5 = (wv[k] & 0x0F0F0F0Fu) | spread4_to_bit4((qh >> (4 * k)) & 0xFu);
                    unsigned h5 = ((wv[k] >> 4) & 0x0F0F0F0Fu) | spread4_to_bit4((qh >> (16 + 4 * k)) & 0xFu);
                    if (!Q51) { l5 = __vsub4(l5, 0x10101010u); h5 = __vsub4(h5, 0x10101010u); }
                    lo[r][k] = (int)l5; hi[r][k] = (int)h5;
                }
            }
            if (Q51) { const unsigned a = ldg_stream((const unsigned *)w.p2 + o); const float2 f = __half22float2(*(const __half2 *)&a); dv[r] = f.x; mv[r] = f.y; }
            else { dv[r] = __half2float(((const __half *)w.p2)[o]); mv[r] = 0.f; }
        }
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            const unsigned char *at = act + t * astride;
            const int4 a0 = *(const int4 *)(at + b * 16), a1 = *(const int4 *)(at + cols / 2 + b * 16);
            const float ad = ((const float *)(at + cols))[b];
            const float as = ((const float *)(at + cols))[nb + b];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                int sdot = __dp4a(lo[r][0], a0.x, 0); sdot = __dp4a(lo[r][1], a0.y, sdot); sdot = __dp4a(lo[r][2], a0.z, sdot); sdot = __dp4a(lo[r][3], a0.w, sdot);
                sdot = __dp4a(hi[r][0], a1.x, sdot); sdot = __dp4a(hi[r][1], a1.y, sdot); sdot = __dp4a(hi[r][2], a1.z, sdot); sdot = __dp4a(hi[r][3], a1.w, sdot);
                if (Q51) { accd[r][t] = fmaf(dv[r] * ad, (float)sdot, accd[r][t]); accm[r][t] = fmaf(mv[r], as, accm[r][t]); }
                else { accd[r][t] += ((float)sdot * dv[r]) * ad; }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) res[r][t] = warp_sum(accd[r][t]) + warp_sum(accm[r][t]);
}

// Q4_K (reached by loading a ggjt file that holds Q4_K tensors; tests/test_block_types_gpu.py): Q5_K without the fifth bits;
// device layout p0 = qs (128 B / super-block), p2 = {scales[12], d, dmin}; canonical order = oracle.cpp dot_canon_q4_K
template <int NT>
__device__ __forceinline__ void dot2_q4k(const QMat &w, int r0, const unsigned char *act, size_t astride, int lane, float (&res)[2][NT]) {
    const int nsb = w.cols / 256;
    const int sub = lane >> 3, j = (lane & 7) >> 1, hf = lane & 1;  // 8 lanes per super-block: (j, half)
    float accd[2][NT], accm[2][NT];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) { accd[r][t] = 0.f; accm[r][t] = 0.f; }
    for (int sb0 = 0; sb0 < nsb; sb0 += 4) {
        const int sb = sb0 + sub;
        if (sb < nsb) {
            uint4 qs[2], sc[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const size_t o = (size_t)(r0 + r) * nsb + sb;
                qs[r] = ldg_stream((const uint4 *)w.p0 + o * 8 + j * 2 + hf);
                sc[r] = ldg_stream((const uint4 *)w.p2 + o);
            }
            int lo[2][4], hi[2][4]; float dd[2], dmin[2]; int sca[2], scb[2], mna[2], mnb[2];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const unsigned qv[4] = {qs[r].x, qs[r].y, qs[r].z, qs[r].w};
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    lo[r][i] = (int)(qv[i] & 0x0F0F0F0Fu);
                    hi[r][i] = (int)((qv[i] >> 4) & 0x0F0F0F0Fu);
                }
                const unsigned char *sp = (const unsigned char *)&sc[r];
                scale_min_k4(sp, 2 * j, sca[r], mna[r]); scale_min_k4(sp, 2 * j + 1, scb[r], mnb[r]);
                const float2 f = __half22float2(*(const __half2 *)&sc[r].w);
                dd[r] = f.x; dmin[r] = f.y;
            }
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const unsigned char *at = act + t * astride;
                const int4 a0 = *(const int4 *)(at + sb * 256 + 64 * j + 16 * hf);
                const int4 a1 = *(const int4 *)(at + sb * 256 + 64 * j + 32 + 16 * hf);
                const float d8 = ((const float *)(at + w.cols))[sb];
                const int16_t *bs = (const int16_t *)(at + w.cols + nsb * 4) + sb * 16;
                const int b0 = bs[4 * j + hf], b1 = bs[4 * j + 2 + hf];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    int s0 = __dp4a(lo[r][0], a0.x, 0); s0 = __dp4a(lo[r][1], a0.y, s0); s0 = __dp4a(lo[r][2], a0.z, s0); s0 = __dp4a(lo[r][3], a0.w, s0);
                    int s1 = __dp4a(hi[r][0], a1.x, 0); s1 = __dp4a(hi[r][1], a1.y, s1); s1 = __dp4a(hi[r][2], a1.z, s1); s1 = __dp4a(hi[r][3], a1.w, s1);
                    accd[r][t] += (dd[r] * d8) * (float)(sca[r] * s0 + scb[r] * s1);
                    accm[r][t] += (dmin[r] * d8) * (float)(mna[r] * b0 + mnb[r] * b1);
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) res[r][t] = warp_sum(accd[r][t]) - warp_sum(accm[r][t]);
}

template <int NT>
__device__ __forceinline__ void dot2_q6k(const QMat &w, int r0, const unsigned char *act, size_t astride, int lane, float (&res)[2][NT]) {
    const int nsb = w.cols / 256;
    const int sub = lane >> 3, n = (lane & 7) >> 2, u = lane & 3;  // 8 lanes per super-block: (n, u)
    float acc[2][NT];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) acc[r][t] = 0.f;
    for (int sb0 = 0; sb0 < nsb; sb0 += 4) {
        const int sb = sb0 + sub;
        if (sb < nsb) {
            int v[2][4][2]; float dd[2]; int sc[2][4];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const size_t o = (size_t)(r0 + r) * nsb + sb;
                const uint2 la = ldg_stream((const uint2 *)((const unsigned char *)w.p0 + o * 128 + 64 * n + 8 * u));
                const uint2 lb = ldg_stream((const uint2 *)((const unsigned char *)w.p0 + o * 128 + 64 * n + 32 + 8 * u));
                const uint2 hh = ldg_stream((const uint2 *)((const unsigned char *)w.p1 + o * 64 + 32 * n + 8 * u));
                const uint4 s16 = ldg_stream((const uint4 *)w.p2 + o);
                dd[r] = __half2float(((const __half *)w.p3)[o]);
                const signed char *sp = (const signed char *)&s16;
#pragma unroll
                for (int kq = 0; kq < 4; ++kq) sc[r][kq] = sp[8 * n + 2 * kq + (u >> 1)];
                const unsigned av[2] = {la.x, la.y}, bv[2] = {lb.x, lb.y}, hv[2] = {hh.x, hh.y};
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    v[r][0][i] = (int)__vsub4((av[i] & 0x0F0F0F0Fu) | ((hv[i] & 0x03030303u) << 4), 0x20202020u);
                    v[r][1][i] = (int)__vsub4((bv[i] & 0x0F0F0F0Fu) | (((hv[i] >> 2) & 0x03030303u) << 4), 0x20202020u);
                    v[r][2][i] = (int)__vsub4(((av[i] >> 4) & 0x0F0F0F0Fu) | (((hv[i] >> 4) & 0x03030303u) << 4), 0x20202020u);
                    v[r][3][i] = (int)__vsub4(((bv[i] >> 4) & 0x0F0F0F0Fu) | (((hv[i] >> 6) & 0x03030303u) << 4), 0x20202020u);
                }
            }
#pragma unroll
            for (int t = 0; t < NT; ++t) {
                const unsigned char *at = act + t * astride;
                const float d8 = ((const float *)(at + w.cols))[sb];
                int2 a[4];
#pragma unroll
                for (int kq = 0; kq < 4; ++kq) a[kq] = *(const int2 *)(at + sb * 256 + 128 * n + 32 * kq + 8 * u);
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    int isum = 0;
#pragma unroll
                    for (int kq = 0; kq < 4; ++kq) { int s = __dp4a(v[r][kq][0], a[kq].x, 0); s = __dp4a(v[r][kq][1], a[kq].y, s); isum += sc[r][kq] * s; }
                    acc[r][t] += (dd[r] * d8) * (float)isum;
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) res[r][t] = warp_sum(acc[r][t]);
}

template <int NT>
__device__ __forceinline__ void dot2_f16(const QMat &w, int r0, const unsigned char *act, size_t astride, int lane, float (&res)[2][NT]) {
    const int nv = w.cols / 8;  // uint4 = 8 halves
    const uint4 *w0 = (const uint4 *)w.p0 + (size_t)r0 * nv, *w1 = w0 + nv;
    float acc[2][NT];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) acc[r][t] = 0.f;
    for (int v0 = 0; v0 < nv; v0 += 128) {
        uint4 q[2][4];
#pragma unroll
        for (int i = 0; i < 4; ++i) { const int v = v0 + i * 32 + lane; if (v < nv) { q[0][i] = ldg_stream(w0 + v); q[1][i] = ldg_stream(w1 + v); } }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int v = v0 + i * 32 + lane;
            if (v < nv) {
#pragma unroll
                for (int t = 0; t < NT; ++t) {
                    const uint4 a = *(const uint4 *)(act + t * astride + (size_t)v * 16);
                    const __half2 *ah = (const __half2 *)&a;
#pragma unroll
                    for (int r = 0; r < 2; ++r) {
                        const __half2 *wh = (const __half2 *)&q[r][i];
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const float2 wf = __half22float2(wh[j]), af = __half22float2(ah[j]);
                            acc[r][t] = fmaf(wf.x, af.x, acc[r][t]); acc[r][t] = fmaf(wf.y, af.y, acc[r][t]);
                        }
                    }
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int t = 0; t < NT; ++t) res[r][t] = warp_sum(acc[r][t]);
}

__device__ __forceinline__ unsigned long long argmax_key(float v, int idx) {  // order-preserving; ties -> lowest index
    unsigned u = __float_as_uint(v);
    u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)idx);
}

// ---------------------------------------------------------------------------------------------
// the matvec family: y[t][r] = W[r] . act(x[t]) for t < ntok (<= NT), with a fused prologue (RMSNorm + quantise)
// and a fused epilogue (RoPE + KV append | residual add | SwiGLU | logits + arg-max)
// ---------------------------------------------------------------------------------------------
// RMSNorm + quantise the op's input rows once (grid = ntok); every matvec CTA then just copies the staged bytes
template <int ACT>
__global__ void __launch_bounds__(kThreads) stage_kernel(const float *x, int x_stride, const float *norm_w, int cols, unsigned char *out, size_t astride) {
    __shared__ double red[34];
    stage_act<ACT>(x + (size_t)blockIdx.x * x_stride, norm_w, cols, out + (size_t)blockIdx.x * astride, red);
}

template <int WT, int NT>
__global__ void __launch_bounds__(kThreads, 2) matvec_kernel(const MatvecArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    constexpr int ACT = act_of(WT);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t astride = act_bytes(ACT, a.w.cols);
    {   // activations were staged once per op by stage_kernel: copy them into shared memory
        const uint4 *src = (const uint4 *)a.staged; uint4 *dst = (uint4 *)smem;
        const int n16 = (int)((size_t)a.ntok * astride / 16);
        for (int i = threadIdx.x; i < n16; i += kThreads) dst[i] = src[i];
    }
    __syncthreads();

    const int row_begin = (blockIdx.x * kWarps + warp) * a.rows_per_warp;
    const int row_end = min(row_begin + a.rows_per_warp, a.w.rows);
    unsigned long long best = 0ull;
    for (int r0 = row_begin; r0 < row_end; r0 += 2) {
        float res[2][NT];
        if (WT == GG_Q4_1 || WT == GG_Q4_0) {
            const unsigned char *row0 = (const unsigned char *)a.w.p0 + (size_t)r0 * a.w.row_bytes;
            dot2_q4<NT, false>(row0, row0 + a.w.row_bytes, a.w.cols / 32, a.w.cols, WT == GG_Q4_1, smem, astride, lane, res);
        }
        else if (WT == GG_Q5_K) dot2_q5k<NT>(a.w, r0, smem, astride, lane, res);
        else if (WT == GG_Q4_K) dot2_q4k<NT>(a.w, r0, smem, astride, lane, res);
        else if (WT == GG_Q5_0 || WT == GG_Q5_1 || WT == GG_Q8_0) dot2_b32<WT, NT>(a.w, r0, smem, astride, lane, res);
        else if (WT == GG_Q6_K) dot2_q6k<NT>(a.w, r0, smem, astride, lane, res);
        else dot2_f16<NT>(a.w, r0, smem, astride, lane, res);

        if (a.epi == EPI_LOGITS) {
            if (lane == 0) {
                a.out[r0] = res[0][0];
                const unsigned long long k0 = argmax_key(res[0][0], r0);
                best = best > k0 ? best : k0;
                if (r0 + 1 < a.n_valid) {
                    a.out[r0 + 1] = res[1][0];
                    const unsigned long long k1 = argmax_key(res[1][0], r0 + 1);
                    best = best > k1 ? best : k1;
                }
            }
            continue;
        }
#pragma unroll
        for (int t = 0; t < NT; ++t) {
            if (lane != t || t >= a.ntok) continue;
            const float v0 = res[0][t], v1 = res[1][t];
            if (a.epi == EPI_QKV) {
                const int E = a.e_local;
                const int part = a.part >= 0 ? a.part : r0 / E, rr = a.part >= 0 ? r0 : r0 % E;
                const int pos = a.state->n_past + t;
                if (part == 2) {
                    *(__half2 *)(a.vcache + (size_t)pos * E + rr) = __floats2half2_rn(v0, v1);
                } else {
                    const float2 cs = a.rope[(size_t)pos * a.half_dim + (rr % (2 * a.half_dim)) / 2];
                    const float o0 = v0 * cs.x - v1 * cs.y, o1 = v0 * cs.y + v1 * cs.x;
                    if (part == 0) *(float2 *)(a.q_out + (size_t)t * E + rr) = make_float2(o0, o1);
                    else *(__half2 *)(a.kcache + (size_t)pos * E + rr) = __floats2half2_rn(o0, o1);
                }
            } else if (a.epi == EPI_RESID) {
                const size_t o = (size_t)t * a.out_stride + r0;
                const float2 rs = *(const float2 *)(a.resid + o);
                *(float2 *)(a.out + o) = make_float2(v0 + rs.x, v1 + rs.y);
            } else if (a.epi == EPI_SWIGLU) {  // rows are interleaved: r0 = gate(ff), r0+1 = up(ff)
                a.out[(size_t)t * a.out_stride + (r0 >> 1)] = lut_f16(a.tab_silu, v0) * v1;
            } else {
                *(float2 *)(a.out + (size_t)t * a.out_stride + r0) = make_float2(v0, v1);
            }
        }
    }
    if (a.epi == EPI_LOGITS && lane == 0 && best) atomicMax(&a.state->argmax_key, best);
}

// ---------------------------------------------------------------------------------------------
// attention over the F16 KV cache for one (head, token): ggml semantics — Q and the soft-max probabilities are
// rounded to F16, dots accumulate in F32, exp through the fp16 LUT, soft-max sum in double (SURVEY §A.3)
// grid (n_head_local, ntok), block 256, dynamic smem = n_ctx * 6 bytes
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ld_kv16(const __half *p) { return *(const uint4 *)p; }
// one (head h, token t) of decode/prefill attention; 256 threads; dyn = n_ctx * 6 bytes of shared scratch
__device__ __forceinline__ void attention_head(const float *__restrict__ q, const __half *__restrict__ kc, const __half *__restrict__ vc, float *__restrict__ out,
                                               int pos, int h, int t, int E, int n_ctx, float kq_scale, const __half *__restrict__ tab_exp,
                                               unsigned char *dyn, double *red, float *redf, __half *qh, float *part /*[16*128]*/) {
    float *sc = (float *)dyn; __half *ph = (__half *)(dyn + (size_t)n_ctx * 4);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nkv = pos + 1;
    // scores: each half-warp takes one key (16 lanes x 8 halves = 128).  Every lane fetches its own 8 q values together with
    // its first batch of K rows (one memory round trip instead of two); q is rounded to F16 as ggml does.
    {
        const int sub = lane >> 4, l16 = lane & 15;
        constexpr int B = 12;  // keys in flight per half-warp (192 keys per pass): all loads of a batch are issued before the first use
        __half2 q2[4];
        bool have_q = false;
        for (int kb0 = warp * 2; kb0 < nkv || !have_q; kb0 += 16 * B) {  // warp-uniform trip counts (both half-warps shuffle together)
            uint4 kv[B];
#pragma unroll
            for (int u = 0; u < B; ++u) {
                const int key = min(kb0 + u * 16 + sub, nkv - 1);  // clamped, unconditional: a predicated load would demote kv[] to local memory
                kv[u] = ld_kv16(kc + (size_t)key * E + h * 128 + l16 * 8);
            }
            if (!have_q) {
                const float *qp = q + (size_t)t * E + h * 128 + l16 * 8;
                float qf[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) qf[e] = qp[e];
#pragma unroll
                for (int j = 0; j < 4; ++j) q2[j] = __floats2half2_rn(qf[2 * j], qf[2 * j + 1]);
                have_q = true;
            }
#pragma unroll
            for (int u = 0; u < B; ++u) {
                if (kb0 + u * 16 >= nkv) break;
                const int key = kb0 + u * 16 + sub;
                float s = 0.f;
                if (key < nkv) {
                    const __half2 *k2 = (const __half2 *)&kv[u];
#pragma unroll
                    for (int j = 0; j < 4; ++j) { const float2 a = __half22float2(k2[j]), b = __half22float2(q2[j]); s = fmaf(a.x, b.x, s); s = fmaf(a.y, b.y, s); }
                }
#pragma unroll
                for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (key < nkv && l16 == 0) sc[key] = s * kq_scale;
            }
        }
    }
    cta_sync<false>();
    float mx = -INFINITY;
    for (int i = tid; i < nkv; i += 256) mx = fmaxf(mx, sc[i]);
    mx = block_max(mx, redf);
    double sum = 0.0;
    for (int i = tid; i < nkv; i += 256) { const float v = lut_f16(tab_exp, sc[i] - mx); sc[i] = v; sum += (double)v; }
    const double tot = block_sum(sum, red);
    const float inv = (float)(1.0 / tot);
    for (int i = tid; i < nkv; i += 256) ph[i] = __float2half_rn(sc[i] * inv);
    cta_sync<false>();
    // P.V : thread = (key group g of 16, dim octet o of 16); groups are combined by a pairwise tree (canonical order)
    {
        const int g = tid >> 4, o = tid & 15;
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = 0.f;
        constexpr int B = 12;
        int key0 = g;
        for (; key0 < nkv; key0 += 16 * B) {  // batch the V loads (192 keys per pass); the FMA order over keys stays sequential
            uint4 vv[B];
#pragma unroll
            for (int u = 0; u < B; ++u) { const int key = min(key0 + 16 * u, nkv - 1); vv[u] = ld_kv16(vc + (size_t)key * E + h * 128 + o * 8); }
#pragma unroll
            for (int u = 0; u < B; ++u) {
                const int key = key0 + 16 * u;
                if (key < nkv) {
                    const float p = __half2float(ph[key]);
                    const __half2 *v2 = (const __half2 *)&vv[u];
#pragma unroll
                    for (int j = 0; j < 4; ++j) { const float2 v = __half22float2(v2[j]); acc[2 * j] = fmaf(v.x, p, acc[2 * j]); acc[2 * j + 1] = fmaf(v.y, p, acc[2 * j + 1]); }
                }
            }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) part[g * 128 + o * 8 + e] = acc[e];
    }
    cta_sync<false>();
    if (tid < 128) {
        float v[16];
#pragma unroll
        for (int g = 0; g < 16; ++g) v[g] = part[g * 128 + tid];
#pragma unroll
        for (int st = 1; st < 16; st <<= 1)
#pragma unroll
            for (int g = 0; g < 16; g += 2 * st) v[g] = v[g] + v[g + st];
        out[(size_t)t * E + h * 128 + tid] = v[0];
    }
}
__global__ void __launch_bounds__(256) attn_kernel(const float *__restrict__ q, const __half *__restrict__ kc, const __half *__restrict__ vc,
                                                   float *__restrict__ out, const DeviceState *st, int E, int n_ctx, float kq_scale,
                                                   const __half *__restrict__ tab_exp) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ double red[34];
    __shared__ float redf[34];
    __shared__ __align__(16) __half qh[128];
    __shared__ float part[16 * 128];
    attention_head(q, kc, vc, out, st->n_past + (int)blockIdx.y, (int)blockIdx.x, (int)blockIdx.y, E, n_ctx, kq_scale, tab_exp, smem, red, redf, qh, part);
}

// ---------------------------------------------------------------------------------------------
// embedding gather (ggml_get_rows on a quantised matrix = dequantise the row), raw ggml blocks
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float dequant_elem(int type, const unsigned char *row, int i) {
    switch (type) {
        case GG_F32: return ((const float *)row)[i];
        case GG_F16: return __half2float(((const __half *)row)[i]);
        case GG_Q4_0: { const unsigned char *b = row + (i / 32) * 18; const int j = i % 32;
            const float d = __half2float(*(const __half *)b); const int qv = j < 16 ? (b[2 + j] & 0xF) : (b[2 + j - 16] >> 4); return (float)(qv - 8) * d; }
        case GG_Q4_1: { const unsigned char *b = row + (i / 32) * 20; const int j = i % 32;
            const float d = __half2float(*(const __half *)b), m = __half2float(*(const __half *)(b + 2));
            const int qv = j < 16 ? (b[4 + j] & 0xF) : (b[4 + j - 16] >> 4); return (float)qv * d + m; }
        case GG_Q5_K: { const unsigned char *b = row + (i / 256) * 176; const int e = i % 256, sub = e / 32, l = e % 32;
            const float d = __half2float(*(const __half *)b), dmin = __half2float(*(const __half *)(b + 2));
            int sc, mn; scale_min_k4(b + 4, sub, sc, mn);
            const unsigned char qb = b[48 + (sub / 2) * 32 + l]; const int nib = (sub & 1) ? (qb >> 4) : (qb & 0xF);
            const int hb = (b[16 + l] >> sub) & 1;
            return (d * (float)sc) * (float)(nib + 16 * hb) - dmin * (float)mn; }
        case GG_Q6_K: { const unsigned char *b = row + (i / 256) * 210; const int e = i % 256, n = e / 128, kq = (e % 128) / 32, l = e % 32;
            const unsigned char lb = b[64 * n + (kq & 1) * 32 + l]; const int nib = (kq >= 2) ? (lb >> 4) : (lb & 0xF);
            const int hb = (b[128 + 32 * n + l] >> (2 * kq)) & 3;
            const int qv = (nib | (hb << 4)) - 32;
            const float d = __half2float(*(const __half *)(b + 208)); const int sc = ((const signed char *)(b + 192))[8 * n + 2 * kq + l / 16];
            return d * (float)sc * (float)qv; }
    }
    return 0.f;
}
// dequant_elem plus the token-embedding types it does not cover (Q4_K, and Q5_0 / Q5_1 / Q8_0 = ggml dequantize_row_q5_0 / q5_1 / q8_0).
// The decode megakernel gathers through dequant_elem alone, so build_mega refuses files whose tok_embeddings need this.
__device__ __forceinline__ float embed_elem(int type, const unsigned char *row, int i) {
    if (type == GG_Q4_K) {
        const unsigned char *b = row + (i / 256) * 144; const int e = i % 256, sub = e / 32, l = e % 32;
        const float d = __half2float(*(const __half *)b), dmin = __half2float(*(const __half *)(b + 2));
        int sc, mn; scale_min_k4(b + 4, sub, sc, mn);
        const unsigned char qb = b[16 + (sub / 2) * 32 + l]; const int nib = (sub & 1) ? (qb >> 4) : (qb & 0xF);
        return (d * (float)sc) * (float)nib - dmin * (float)mn;
    }
    const int j = i % 32, jj = j & 15;
    if (type == GG_Q8_0) { const unsigned char *b = row + (i / 32) * 34; return (float)(int)(signed char)b[2 + j] * __half2float(*(const __half *)b); }
    if (type == GG_Q5_0 || type == GG_Q5_1) {
        const int hdr = type == GG_Q5_1 ? 4 : 2;
        const unsigned char *b = row + (i / 32) * (hdr + 20);
        const unsigned qh = b[hdr] | (b[hdr + 1] << 8) | (b[hdr + 2] << 16) | ((unsigned)b[hdr + 3] << 24);
        const int q = (j < 16 ? (b[hdr + 4 + jj] & 0xF) : (b[hdr + 4 + jj] >> 4)) | (int)(((qh >> j) & 1u) << 4);
        const float d = __half2float(*(const __half *)b);
        return type == GG_Q5_1 ? (float)q * d + __half2float(*(const __half *)(b + 2)) : (float)(q - 16) * d;
    }
    return dequant_elem(type, row, i);
}
// rows of one pass: ids[t] >= 0 = token (gather + dequantise), ids[t] < 0 = embedding row -1 - ids[t] of `emb` (the 32 image rows).
// The per-op decode graph passes DeviceState::tokens as `ids` (one row, no `emb`).
__global__ void embed_rows_kernel(int type, const unsigned char *tok, size_t row_bytes, int E, const int *ids, const float *emb, float *x) {
    const int t = blockIdx.x, id = ids[t];
    if (id >= 0) {
        const unsigned char *row = tok + (size_t)id * row_bytes;
        for (int i = threadIdx.x; i < E; i += blockDim.x) x[(size_t)t * E + i] = embed_elem(type, row, i);
    } else {
        const float *src = emb + (size_t)(-1 - id) * E;
        for (int i = threadIdx.x; i < E; i += blockDim.x) x[(size_t)t * E + i] = src[i];
    }
}
__global__ void finalize_kernel(DeviceState *st, int want_logits, int *argmax_out) {
    if (threadIdx.x == 0) {
        if (want_logits) {
            const int id = (int)(0xFFFFFFFFu - (unsigned)(st->argmax_key & 0xFFFFFFFFull));
            st->argmax_id = id; st->tokens[0] = id; st->argmax_key = 0ull;
            if (argmax_out) *argmax_out = id;
        }
        st->n_past += st->n_tok;
        st->n_tok = 1;  // default next step: single-token decode chained on the device state
    }
}
__global__ void add_kernel(float *x, const float *y, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] += y[i];
}

// ---------------------------------------------------------------------------------------------
// load-time repack kernels: raw ggml blocks (row-major) -> SoA planes.  dst_row = r * row_mul + row_off.
// src block range [blk0, blk0 + nblk) of each source row (tensor-parallel column shards).
// ---------------------------------------------------------------------------------------------
__global__ void repack_q4(const unsigned char *src, int src_nb, int blk0, int nblk, int rows, bool q41, unsigned char *dst, int dst_nb, int dst_row_bytes, int row_mul, int row_off, int dst_blk0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * nblk) return;
    const int r = (int)(i / nblk), b = (int)(i % nblk);
    const int bs = q41 ? 20 : 18, hdr = q41 ? 4 : 2;
    const unsigned char *p = src + ((size_t)r * src_nb + blk0 + b) * bs;
    unsigned char *drow = dst + (size_t)(r * row_mul + row_off) * (size_t)dst_row_bytes;
    unsigned w[4];
    for (int j = 0; j < 4; ++j) w[j] = p[hdr + 4 * j] | (p[hdr + 4 * j + 1] << 8) | (p[hdr + 4 * j + 2] << 16) | ((unsigned)p[hdr + 4 * j + 3] << 24);
    ((uint4 *)drow)[dst_blk0 + b] = make_uint4(w[0], w[1], w[2], w[3]);
    unsigned char *sc = drow + (size_t)dst_nb * 16;
    if (q41) ((unsigned *)sc)[dst_blk0 + b] = p[0] | (p[1] << 8) | (p[2] << 16) | ((unsigned)p[3] << 24);
    else ((unsigned short *)sc)[dst_blk0 + b] = (unsigned short)(p[0] | (p[1] << 8));
}
__global__ void repack_q5k(const unsigned char *src, int src_nb, int blk0, int nblk, int rows, unsigned char *dst, int dst_nb, int dst_row_bytes, int row_mul, int row_off, int dst_blk0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * nblk) return;
    const int r = (int)(i / nblk), b = (int)(i % nblk);
    const unsigned char *p = src + ((size_t)r * src_nb + blk0 + b) * 176;   // block_q5_K: d, dmin, scales[12], qh[32], qs[128]
    unsigned char *row = dst + (size_t)(r * row_mul + row_off) * (size_t)dst_row_bytes;   // row-packed: [nb x qs][nb x qh][nb x {scales, d, dmin}]
    unsigned char *qs = row + (size_t)(dst_blk0 + b) * 128, *qh = row + (size_t)dst_nb * 128 + (size_t)(dst_blk0 + b) * 32, *sc = row + (size_t)dst_nb * 160 + (size_t)(dst_blk0 + b) * 16;
    for (int j = 0; j < 128; ++j) qs[j] = p[48 + j];
    for (int j = 0; j < 32; ++j) qh[j] = p[16 + j];
    for (int j = 0; j < 12; ++j) sc[j] = p[4 + j];
    for (int j = 0; j < 4; ++j) sc[12 + j] = p[j];
}
__global__ void repack_b32(int type, const unsigned char *src, int src_nb, int blk0, int nblk, int rows, unsigned char *p0, unsigned char *p1, unsigned char *p2, int dst_nb, int row_mul, int row_off, int dst_blk0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * nblk) return;
    const int r = (int)(i / nblk), b = (int)(i % nblk);
    const size_t o = (size_t)(r * row_mul + row_off) * dst_nb + dst_blk0 + b;
    if (type == GG_Q8_0) {
        const unsigned char *p = src + ((size_t)r * src_nb + blk0 + b) * 34;  // block_q8_0: d, qs[32]
        for (int j = 0; j < 32; ++j) p0[o * 32 + j] = p[2 + j];
        p2[o * 2] = p[0]; p2[o * 2 + 1] = p[1];
    } else {
        const int hdr = type == GG_Q5_1 ? 4 : 2;                              // block_q5_0: d, qh[4], qs[16]; block_q5_1: d, m, qh[4], qs[16]
        const unsigned char *p = src + ((size_t)r * src_nb + blk0 + b) * (hdr + 20);
        for (int j = 0; j < 16; ++j) p0[o * 16 + j] = p[hdr + 4 + j];
        for (int j = 0; j < 4; ++j) p1[o * 4 + j] = p[hdr + j];
        for (int j = 0; j < hdr; ++j) p2[o * hdr + j] = p[j];
    }
}
__global__ void repack_q4k(const unsigned char *src, int src_nb, int blk0, int nblk, int rows, unsigned char *qs, unsigned char *sc, int dst_nb, int row_mul, int row_off, int dst_blk0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * nblk) return;
    const int r = (int)(i / nblk), b = (int)(i % nblk);
    const unsigned char *p = src + ((size_t)r * src_nb + blk0 + b) * 144;  // block_q4_K: d, dmin, scales[12], qs[128]
    const size_t o = (size_t)(r * row_mul + row_off) * dst_nb + dst_blk0 + b;
    for (int j = 0; j < 128; ++j) qs[o * 128 + j] = p[16 + j];
    for (int j = 0; j < 12; ++j) sc[o * 16 + j] = p[4 + j];
    for (int j = 0; j < 4; ++j) sc[o * 16 + 12 + j] = p[j];
}
__global__ void repack_q6k(const unsigned char *src, int src_nb, int blk0, int nblk, int rows, unsigned char *ql, unsigned char *qh, unsigned char *sc, unsigned short *d, int dst_nb, int row_mul, int row_off, int dst_blk0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * nblk) return;
    const int r = (int)(i / nblk), b = (int)(i % nblk);
    const unsigned char *p = src + ((size_t)r * src_nb + blk0 + b) * 210;
    const size_t o = (size_t)(r * row_mul + row_off) * dst_nb + dst_blk0 + b;
    for (int j = 0; j < 128; ++j) ql[o * 128 + j] = p[j];
    for (int j = 0; j < 64; ++j) qh[o * 64 + j] = p[128 + j];
    for (int j = 0; j < 16; ++j) sc[o * 16 + j] = p[192 + j];
    d[o] = (unsigned short)(p[208] | (p[209] << 8));
}
__global__ void repack_f16(const unsigned short *src, int src_cols, int col0, int ncols, int rows, unsigned short *dst, int dst_cols, int row_mul, int row_off, int dst_col0) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)rows * ncols) return;
    const int r = (int)(i / ncols), c = (int)(i % ncols);
    dst[(size_t)(r * row_mul + row_off) * dst_cols + dst_col0 + c] = src[(size_t)r * src_cols + col0 + c];
}

}  // namespace k
}  // namespace mg4
