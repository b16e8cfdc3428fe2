/* pauli_rot.cuh -- device steps of a rotation sweep on tiles staged in shared memory as re / im planes, shared by
 * k_pauli_rot (pauli_rot.cu) and the adjoint sweep of pauli_grad.cu.  T is the tile bits (amplitudes per slot = 2^T);
 * amplitude m of the planes is slot m >> T, tile coordinate m & (2^T - 1). */
#pragma once
#include "pauli.h"

#define ROT_TWO_PI 6.283185307179586

/* (re, im) * i^w */
template <typename R>
__device__ __forceinline__ void mul_iw(R &re, R &im, uint32_t w)
{
    const R r = re, i = im;
    switch (w) {
    case 0: break;
    case 1: re = -i; im = r; break;
    case 2: re = -r; im = -i; break;
    default: re = i; im = -r; break;
    }
}

/* one pairing rotation: pair (m0, m0 ^ F), F = slot flip << T | xin */
template <typename R, int T>
__device__ __forceinline__ void rot_pairs(R *sre, R *sim, const RotOp &op, uint64_t base, int ns, uint32_t tid)
{
    const uint32_t F = ((op.flags >> 1) & 3u) << T | op.xin;
    const int h = 31 - __clz(F);
    const uint32_t lowm = (1u << h) - 1, cmask = (1u << T) - 1, sp = (op.flags >> 3) & 3u, w = (op.flags >> 5) & 3u;
    const uint32_t tpar = __popcll(base & op.zout) & 1;
    const R c = (R)op.c, s = (R)op.s;
    const uint32_t npairs = (uint32_t)ns << (T - 1);
    for (uint32_t p = tid; p < npairs; p += ROT_THREADS) {
        const uint32_t m0 = ((p & ~lowm) << 1) | (p & lowm), m1 = m0 ^ F;
        const uint32_t par0 = (__popc(m0 & cmask & op.zin) + __popc((m0 >> T) & sp) + tpar) & 1;
        const uint32_t par1 = (__popc(m1 & cmask & op.zin) + __popc((m1 >> T) & sp) + tpar) & 1;
        const R a0r = sre[m0], a0i = sim[m0], a1r = sre[m1], a1i = sim[m1];
        R t1r = a1r, t1i = a1i, t0r = a0r, t0i = a0i;
        mul_iw(t1r, t1i, w);
        mul_iw(t0r, t0i, w);
        const R s1 = par1 ? -s : s, s0 = par0 ? -s : s;   /* new a_j = c a_j + s sigma_{j^x} i^w a_{j^x} */
        sre[m0] = c * a0r + s1 * t1r; sim[m0] = c * a0i + s1 * t1i;
        sre[m1] = c * a1r + s0 * t0r; sim[m1] = c * a1i + s0 * t0i;
    }
}

/* a stretch of diagonal rotations: m = slot << T | i << ROT_TB | tid */
template <typename R, int T>
__device__ __forceinline__ void rot_diag(R *sre, R *sim, const RotOp &op, const RotDiag *diag, uint64_t base, int ns, uint32_t tid)
{
    constexpr int NI = 1 << (T - ROT_TB);   /* amplitudes per thread and slot: m = tid | i << ROT_TB */
    const RotDiag *d = diag + op.d0;
    for (int slot = 0; slot < ns; slot++) {
        double C[NI];
#pragma unroll
        for (int p = 0; p < NI; p++) {   /* C[p]: signed angle sum of the rotations whose Z on the bits of i is p */
            double acc = 0.0;
            for (int k = op.poff[p]; k < op.poff[p + 1]; k++) {
                const RotDiag e = d[k];
                const int par = (__popc(tid & e.zt) + __popcll(base & e.zout) + __popc((uint32_t)slot & e.sp)) & 1;
                acc += par ? -e.theta : e.theta;
            }
            C[p] = acc;
        }
#pragma unroll
        for (int hb = 1; hb < NI; hb <<= 1)   /* angle of amplitude i = sum_p C[p] (-1)^{popc(i & p)} */
#pragma unroll
            for (int i = 0; i < NI; i++)
                if (!(i & hb)) { const double u = C[i], v = C[i + hb]; C[i] = u + v; C[i + hb] = u - v; }
#pragma unroll
        for (int i = 0; i < NI; i++) {
            double ph = 0.5 * C[i];
            ph -= ROT_TWO_PI * rint(ph * (1.0 / ROT_TWO_PI));
            R cs, sn;
            if (sizeof(R) == 4) { float fc, fs; sincosf((float)ph, &fs, &fc); cs = (R)fc; sn = (R)fs; }
            else { double dc, ds; sincos(ph, &ds, &dc); cs = (R)dc; sn = (R)ds; }
            const uint32_t m = ((uint32_t)slot << T) | ((uint32_t)i << ROT_TB) | tid;
            const R re = sre[m], im = sim[m];   /* a * exp(-i ph) */
            sre[m] = re * cs + im * sn;
            sim[m] = im * cs - re * sn;
        }
    }
}

/* stage slot `slot` of a tile group: 2^UB 16-byte units at ub | (unit offsets of bits k), into the planes */
template <typename R, int UB>
__device__ __forceinline__ void stage_tile(R *sre, R *sim, const uint4 *src, uint64_t ub, const uint64_t *uoff, int slot, uint32_t tid)
{
#pragma unroll
    for (int k = 0; k < (1 << UB) / ROT_THREADS; k++) {
        uint64_t ko = 0;
#pragma unroll
        for (int b = 0; b < UB - ROT_TB; b++) if ((k >> b) & 1) ko |= uoff[ROT_TB + b];
        const uint4 v = __ldcs(src + (ub | ko));
        const uint32_t u = ((uint32_t)slot << UB) | tid | ((uint32_t)k << ROT_TB);
        if (sizeof(R) == 4) {   /* unit { re0 re1 im0 im1 }: amplitudes 2u, 2u + 1 */
            reinterpret_cast<float2 *>(sre)[u] = make_float2(__uint_as_float(v.x), __uint_as_float(v.y));
            reinterpret_cast<float2 *>(sim)[u] = make_float2(__uint_as_float(v.z), __uint_as_float(v.w));
        } else {                /* unit { re im } */
            reinterpret_cast<uint2 *>(sre)[u] = make_uint2(v.x, v.y);
            reinterpret_cast<uint2 *>(sim)[u] = make_uint2(v.z, v.w);
        }
    }
}

/* write slot `slot` of the planes back to dst, the inverse of stage_tile */
template <typename R, int UB>
__device__ __forceinline__ void store_tile(uint4 *dst, const R *sre, const R *sim, uint64_t ub, const uint64_t *uoff, int slot, uint32_t tid)
{
#pragma unroll
    for (int k = 0; k < (1 << UB) / ROT_THREADS; k++) {
        uint64_t ko = 0;
#pragma unroll
        for (int b = 0; b < UB - ROT_TB; b++) if ((k >> b) & 1) ko |= uoff[ROT_TB + b];
        const uint32_t u = ((uint32_t)slot << UB) | tid | ((uint32_t)k << ROT_TB);
        uint4 v;
        if (sizeof(R) == 4) {
            const float2 r = reinterpret_cast<const float2 *>(sre)[u], i = reinterpret_cast<const float2 *>(sim)[u];
            v = make_uint4(__float_as_uint(r.x), __float_as_uint(r.y), __float_as_uint(i.x), __float_as_uint(i.y));
        } else {
            const uint2 r = reinterpret_cast<const uint2 *>(sre)[u], i = reinterpret_cast<const uint2 *>(sim)[u];
            v = make_uint4(r.x, r.y, i.x, i.y);
        }
        __stcs(dst + (ub | ko), v);
    }
}
