// sphsm_sm.cuh — subsystem (3): linear and quadratic shape matching (one global cluster).
//   k_rest_pass1/2 + k_rest_finalize   rest-state sums (original centre of mass, Aqq, A9qq and their inverses);
//                                      depend only on mOriginalPos / mass / mFixed, so cached between steps
//   k_moments + k_moments_reduce       per-step sums: warp-shuffle + block reduction of double accumulators,
//                                      one partial per block, fixed-order final sum (deterministic)
//   k_sm_solve                         single thread: centres, flip guard, 3x3 Jacobi polar decomposition,
//                                      A = Apq*Aqq^-1 (or the 3x9 quadratic matrix), volume conservation, T
//   k_sm_strict                        strict mode: the reference's sequential float sums in original order
//   k_goal_cvel                        goal positions + predicted / corrected velocity per particle
// Replaces projectPositions / apply_external_forces / calculate_corrected_velocity (reference cpp:215-446,
// 653-667) and m3Matrix::{polarDecomposition,eigenDecomposition,jacobiRotate,invert,determinant} (Math3D/
// m3Matrix.cpp:3-113, m3Matrix.h:288-318), m9Matrix::invert (Math3D/m9Matrix.cpp:10-102).
#pragma once
#include "sphsm_comm.cuh"
#include "sphsm_sort.cuh"  // ordered_source (the gather applies the in-cell order)
#include "sphsm_types.cuh"

namespace sphsm {

using SA = Ar<true>;  // the O(1) matrix algebra always runs in the reference's op order, one rounding per op

#define M3(a, i, j) (a)[(i) * 3 + (j)]

__device__ inline float det3(const float *m) {  // m3Matrix.h:288-291
    float a = SA::sub(SA::mul(M3(m, 1, 1), M3(m, 2, 2)), SA::mul(M3(m, 2, 1), M3(m, 1, 2)));
    float b = SA::sub(SA::mul(M3(m, 1, 0), M3(m, 2, 2)), SA::mul(M3(m, 2, 0), M3(m, 1, 2)));
    float c = SA::sub(SA::mul(M3(m, 1, 0), M3(m, 2, 1)), SA::mul(M3(m, 1, 1), M3(m, 2, 0)));
    return SA::add(SA::sub(SA::mul(M3(m, 0, 0), a), SA::mul(M3(m, 0, 1), b)), SA::mul(M3(m, 0, 2), c));
}

__device__ inline bool invert3(float *m) {  // m3Matrix.h:293-318
    float d = det3(m);
    if (d == 0.0f) return false;
    d = SA::div(1.0f, d);
    float r[9];
    r[0] = SA::mul(SA::sub(SA::mul(M3(m, 1, 1), M3(m, 2, 2)), SA::mul(M3(m, 1, 2), M3(m, 2, 1))), d);
    r[1] = SA::mul(-SA::sub(SA::mul(M3(m, 0, 1), M3(m, 2, 2)), SA::mul(M3(m, 0, 2), M3(m, 2, 1))), d);
    r[2] = SA::mul(SA::sub(SA::mul(M3(m, 0, 1), M3(m, 1, 2)), SA::mul(M3(m, 0, 2), M3(m, 1, 1))), d);
    r[3] = SA::mul(-SA::sub(SA::mul(M3(m, 1, 0), M3(m, 2, 2)), SA::mul(M3(m, 1, 2), M3(m, 2, 0))), d);
    r[4] = SA::mul(SA::sub(SA::mul(M3(m, 0, 0), M3(m, 2, 2)), SA::mul(M3(m, 0, 2), M3(m, 2, 0))), d);
    r[5] = SA::mul(-SA::sub(SA::mul(M3(m, 0, 0), M3(m, 1, 2)), SA::mul(M3(m, 0, 2), M3(m, 1, 0))), d);
    r[6] = SA::mul(SA::sub(SA::mul(M3(m, 1, 0), M3(m, 2, 1)), SA::mul(M3(m, 1, 1), M3(m, 2, 0))), d);
    r[7] = SA::mul(-SA::sub(SA::mul(M3(m, 0, 0), M3(m, 2, 1)), SA::mul(M3(m, 0, 1), M3(m, 2, 0))), d);
    r[8] = SA::mul(SA::sub(SA::mul(M3(m, 0, 0), M3(m, 1, 1)), SA::mul(M3(m, 0, 1), M3(m, 1, 0))), d);
    for (int i = 0; i < 9; i++) m[i] = r[i];
    return true;
}

__device__ inline float dot3s(float a0, float b0, float a1, float b1, float a2, float b2) {
    return SA::add(SA::add(SA::mul(a0, b0), SA::mul(a1, b1)), SA::mul(a2, b2));
}
__device__ inline void mul3(float *out, const float *l, const float *r) {  // m3Matrix.h:223-239
    float t[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) t[i * 3 + j] = dot3s(M3(l, i, 0), M3(r, 0, j), M3(l, i, 1), M3(r, 1, j), M3(l, i, 2), M3(r, 2, j));
    for (int i = 0; i < 9; i++) out[i] = t[i];
}
__device__ inline void mul3_tl(float *out, const float *l, const float *r) {  // multiplyTransposedLeft, m3Matrix.h:241-257
    float t[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) t[i * 3 + j] = dot3s(M3(l, 0, i), M3(r, 0, j), M3(l, 1, i), M3(r, 1, j), M3(l, 2, i), M3(r, 2, j));
    for (int i = 0; i < 9; i++) out[i] = t[i];
}

// Jacobi rotation, shared by the 3x3 and 9x9 code (m3Matrix.cpp:3-35, m9Matrix.cpp:10-43).  In those two files the
// unqualified fabs/sqrt on floats are the DOUBLE C functions (SURVEY.md Q16), restated with explicit doubles.
__device__ inline void jacobi_rotate(float *A, float *R, int n, int p, int q) {
#define EL(a, i, j) (a)[(i) * n + (j)]
    float d = SA::div(SA::sub(EL(A, p, p), EL(A, q, q)), SA::mul(2.0f, EL(A, p, q)));
    float t = (float)__ddiv_rn(1.0, __dadd_rn(fabs((double)d), __dsqrt_rn((double)SA::add(SA::mul(d, d), 1.0f))));
    if (d < 0.0f) t = -t;
    float c = (float)__ddiv_rn(1.0, __dsqrt_rn((double)SA::add(SA::mul(t, t), 1.0f)));
    float s = SA::mul(t, c);
    EL(A, p, p) = SA::add(EL(A, p, p), SA::mul(t, EL(A, p, q)));
    EL(A, q, q) = SA::sub(EL(A, q, q), SA::mul(t, EL(A, p, q)));
    EL(A, p, q) = EL(A, q, p) = 0.0f;
    for (int k = 0; k < n; k++) {
        if (k != p && k != q) {
            float Akp = SA::add(SA::mul(c, EL(A, k, p)), SA::mul(s, EL(A, k, q)));
            float Akq = SA::add(SA::mul(-s, EL(A, k, p)), SA::mul(c, EL(A, k, q)));
            EL(A, k, p) = EL(A, p, k) = Akp;
            EL(A, k, q) = EL(A, q, k) = Akq;
        }
    }
    for (int k = 0; k < n; k++) {
        float Rkp = SA::add(SA::mul(c, EL(R, k, p)), SA::mul(s, EL(R, k, q)));
        float Rkq = SA::add(SA::mul(-s, EL(R, k, p)), SA::mul(c, EL(R, k, q)));
        EL(R, k, p) = Rkp;
        EL(R, k, q) = Rkq;
    }
}
// m3Matrix.cpp:38-70 / m9Matrix.cpp:47-76: at most 20 rotations; pivot = FIRST maximum |off-diagonal|; stop only
// when that maximum is <= 0.
__device__ inline void eigen_decomposition(float *A, float *R, int n) {
    for (int i = 0; i < n; i++)
        for (int j = 0; j < n; j++) EL(R, i, j) = (i == j) ? 1.0f : 0.0f;
    for (int iter = 0; iter < 20; iter++) {
        int p = 0, q = 0;
        float mx = -1.0f;
        for (int i = 0; i < n - 1; i++)
            for (int j = i + 1; j < n; j++) {
                float a = fabsf(EL(A, i, j));
                if (mx < 0.0f || a > mx) { p = i; q = j; mx = a; }
            }
        if (mx <= 0.0f) break;
        jacobi_rotate(A, R, n, p, q);
    }
#undef EL
}

__device__ inline void polar3(const float *A, float *R) {  // m3Matrix.cpp:73-113
    float ATA[9], U[9], S1[9];
    mul3_tl(ATA, A, A);
    eigen_decomposition(ATA, U, 3);
    float l[3];
    for (int k = 0; k < 3; k++) {
        float v = ATA[k * 3 + k];
        l[k] = (v <= 0.0f) ? 0.0f : (float)__ddiv_rn(1.0, __dsqrt_rn((double)v));
    }
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++)
            S1[i * 3 + j] = SA::add(SA::add(SA::mul(SA::mul(l[0], M3(U, i, 0)), M3(U, j, 0)), SA::mul(SA::mul(l[1], M3(U, i, 1)), M3(U, j, 1))),
                                    SA::mul(SA::mul(l[2], M3(U, i, 2)), M3(U, j, 2)));
    mul3(R, A, S1);
}

// m9Matrix.cpp:80-102 — the 20-rotation TRUNCATED Jacobi inverse (Q7).  A, R: 81-float scratch.
__device__ inline void invert9(float *m, float *A, float *R) {
    for (int i = 0; i < 81; i++) A[i] = m[i];
    eigen_decomposition(A, R, 9);
    float d[9];
    for (int i = 0; i < 9; i++) {
        d[i] = A[i * 9 + i];
        if (d[i] != 0.0f) d[i] = SA::div(1.0f, d[i]);
    }
    for (int i = 0; i < 9; i++)
        for (int j = 0; j < 9; j++) {
            float a = 0.0f;
            for (int k = 0; k < 9; k++) a = SA::add(a, SA::mul(SA::mul(d[k], R[i * 9 + k]), R[j * 9 + k]));
            m[i * 9 + j] = a;
        }
}

// Everything after the sums (cpp:294-322 linear, 388-427 quadratic).  Inputs: sm.cm, sm.ocm, Apq9 (3x9 row-major:
// sum m p q9^T; the linear Apq is its first three columns), sm.AqqInv / sm.A9qqInv.  Output: sm.xform, sm.R.
__device__ inline void sm_solve(const DevParams &p, SmState &sm, const float *Apq9) {
    float Apq[9];
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 3; b++) M3(Apq, a, b) = Apq9[a * 9 + b];
    if (!p.allow_flip && det3(Apq) < 0.0f) {  // cpp:294-299 (sic: r01, r11, r22)
        M3(Apq, 0, 1) = -M3(Apq, 0, 1);
        M3(Apq, 1, 1) = -M3(Apq, 1, 1);
        M3(Apq, 2, 2) = -M3(Apq, 2, 2);
    }
    float *R = sm.R;
    polar3(Apq, R);
    for (int i = 0; i < 27; i++) sm.xform[i] = 0.0f;
    if (!p.quadratic) {
        float A[9];
        // A = Aqq; A.invert() (no-op when det == 0); A.multiply(Apq, A)  cpp:307-309
        for (int i = 0; i < 9; i++) A[i] = sm.aqq_inv_ok ? sm.AqqInv[i] : sm.Aqq[i];
        mul3(A, Apq, A);
        if (p.volume) {  // cpp:311-320
            float det = det3(A);
            if (det != 0.0f) {
                det = SA::div(1.0f, SA::sqrt(fabsf(det)));
                if (det > 2.0f) det = 2.0f;
                for (int i = 0; i < 9; i++) A[i] = SA::mul(A[i], det);
            }
        }
        float omb = SA::sub(1.0f, p.beta);
        for (int i = 0; i < 9; i++) sm.xform[i] = SA::add(SA::mul(R[i], omb), SA::mul(A[i], p.beta));  // cpp:322
    } else {
        float *A9 = sm.xform;  // 3x9
        for (int i = 0; i < 3; i++)
            for (int j = 0; j < 9; j++) {  // cpp:391-403
                float a = 0.0f;
                for (int k = 0; k < 9; k++) a = SA::add(a, SA::mul(Apq9[i * 9 + k], sm.A9qqInv[k * 9 + j]));
                a = SA::mul(a, p.beta);
                if (j < 3) a = SA::add(a, SA::mul(SA::sub(1.0f, p.beta), M3(R, i, j)));
                A9[i * 9 + j] = a;
            }
#define Q(i, j) A9[(i) * 9 + (j)]
        float det = SA::add(SA::sub(SA::mul(Q(0, 0), SA::sub(SA::mul(Q(1, 1), Q(2, 2)), SA::mul(Q(2, 1), Q(1, 2)))),
                                    SA::mul(Q(0, 1), SA::sub(SA::mul(Q(1, 0), Q(2, 2)), SA::mul(Q(2, 0), Q(1, 2))))),
                            SA::mul(Q(0, 2), SA::sub(SA::mul(Q(1, 0), Q(2, 1)), SA::mul(Q(1, 1), Q(2, 0)))));  // cpp:405-408
        if (!p.allow_flip && det < 0.0f) {  // cpp:410-414
            Q(0, 1) = -Q(0, 1);
            Q(1, 1) = -Q(1, 1);
            Q(2, 2) = -Q(2, 2);
        }
#undef Q
        if (p.volume && det != 0.0f) {  // cpp:416-427: the PRE-flip determinant scales all 27 entries
            det = SA::div(1.0f, SA::sqrt(fabsf(det)));
            if (det > 2.0f) det = 2.0f;
            for (int i = 0; i < 27; i++) A9[i] = SA::mul(A9[i], det);
        }
    }
}

__device__ __forceinline__ void make_q9(float qx, float qy, float qz, float *q9) {  // cpp:348-350
    q9[0] = qx; q9[1] = qy; q9[2] = qz;
    q9[3] = __fmul_rn(qx, qx); q9[4] = __fmul_rn(qy, qy); q9[5] = __fmul_rn(qz, qz);
    q9[6] = __fmul_rn(qx, qy); q9[7] = __fmul_rn(qy, qz); q9[8] = __fmul_rn(qz, qx);
}

// ---------------------------------------------------------------------------------------------------
// block-wide sum of NACC doubles per thread -> out[NACC] (thread 0 writes).  256 threads.
template <int NACC>
__device__ __forceinline__ void block_reduce_store(double *acc, double *out) {
    __shared__ double s_part[8][NACC];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < NACC; k++) {
        double v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) s_part[warp][k] = v;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < NACC; k += blockDim.x) {
        double v = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) v += s_part[w][k];
        out[k] = v;
    }
}

// rest pass 1: [0] sum m', [1] sum m, [2..4] sum m' X      (cpp:244-251; fixed particles weigh x100 here, Q4)
// In slab mode (p.slab_on) every sum covers the particles this rank owns; the partial sums are allreduced by the host.
__global__ void __launch_bounds__(256) k_rest_pass1(const __grid_constant__ DevParams p, const float4 *__restrict__ P, const float4 *__restrict__ O,
                                                    double *partial) {
    const int n = p.n;
    double acc[5] = {0, 0, 0, 0, 0};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 q4 = P[i];
        if (p.slab_on && !slab_owned(p, q4)) continue;
        float m = q4.w;
        float4 o = O[i];
        float mf = __float_as_int(o.w) ? __fmul_rn(m, 100.0f) : m;
        acc[0] += mf; acc[1] += m;
        acc[2] += (double)__fmul_rn(o.x, mf); acc[3] += (double)__fmul_rn(o.y, mf); acc[4] += (double)__fmul_rn(o.z, mf);
    }
    block_reduce_store<5>(acc, partial + (size_t)blockIdx.x * 5);
}
// rest pass 2, blockIdx.y = row r of [ A9qq (rows 0..8) ; sum m q9 (row 9) ]: 9 doubles per block
__global__ void __launch_bounds__(256) k_rest_pass2(const __grid_constant__ DevParams p, const float4 *__restrict__ P, const float4 *__restrict__ O,
                                                    const SmState *sm, double *partial) {
    const int n = p.n;
    const int row = blockIdx.y;
    const float ox = sm->ocm[0], oy = sm->ocm[1], oz = sm->ocm[2];
    double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float4 q4 = P[i];
        if (p.slab_on && !slab_owned(p, q4)) continue;
        float m = q4.w;
        float4 o = O[i];
        float q9[9];
        make_q9(__fsub_rn(o.x, ox), __fsub_rn(o.y, oy), __fsub_rn(o.z, oz), q9);
        float w = (row < 9) ? __fmul_rn(m, q9[row]) : m;  // m * q9[j] * q9[k], cpp:385
#pragma unroll
        for (int k = 0; k < 9; k++) acc[k] += (double)__fmul_rn(w, q9[k]);
    }
    block_reduce_store<9>(acc, partial + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 9);
}
__global__ void k_rest_finalize1(const double *__restrict__ tot, SmState *sm) {
    sm->Mfix = tot[0];
    sm->M = tot[1];
    float mass = (float)tot[0];
    for (int a = 0; a < 3; a++) {
        sm->SmpX[a] = tot[2 + a];
        sm->ocm[a] = __fdiv_rn((float)tot[2 + a], mass);  // originalCm /= mass, cpp:254
    }
}
// tot: 10 rows x 9
__global__ void k_rest_finalize2(const double *__restrict__ tot, SmState *sm, float *scratch /*162*/) {
    for (int i = 0; i < 81; i++) sm->A9qq[i] = (float)tot[i];
    for (int k = 0; k < 9; k++) sm->Smq9[k] = tot[81 + k];
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 3; b++) sm->Aqq[a * 3 + b] = (float)tot[a * 9 + b];
    for (int i = 0; i < 9; i++) sm->AqqInv[i] = sm->Aqq[i];
    sm->aqq_inv_ok = invert3(sm->AqqInv) ? 1 : 0;
    for (int i = 0; i < 81; i++) sm->A9qqInv[i] = sm->A9qq[i];
    invert9(sm->A9qqInv, scratch, scratch + 81);
}

// per-step sums: [0..2] sum m' x, [3..5] sum m x, [6 + a*NB + b] sum m x_a q9_b   (NB = 3 linear, 9 quadratic)
// rng != nullptr: the slots [rng[0], rng[1]) are summed, read from device memory (slab step: the rank's owned range)
template <int NB>
__global__ void __launch_bounds__(256) k_moments(const __grid_constant__ DevParams p, const float4 *__restrict__ P, const float4 *__restrict__ O,
                                                 const SmState *sm, double *partial, const int *__restrict__ rng) {
    const int first = rng ? rng[0] : 0, n = rng ? rng[1] : p.n;
    constexpr int NACC = 6 + 3 * NB;
    const float ox = sm->ocm[0], oy = sm->ocm[1], oz = sm->ocm[2];
    double acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; k++) acc[k] = 0.0;
    auto add = [&](const float4 q4, const float4 o) {
        if (p.slab_on && !slab_owned(p, q4)) return;
        float m = q4.w;
        float mf = __float_as_int(o.w) ? __fmul_rn(m, 100.0f) : m;
        acc[0] += (double)__fmul_rn(q4.x, mf); acc[1] += (double)__fmul_rn(q4.y, mf); acc[2] += (double)__fmul_rn(q4.z, mf);
        double mx = (double)m * (double)q4.x, my = (double)m * (double)q4.y, mz = (double)m * (double)q4.z;
        acc[3] += mx; acc[4] += my; acc[5] += mz;
        float q9[9];
        make_q9(__fsub_rn(o.x, ox), __fsub_rn(o.y, oy), __fsub_rn(o.z, oz), q9);
#pragma unroll
        for (int b = 0; b < NB; b++) {
            double qb = (double)q9[b];
            acc[6 + b] += mx * qb;
            acc[6 + NB + b] += my * qb;
            acc[6 + 2 * NB + b] += mz * qb;
        }
    };
    // a thread adds its particles in the same order as ever (i, i + stride, ...), but with the records of MOM_UNROLL of them in
    // flight: at 16 warps per SM (96 registers of double accumulators) one particle per thread left the kernel at 45 % of HBM speed
    constexpr int MOM_UNROLL = 4;
    const int stride = gridDim.x * blockDim.x;
    int i = first + blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (MOM_UNROLL - 1) * stride < n; i += MOM_UNROLL * stride) {
        float4 q[MOM_UNROLL], o[MOM_UNROLL];
#pragma unroll
        for (int u = 0; u < MOM_UNROLL; u++) {
            q[u] = P[i + u * stride];
            o[u] = O[i + u * stride];
        }
#pragma unroll
        for (int u = 0; u < MOM_UNROLL; u++) add(q[u], o[u]);
    }
    for (; i < n; i += stride) add(P[i], O[i]);
    block_reduce_store<NACC>(acc, partial + (size_t)blockIdx.x * NACC);
}

// totals layout as k_moments.  One thread: cm, Apq9 = sum m x q9^T - cm (sum m q9)^T, then the reference algebra.
__global__ void k_sm_solve(const __grid_constant__ DevParams p, const double *__restrict__ tot, SmState *sm) {
    const int NB = p.quadratic ? 9 : 3;
    float mass = (float)sm->Mfix;
    double cmd[3];
    for (int a = 0; a < 3; a++) {
        sm->cm[a] = __fdiv_rn((float)tot[a], mass);  // cm /= mass, cpp:253
        cmd[a] = (double)sm->cm[a];
    }
    float Apq9[27];
    for (int a = 0; a < 3; a++)
        for (int b = 0; b < 9; b++) Apq9[a * 9 + b] = (b < NB) ? (float)(tot[6 + a * NB + b] - cmd[a] * sm->Smq9[b]) : 0.0f;
    sm_solve(p, *sm, Apq9);
}

// strict mode: the reference's own loops — sequential float accumulation in ORIGINAL particle order (cpp:244-292,
// 343-386), one thread.  slot_of[i] = sorted slot of original particle i.
__global__ void k_sm_strict(const __grid_constant__ DevParams p, const float4 *__restrict__ P, const float4 *__restrict__ O,
                            const int *__restrict__ slot_of, SmState *sm, float *scratch /*162*/) {
    const int n = p.n;
    float mass = 0.0f, cm[3] = {0, 0, 0}, ocm[3] = {0, 0, 0};
    for (int i = 0; i < n; i++) {
        int s = slot_of[i];
        float4 q4 = P[s], o = O[s];
        float m = q4.w;
        if (__float_as_int(o.w)) m = SA::mul(m, 100.0f);
        mass = SA::add(mass, m);
        cm[0] = SA::add(cm[0], SA::mul(q4.x, m)); cm[1] = SA::add(cm[1], SA::mul(q4.y, m)); cm[2] = SA::add(cm[2], SA::mul(q4.z, m));
        ocm[0] = SA::add(ocm[0], SA::mul(o.x, m)); ocm[1] = SA::add(ocm[1], SA::mul(o.y, m)); ocm[2] = SA::add(ocm[2], SA::mul(o.z, m));
    }
    for (int a = 0; a < 3; a++) { cm[a] = SA::div(cm[a], mass); ocm[a] = SA::div(ocm[a], mass); }
    float Apq9[27], Aqq[9];
    for (int i = 0; i < 27; i++) Apq9[i] = 0.0f;
    for (int i = 0; i < 9; i++) Aqq[i] = 0.0f;
    float *A9qq = sm->A9qq;
    if (p.quadratic)
        for (int i = 0; i < 81; i++) A9qq[i] = 0.0f;
    const int NB = p.quadratic ? 9 : 3;
    for (int i = 0; i < n; i++) {
        int s = slot_of[i];
        float4 q4 = P[s], o = O[s];
        float pp[3] = {SA::sub(q4.x, cm[0]), SA::sub(q4.y, cm[1]), SA::sub(q4.z, cm[2])};
        float q9[9];
        make_q9(SA::sub(o.x, ocm[0]), SA::sub(o.y, ocm[1]), SA::sub(o.z, ocm[2]), q9);
        float m = q4.w;
        for (int a = 0; a < 3; a++) {
            float mp = SA::mul(m, pp[a]);
            for (int b = 0; b < NB; b++) Apq9[a * 9 + b] = SA::add(Apq9[a * 9 + b], SA::mul(mp, q9[b]));
        }
        for (int a = 0; a < 3; a++) {
            float mq = SA::mul(m, q9[a]);
            for (int b = 0; b < 3; b++) Aqq[a * 3 + b] = SA::add(Aqq[a * 3 + b], SA::mul(mq, q9[b]));
        }
        if (p.quadratic)
            for (int j = 0; j < 9; j++) {
                float mq = SA::mul(m, q9[j]);
                for (int k = 0; k < 9; k++) A9qq[j * 9 + k] = SA::add(A9qq[j * 9 + k], SA::mul(mq, q9[k]));
            }
    }
    for (int a = 0; a < 3; a++) { sm->cm[a] = cm[a]; sm->ocm[a] = ocm[a]; }
    for (int i = 0; i < 9; i++) { sm->Aqq[i] = Aqq[i]; sm->AqqInv[i] = Aqq[i]; }
    sm->aqq_inv_ok = invert3(sm->AqqInv) ? 1 : 0;
    if (p.quadratic) {
        for (int i = 0; i < 81; i++) sm->A9qqInv[i] = A9qq[i];
        invert9(sm->A9qqInv, scratch, scratch + 81);
    }
    sm_solve(p, *sm, Apq9);
}

// goal position (cpp:324-329 / 429-444), predicted velocity (cpp:226-231), corrected velocity (cpp:661-666), and the
// neighbour volume m/dens of the PREVIOUS step's density that pass A needs (Q10) — for one particle.
// prev_goal: used instead of T*q + cm when projectPositions returned early (n <= 1, cpp:236).
template <bool STRICT>
__device__ __forceinline__ float4 goal_cvel_one(const DevParams &p, const SmState *__restrict__ sm, const float4 *__restrict__ cold_goal,
                                                const float4 *__restrict__ cold_pv, const float4 q4, const float4 v4, const float4 o,
                                                const float4 *prev_goal, float4 &goal, float4 &pv) {
    using A = Ar<STRICT>;
    const int flags = __float_as_int(o.w);
    float gx, gy, gz, px, py, pz;
    if (!flags) {
        const float qx = A::sub(o.x, sm->ocm[0]), qy = A::sub(o.y, sm->ocm[1]), qz = A::sub(o.z, sm->ocm[2]);
        const float *T = sm->xform;
        if (prev_goal) {
            gx = prev_goal->x; gy = prev_goal->y; gz = prev_goal->z;
        } else if (!p.quadratic) {
            gx = A::add(A::add(A::add(A::mul(T[0], qx), A::mul(T[1], qy)), A::mul(T[2], qz)), sm->cm[0]);
            gy = A::add(A::add(A::add(A::mul(T[3], qx), A::mul(T[4], qy)), A::mul(T[5], qz)), sm->cm[1]);
            gz = A::add(A::add(A::add(A::mul(T[6], qx), A::mul(T[7], qy)), A::mul(T[8], qz)), sm->cm[2]);
        } else {
            float g[3];
#pragma unroll
            for (int r = 0; r < 3; r++) {
                const float *t = T + r * 9;
                float acc = A::add(A::add(A::mul(t[0], qx), A::mul(t[1], qy)), A::mul(t[2], qz));
                acc = A::add(acc, A::mul(A::mul(t[3], qx), qx));
                acc = A::add(acc, A::mul(A::mul(t[4], qy), qy));
                acc = A::add(acc, A::mul(A::mul(t[5], qz), qz));
                acc = A::add(acc, A::mul(A::mul(t[6], qx), qy));
                acc = A::add(acc, A::mul(A::mul(t[7], qy), qz));
                acc = A::add(acc, A::mul(A::mul(t[8], qz), qx));
                g[r] = A::add(acc, sm->cm[r]);
            }
            gx = g[0]; gy = g[1]; gz = g[2];
        }
        px = A::add(v4.x, A::div(A::mul(p.gravity[0], p.dt), q4.w));
        py = A::add(v4.y, A::div(A::mul(p.gravity[1], p.dt), q4.w));
        pz = A::add(v4.z, A::div(A::mul(p.gravity[2], p.dt), q4.w));
    } else {
        const float4 cg = cold_goal[flags - 1], cp = cold_pv[flags - 1];
        gx = cg.x; gy = cg.y; gz = cg.z;
        px = cp.x; py = cp.y; pz = cp.z;
    }
    float4 c;
    c.x = A::add(px, A::mul(A::mul(A::sub(gx, q4.x), p.inv_dt), p.alpha));
    c.y = A::add(py, A::mul(A::mul(A::sub(gy, q4.y), p.inv_dt), p.alpha));
    c.z = A::add(pz, A::mul(A::mul(A::sub(gz, q4.z), p.inv_dt), p.alpha));
    c.w = __fdiv_rn(q4.w, v4.w);  // np->mass / np->dens with the previous step's density, cpp:696
    goal = make_float4(gx, gy, gz, 0.0f);
    pv = make_float4(px, py, pz, 0.0f);
    return c;
}

// store: bit 0 = corrected_vel (C), bit 1 = mGoalPos, bit 2 = predicted_vel — the sub-stages apply_external_forces
// (cpp:215-232) and projectPositions (cpp:234-446) store only their own output; the full stage stores all three.
template <bool STRICT, bool DIAG>
__global__ void __launch_bounds__(256) k_goal_cvel(const __grid_constant__ DevParams p, Arrays a, const SmState *__restrict__ sm, int keep_goal,
                                                   int store) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= p.n) return;
    float4 goal, pv, prev;
    if (keep_goal) prev = a.GOAL[s];
    const float4 c = goal_cvel_one<STRICT>(p, sm, a.COLD_GOAL, a.COLD_PV, a.P[s], a.VEL[s], a.O[s], keep_goal ? &prev : nullptr, goal, pv);
    if (store & 1) a.C[s] = c;
    if (DIAG) {
        if (store & 2) a.GOAL[s] = goal;
        if (store & 4) a.PV[s] = pv;
    }
}

// Fused fast path: gather the persistent state into the new slot order AND apply stage 2's per-particle map while the
// values are in registers (the shape-matching transform of this step was already solved at the end of the previous
// step from pass B's moment partials).  Saves the separate 48 B/particle re-read of k_goal_cvel.
template <bool DIAG>
__global__ void __launch_bounds__(256) k_reorder_goal(const __grid_constant__ DevParams p, const uint32_t *__restrict__ vals, Arrays src,
                                                      Arrays dst, const SmState *__restrict__ sm, const int *__restrict__ n_dev,
                                                      const uint32_t *__restrict__ skey, const int *__restrict__ cell_start, int order_cells,
                                                      uint32_t *__restrict__ vals_out) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= (n_dev ? *n_dev : p.n)) return;  // n_dev: the live count is still on its way to the host (slab step)
    uint32_t v;
    if (order_cells > 0) {  // counting sort: the cell's canonical order is applied here (ordered_source)
        v = ordered_source(vals, skey, cell_start, src.ID, order_cells, s);
        vals_out[s] = v;
    } else v = vals[s];
    const float4 p4 = src.P[v], v4 = src.VEL[v], o4 = src.O[v], e4 = src.E[v];
    dst.P[s] = p4;
    // pass B writes VEL = (vel, dens) of every particle it integrates without reading it (the old velocity is not an input of
    // cpp:605, the density travels in S); only a FIXED particle keeps its velocity (cpp:603), so only that one is carried over
    if (__float_as_int(o4.w)) dst.VEL[s] = v4;
    dst.O[s] = o4;
    dst.E[s] = e4;
    dst.ID[s] = src.ID[v];
    dst.PB[s] = make_float4(p4.x, p4.y, p4.z, e4.x);
    float4 goal, pv;
    dst.C[s] = goal_cvel_one<false>(p, sm, src.COLD_GOAL, src.COLD_PV, p4, v4, o4, nullptr, goal, pv);
    if (DIAG) {
        dst.GOAL[s] = goal;
        dst.PV[s] = pv;
    }
}

// totals[k] = sum over blocks of partial[b * nacc + k]; one block per accumulator, fixed order (deterministic)
// err != nullptr: one more block (blockIdx.x == nacc) stores the rank's error state as totals[nacc] for the moment allreduce of the
// slab step (every rank learns in the same step that some rank failed)
__global__ void __launch_bounds__(256) k_sum_partials_par(const double *__restrict__ partial, int blocks, int nacc, double *totals,
                                                          const int *__restrict__ err = nullptr) {
    __shared__ double s[256];
    const int k = blockIdx.x;
    if (k == nacc) {
        if (threadIdx.x == 0) totals[nacc] = (err[0] | err[1] | err[2]) ? 1.0 : 0.0;
        return;
    }
    double v = 0.0;
    for (int b = threadIdx.x; b < blocks; b += 256) v += partial[(size_t)b * nacc + k];
    s[threadIdx.x] = v;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) totals[k] = s[0];
}

}  // namespace sphsm
