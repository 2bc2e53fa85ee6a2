// sphsm_pass4w.cuh — the neighbour passes with ONE WARP PER PARTICLE, for small particle sets.
//
// The reference's own inputs (Resources/*.csv: ~5k particles, up to 75 per cell, ~136 candidates and up to 176 in-range
// neighbours per particle) put 40 blocks on 148 SMs with the thread-per-particle kernels of sphsm_pass4.cuh, each thread
// walking its candidates alone: the step is latency-bound (cfg2: pass A 159 us, pass B 266 us for 5211 particles).  Below
// ~32k particles there are more SM lanes than particles, so a warp takes one particle: its lanes stride over the candidates of
// each stencil row (coalesced), do the in-range work where it applies, and the per-lane partial sums meet in a butterfly
// reduction.  Same arithmetic per term as sphsm_pass4.cuh (exact r^2 against the same thresholds, so neighbour-set membership
// is bit-exact); only the order of the floating-point sums differs, within the fast path's 1e-5.
#pragma once
#include "sphsm_pass4.cuh"

namespace sphsm {

constexpr int PTW = 256;            // threads per block = 8 particles
constexpr int WARP_PATH_MAX = 32768;  // particles per launch up to which the warp-per-particle kernels are used

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// the nine stencil rows of the padded cell table in the reference's order; f(s, e) gets each row's slot range
template <class F>
__device__ __forceinline__ void for_each_row(const DevParams &p, const int *__restrict__ cell_start, int key0, int cc, F &&f) {
    const int ga = p.ga, gagb = p.ga * p.gb;
    const int *center = cell_start + (key0 - 1);
#pragma unroll 1
    for (int dc = -1; dc <= 1; dc++) {
        const int c2 = cc + dc;
        if (c2 < p.c_off || c2 >= p.c_off + p.gcl) continue;
#pragma unroll
        for (int k = -1; k <= 1; k++) {
            const int *q = center + dc * gagb + k * ga;
            f(__ldg(q), __ldg(q + 3));
        }
    }
}

// ---------------------------------------------------------------------------------------------------
// pass A: density / pressure + XSPH intermediate velocity (reference cpp:448-513, 669-701)
__global__ void __launch_bounds__(PTW) k_pass_a4w(const __grid_constant__ DevParams p, Arrays a, const int *__restrict__ cell_start, int count,
                                                  const int *__restrict__ rng) {
    const int w = (blockIdx.x * PTW + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= count) return;
    const int i = launch_slot(launch_range(p, rng), w);
    if (i < 0) return;
    const float4 pi = a.P[i];
    const float4 ci = a.C[i];
    const float4 *__restrict__ P = a.P;
    const float4 *__restrict__ C = a.C;
    const float h2 = p.h2, c6 = p.c_poly6;
    const float2 nxy = make_float2(-pi.x, -pi.y);
    const float nz = -pi.z;
    float dens = 0.0f, ux = 0.0f, uy = 0.0f, uz = 0.0f;
    int ca, cb, cc;
    if (cell_coords(p, pi.x, pi.y, pi.z, ca, cb, cc)) {
        for_each_row(p, cell_start, cell_key(p, ca, cb, cc), cc, [&](int s, int e) {
            for (int j = s + lane; j < e; j += 32) {
                const float4 pj = __ldg(P + j);
                const float r2 = dist2_packed(__fadd2_rn(make_float2(pj.x, pj.y), nxy), pj.z + nz);
                if (r2 <= h2) {  // Poly6 support, cpp:151
                    const float4 cj = __ldg(C + j);
                    const float x = h2 - r2;
                    const float wgt = c6 * x * x * x;  // Poly6, cpp:151 (float on the fast path)
                    dens = fmaf(pj.w, wgt, dens);
                    const float t = wgt * cj.w;
                    ux = fmaf(cj.x - ci.x, t, ux);
                    uy = fmaf(cj.y - ci.y, t, uy);
                    uz = fmaf(cj.z - ci.z, t, uz);
                }
            }
        });
    }
    dens = warp_sum(dens);
    ux = warp_sum(ux);
    uy = warp_sum(uy);
    uz = warp_sum(uz);
    if (lane == 0) pass_a_finish(p, a, i, pi, ci, dens, ux, uy, uz);
}

// ---------------------------------------------------------------------------------------------------
// pass B: ionic cell model + pressure / viscosity force + SPH Laplacian of Vm + integration and walls
// (reference cpp:575-593, 515-573, 598-651)
template <bool DIAG, bool EGM>
__global__ void __launch_bounds__(PTW) k_pass_b4w(const __grid_constant__ DevParams p, Arrays a, float4 *__restrict__ Pout,
                                                  const int *__restrict__ cell_start, uint32_t *__restrict__ next_keys,
                                                  uint32_t *__restrict__ next_rank, uint32_t *__restrict__ cell_count, int count,
                                                  const int *__restrict__ rng) {
    const int w = (blockIdx.x * PTW + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= count) return;
    const int i = launch_slot(launch_range(p, rng), w);
    if (i < 0) return;
    const float4 pi = a.P[i];
    const float4 vi = a.V[i];
    float4 e4 = a.E[i];
    const float2 si = a.S[i];  // (pres, dens)
    const bool fixed = __float_as_int(a.O[i].w) != 0;
    const float pres_i = si.x;
    const float Vm_i = e4.x;
    const float inv_mass = rcp_ftz(pi.w);
    cell_model<false>(p, e4.x, pi.w, e4.y, e4.z);

    const float4 *__restrict__ PB = a.PB;
    const float4 *__restrict__ V = a.V;
    const float2 *__restrict__ S = a.S;
    const float *__restrict__ VN = a.VN;
    const float sp2 = p.r2_spiky;
    const float a1 = p.bs_a1, b1 = p.bs_b1, a2 = p.bs_a2, b2 = p.bs_b2;
    const float hh = p.h, cs_half = 0.5f * p.c_spiky, cs_mu = p.c_spiky * p.mu;
    const float2 nxy = make_float2(-pi.x, -pi.y), nzv = make_float2(-pi.z, -Vm_i);
    float ax = 0.0f, ay = 0.0f, az = 0.0f, L = 0.0f;
    int ca, cb, cc;
    if (cell_coords(p, pi.x, pi.y, pi.z, ca, cb, cc)) {
        for_each_row(p, cell_start, cell_key(p, ca, cb, cc), cc, [&](int s, int e) {
            for (int j = s + lane; j < e; j += 32) {
                const float4 pj = __ldg(PB + j);
                const float vol = __ldg(VN + j);
                const float2 dxy = __fadd2_rn(make_float2(pj.x, pj.y), nxy);   // (x_j - x_i, y_j - y_i)
                const float2 dzv = __fadd2_rn(make_float2(pj.z, pj.w), nzv);   // (z_j - z_i, Vm_j - Vm_i)
                const float r2 = dist2_packed(dxy, dzv.x);
                if (r2 > 1e-12f) {  // INF, SPH_SM_monodomain.h:24, cpp:546
                    const float r = sqrt_ftz(r2);
                    const float bs = fminf(fmaf(a1, r, b1), fmaxf(fmaf(a2, r, b2), 0.0f));  // B_spline_2, cpp:188-197
                    L = fmaf(dzv.y * vol, bs, L);                                            // cpp:563
                    if (r2 <= sp2) {  // Spiky / Visco support r <= h, cpp:157,163
                        const float4 vj = __ldg(V + j);
                        const float pres_j = __ldg(&S[j].x);
                        const float inv_r = rsqrt_ftz(r2);
                        const float hr = fmaf(-r2, inv_r, hh);
                        const float t = vj.w * hr;
                        const float fpr = (t * hr) * (inv_r * cs_half) * (pres_i + pres_j);  // = -(Force_pressure / dis), cpp:553-554
                        const float fv = t * cs_mu;                                           // Force_viscosity, cpp:559
                        ax = fmaf(-dxy.x, fpr, ax);  // (pos_i - pos_j) * fpr
                        ay = fmaf(-dxy.y, fpr, ay);
                        az = fmaf(-dzv.x, fpr, az);
                        ax = fmaf(vj.x - vi.x, fv, ax);
                        ay = fmaf(vj.y - vi.y, fv, ay);
                        az = fmaf(vj.z - vi.z, fv, az);
                    }
                }
            }
        });
    }
    ax = warp_sum(ax);
    ay = warp_sum(ay);
    az = warp_sum(az);
    L = warp_sum(L);
    if (lane == 0) pass_b_finish<DIAG, EGM>(p, a, Pout, i, pi, vi, e4, si.y, fixed, ax, ay, az, L, inv_mass, next_keys, next_rank, cell_count);
}

}  // namespace sphsm
