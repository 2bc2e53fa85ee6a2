// sphsm_pass.cuh — subsystems (2), (4), (5): the two neighbour passes and the per-particle maps.
//   k_pass_a<STRICT, DENS, XSPH>    density / pressure (cpp:448-513) and XSPH intermediate velocity (cpp:669-701);
//                                   the two are independent (XSPH uses the previous step's density, Q10) and share
//                                   one sweep over the 27-cell stencil
//   k_pass_b<STRICT, MODE>          ionic cell model (cpp:575-593) + pressure/viscosity force + SPH Laplacian of Vm
//                                   (cpp:515-573) + integration, Vm clamp and walls (cpp:598-651) in one sweep;
//                                   MODE selects the fused sweep of the strict step or the force-only stage 6 of
//                                   sphsm_stage() (the only mode of the fast form: the fast step runs sphsm_pass4*.cuh);
//                                   MODE | PB_EGM also stores the electrogram source vol * L (sphsm_egm.cuh)
//   k_cell_model, k_update          the stand-alone per-particle stages for sphsm_stage()
// v1 mapping: one thread per particle over the cell-sorted SoA arrays; neighbouring threads sit in the same or
// adjacent cells, so their float4 gathers hit the same L1 lines.
#pragma once
#include "sphsm_types.cuh"

namespace sphsm {

// Poly6 (cpp:149-152).  STRICT restates the double pow(float,int) promotion; FAST evaluates in float.
template <bool STRICT>
__device__ __forceinline__ float poly6(const DevParams &p, float r2) {
    if (STRICT) {
        double x = (double)__fsub_rn(p.h2, r2);
        return (float)__dmul_rn((double)p.c_poly6, __dmul_rn(__dmul_rn(x, x), x));
    } else {
        float x = p.h2 - r2;
        return p.c_poly6 * x * x * x;
    }
}

template <bool STRICT, bool DENS, bool XSPH>
__global__ void __launch_bounds__(128) k_pass_a(const __grid_constant__ DevParams p, Arrays a, const int *__restrict__ cell_start) {
    using A = Ar<STRICT>;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const float4 pi = a.P[i];
    float4 ci = make_float4(0, 0, 0, 0);
    if (XSPH) ci = a.C[i];
    int ca, cb, cc;
    float dens = 0.0f, pvx = 0.0f, pvy = 0.0f, pvz = 0.0f;
    if (cell_coords(p, pi.x, pi.y, pi.z, ca, cb, cc)) {
        const float4 *__restrict__ P = a.P;
        const float4 *__restrict__ C = a.C;
        for_each_candidate(p, cell_start, ca, cb, cc, [&](int j) {
            const float4 pj = __ldg(P + j);
            const float dx = __fsub_rn(pi.x, pj.x), dy = __fsub_rn(pi.y, pj.y), dz = __fsub_rn(pi.z, pj.z);
            const float r2 = dist2_exact(dx, dy, dz);
            if (r2 <= p.h2) {  // Poly6 support (r2 >= 0 always holds), cpp:151
                const float w = poly6<STRICT>(p, r2);
                if (DENS) dens = A::add(dens, A::mul(pj.w, w));
                if (XSPH) {
                    const float4 cj = __ldg(C + j);
                    pvx = A::add(pvx, A::mul(A::mul(A::sub(cj.x, ci.x), w), cj.w));
                    pvy = A::add(pvy, A::mul(A::mul(A::sub(cj.y, ci.y), w), cj.w));
                    pvz = A::add(pvz, A::mul(A::mul(A::sub(cj.z, ci.z), w), cj.w));
                }
            }
        });
    }
    if (DENS) {
        const float4 e = a.E[i];
        dens = A::add(dens, A::mul(pi.w, p.poly6_self));  // the extra self term, cpp:483 (Q1)
        float pres = A::mul(p.K, A::sub(dens, p.rho0));
        pres = A::sub(pres, A::mul(e.x, p.voltage_constant));  // cpp:491
        if (e.w > 0.0f) pres = fminf(fmaxf(pres, -p.max_pressure), p.max_pressure);
        else pres = -0.0f;  // cpp:493-503 (Q2)
        a.VEL[i].w = dens;
        a.S[i] = make_float2(pres, e.x);
        a.V[i].w = __fdiv_rn(pi.w, dens);  // np->mass / np->dens as pass B reads it, cpp:551
    }
    if (XSPH) {
        float4 *v = a.V + i;
        v->x = A::add(ci.x, A::mul(pvx, p.mix));
        v->y = A::add(ci.y, A::mul(pvy, p.mix));
        v->z = A::add(ci.z, A::mul(pvz, p.mix));
    }
}

// calculate_cell_model for one particle (cpp:579-592): Iion in double after the `1.0` literal, w in float,
// both from the OLD w.
template <bool STRICT>
__device__ __forceinline__ void cell_model(const DevParams &p, float Vm, float mass, float &Iion, float &w) {
    using A = Ar<STRICT>;
    const float u = A::div(A::sub(Vm, p.Vr), p.fh_denom);
    const float c1 = A::mul(A::mul(p.C1, u), A::sub(u, p.fh_asd));
    const double t = A::dadd(A::dmul((double)c1, A::dadd((double)u, -1.0)), (double)A::mul(p.C2, w));
    Iion = (float)A::dadd((double)Iion, A::ddiv(A::dmul((double)p.dt, t), (double)mass));
    w = A::add(w, A::div(A::mul(A::mul(p.dt, p.C3), A::sub(u, A::mul(p.C4, w))), mass));
}

// Update_Properties for one particle (cpp:602-649)
template <bool STRICT>
__device__ __forceinline__ void integrate(const DevParams &p, bool fixed, float mass, float ivx, float ivy, float ivz, float ax, float ay,
                                          float az, float inter_vm, float &x, float &y, float &z, float &vx, float &vy, float &vz, float &Vm) {
    using A = Ar<STRICT>;
    if (!fixed) {
        vx = A::add(ivx, A::div(A::mul(ax, p.dt), mass));
        vy = A::add(ivy, A::div(A::mul(ay, p.dt), mass));
        vz = A::add(ivz, A::div(A::mul(az, p.dt), mass));
        x = A::add(x, A::mul(vx, p.dt));
        y = A::add(y, A::mul(vy, p.dt));
        z = A::add(z, A::mul(vz, p.dt));
    }
    Vm = A::add(Vm, A::div(A::mul(inter_vm, p.dt), mass));
    if (Vm > p.max_voltage) Vm = p.max_voltage;
    else if (Vm < -p.max_voltage) Vm = -p.max_voltage;
    if (x < 0.0f) { vx = A::mul(vx, p.wall_hit); x = 0.0f; }
    if (x >= p.world[0]) { vx = A::mul(vx, p.wall_hit); x = __fsub_rn(p.world[0], 0.0001f); }
    if (y < 0.0f) { vy = A::mul(vy, p.wall_hit); y = 0.0f; }
    if (y >= p.world[1]) { vy = A::mul(vy, p.wall_hit); y = __fsub_rn(p.world[1], 0.0001f); }
    if (z < 0.0f) { vz = A::mul(vz, p.wall_hit); z = 0.0f; }
    if (z >= p.world[2]) { vz = A::mul(vz, p.wall_hit); z = __fsub_rn(p.world[2], 0.0001f); }
    // bounds.clamp (m3Bounds.h:84-88): max(min) then min(max) with bounds [0, world]
    if (0.0f > x) x = 0.0f;
    if (p.world[0] < x) x = p.world[0];
    if (0.0f > y) y = 0.0f;
    if (p.world[1] < y) y = p.world[1];
    if (0.0f > z) z = 0.0f;
    if (p.world[2] < z) z = p.world[2];
}

constexpr int PB_FORCE_ONLY = 0;  // stage 6: writes ACC = (acc, Inter_Vm)
constexpr int PB_FUSED = 1;       // stages 5+6+7 in one sweep: cell model, force, integration; new pos -> Pout
constexpr int PB_FUSED_DIAG = 2;  // PB_FUSED + ACC for the diagnostics download
constexpr int PB_EGM = 4;         // flag on any of the above: Q = vol * L for the electrograms

template <bool STRICT, int MODE_EGM>
__global__ void __launch_bounds__(128) k_pass_b(const __grid_constant__ DevParams p, Arrays a, float4 *__restrict__ Pout,
                                                const int *__restrict__ cell_start) {
    using A = Ar<STRICT>;
    constexpr int MODE = MODE_EGM & ~PB_EGM;
    static_assert(STRICT || MODE == PB_FORCE_ONLY, "the fast step runs k_pass_b4 / k_pass_b4w; only sphsm_stage's force pass is fast here");
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    const float4 pi = a.P[i];
    const float4 vi = a.V[i];
    const float2 si = a.S[i];
    float4 e = a.E[i];
    if (MODE != PB_FORCE_ONLY) cell_model<STRICT>(p, e.x, pi.w, e.y, e.z);
    float ax = 0.0f, ay = 0.0f, az = 0.0f, L = 0.0f;
    int ca, cb, cc;
    if (cell_coords(p, pi.x, pi.y, pi.z, ca, cb, cc)) {
        const float4 *__restrict__ P = a.P;
        const float4 *__restrict__ V = a.V;
        const float2 *__restrict__ S = a.S;
        for_each_candidate(p, cell_start, ca, cb, cc, [&](int j) {
            const float4 pj = __ldg(P + j);
            const float dx = __fsub_rn(pi.x, pj.x), dy = __fsub_rn(pi.y, pj.y), dz = __fsub_rn(pi.z, pj.z);
            const float r2 = dist2_exact(dx, dy, dz);
            if (STRICT) {
                if (r2 > 1e-12f) {  // INF, SPH_SM_monodomain.h:24, cpp:546
                    const float dis = __fsqrt_rn(r2);
                    const float4 vj = __ldg(V + j);
                    const float2 sj = __ldg(S + j);
                    const float vol = vj.w;
                    float sp = 0.0f, vs = 0.0f;
                    if (dis <= p.h) {
                        const float hr = __fsub_rn(p.h, dis);
                        sp = __fmul_rn(__fmul_rn(-p.c_spiky, hr), hr);  // Spiky, cpp:157
                        vs = __fmul_rn(p.c_spiky, hr);                  // Visco, cpp:163 (Spiky constant, Q14)
                    }
                    const float fp = __fmul_rn(__fdiv_rn(__fmul_rn(vol, __fadd_rn(si.x, sj.x)), 2.0f), sp);  // cpp:553
                    ax = __fsub_rn(ax, __fdiv_rn(__fmul_rn(dx, fp), dis));
                    ay = __fsub_rn(ay, __fdiv_rn(__fmul_rn(dy, fp), dis));
                    az = __fsub_rn(az, __fdiv_rn(__fmul_rn(dz, fp), dis));
                    const float fv = __fmul_rn(__fmul_rn(vol, p.mu), vs);  // cpp:559
                    ax = __fadd_rn(ax, __fmul_rn(__fsub_rn(vj.x, vi.x), fv));
                    ay = __fadd_rn(ay, __fmul_rn(__fsub_rn(vj.y, vi.y), fv));
                    az = __fadd_rn(az, __fmul_rn(__fsub_rn(vj.z, vi.z), fv));
                    // B_spline_2, cpp:188-197 (double intermediates; `2 - q` is a float subtraction)
                    const float q = __fdiv_rn(dis, p.h);
                    float b2 = 0.0f;
                    if (q < 1.0f) b2 = (float)__dmul_rn((double)p.c_bspline, __dadd_rn(-3.0, __dmul_rn(4.5, (double)q)));
                    else if (q < 2.0f) b2 = (float)__dmul_rn((double)p.c_bspline, __dmul_rn(1.5, (double)__fsub_rn(2.0f, q)));
                    L = __fadd_rn(L, __fmul_rn(__fmul_rn(__fsub_rn(sj.y, si.y), vol), b2));  // cpp:563
                }
            } else {
                if (r2 > 1e-12f && r2 <= p.r2_q2) {  // outside 2h every term is exactly zero
                    const float4 vj = __ldg(V + j);
                    const float2 sj = __ldg(S + j);
                    const float inv_r = rsqrtf(r2);
                    const float r = r2 * inv_r;
                    const float vol = vj.w;
                    const bool inner = r2 <= p.r2_q1;
                    const float b2 = fmaf(inner ? p.bs_a1 : p.bs_a2, r, inner ? p.bs_b1 : p.bs_b2);
                    L = fmaf((sj.y - si.y) * vol, b2, L);
                    if (r2 <= p.r2_spiky) {
                        const float hr = p.h - r;
                        const float t = vol * hr * p.c_spiky;
                        const float fpr = t * (si.x + sj.x) * (0.5f * hr) * inv_r;  // = -(Force_pressure / dis)
                        const float fv = t * p.mu;
                        ax = fmaf(dx, fpr, ax);
                        ay = fmaf(dy, fpr, ay);
                        az = fmaf(dz, fpr, az);
                        ax = fmaf(vj.x - vi.x, fv, ax);
                        ay = fmaf(vj.y - vi.y, fv, ay);
                        az = fmaf(vj.z - vi.z, fv, az);
                    }
                }
            }
        });
    }
    const float dens = a.VEL[i].w;
    ax = A::div(ax, dens);  // cpp:568
    ay = A::div(ay, dens);
    az = A::div(az, dens);
    // cpp:571: Inter_Vm += (sigma/(Beta*Cm))*Inter_Vm - ((Iion - stim*dt/mass)/Cm)   (the += form, Q9)
    const float ivm = A::add(L, A::sub(A::mul(p.diff_coef, L), A::div(A::sub(e.y, A::div(A::mul(e.w, p.dt), pi.w)), p.Cm)));
    if (MODE == PB_FORCE_ONLY || MODE == PB_FUSED_DIAG) a.ACC[i] = make_float4(ax, ay, az, ivm);
    if (MODE_EGM & PB_EGM) a.Q[i] = A::mul(vi.w, L);
    if (MODE != PB_FORCE_ONLY) {
        float4 v4 = a.VEL[i];
        const bool fixed = __float_as_int(a.O[i].w) != 0;
        float x = pi.x, y = pi.y, z = pi.z;
        integrate<STRICT>(p, fixed, pi.w, vi.x, vi.y, vi.z, ax, ay, az, ivm, x, y, z, v4.x, v4.y, v4.z, e.x);
        Pout[i] = make_float4(x, y, z, pi.w);
        a.VEL[i] = v4;
        a.E[i] = e;
    }
}

template <bool STRICT>
__global__ void __launch_bounds__(256) k_cell_model(const __grid_constant__ DevParams p, Arrays a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    float4 e = a.E[i];
    cell_model<STRICT>(p, e.x, a.P[i].w, e.y, e.z);
    a.E[i] = e;
}

// stage 7 alone: reads inter_vel (V.xyz) and ACC = (acc, Inter_Vm); positions updated in place
template <bool STRICT>
__global__ void __launch_bounds__(256) k_update(const __grid_constant__ DevParams p, Arrays a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.n) return;
    float4 pi = a.P[i], v4 = a.VEL[i], e = a.E[i];
    const float4 vi = a.V[i], acc = a.ACC[i];
    const bool fixed = __float_as_int(a.O[i].w) != 0;
    integrate<STRICT>(p, fixed, pi.w, vi.x, vi.y, vi.z, acc.x, acc.y, acc.z, acc.w, pi.x, pi.y, pi.z, v4.x, v4.y, v4.z, e.x);
    a.P[i] = pi;
    a.VEL[i] = v4;
    a.E[i] = e;
}

// refresh the derived neighbour copies before a stand-alone stage (any call order stays reference-exact)
__global__ void __launch_bounds__(256) k_refresh_derived(int n, Arrays a, int vol_old, int vol_new_vm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float m = a.P[i].w, dens = a.VEL[i].w;
    if (vol_old) a.C[i].w = __fdiv_rn(m, dens);
    if (vol_new_vm) {
        const float4 p4 = a.P[i];
        const float vm = a.E[i].x;
        a.V[i].w = __fdiv_rn(m, dens);
        a.S[i].y = vm;
        a.PB[i] = make_float4(p4.x, p4.y, p4.z, vm);
    }
}

// Neighbour sets by the same traversal (sphsm_get_neighbor_sets): original indices of the members, unsorted.
__global__ void k_neighbor_sets(const __grid_constant__ DevParams p, Arrays a, const int *__restrict__ cell_start,
                                const int *__restrict__ slot_of, const int *__restrict__ query, int n_query, int kind, int cap,
                                int *counts, int *indices) {
    const int qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= n_query) return;
    const int i = slot_of[query[qi]];
    const float4 pi = a.P[i];
    int ca, cb, cc, cnt = 0;
    if (cell_coords(p, pi.x, pi.y, pi.z, ca, cb, cc)) {
        for_each_candidate(p, cell_start, ca, cb, cc, [&](int j) {
            const float4 pj = a.P[j];
            const float r2 = dist2_exact(__fsub_rn(pi.x, pj.x), __fsub_rn(pi.y, pj.y), __fsub_rn(pi.z, pj.z));
            bool in;
            if (kind == 0) in = true;
            else if (kind == 1) in = r2 <= p.h2;
            else if (kind == 2) in = r2 > 1e-12f && r2 <= p.r2_spiky;
            else in = r2 > 1e-12f && r2 <= p.r2_q2;
            if (in) {
                if (cnt < cap) indices[(size_t)qi * cap + cnt] = a.ID[j];
                cnt++;
            }
        });
    }
    counts[qi] = cnt;
}

}  // namespace sphsm
