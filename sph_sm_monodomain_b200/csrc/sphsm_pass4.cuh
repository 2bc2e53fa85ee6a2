// sphsm_pass4.cuh — the production (fast-path) neighbour passes, fourth generation.
//
// Two-phase scheme (phase 1 sweeps the stencil rows and lists the in-range candidates per lane
// in shared memory, phase 2 does the heavy in-range terms with every lane busy), rebuilt around the instruction counts of
// the r01_v6 ncu source pages (pass B: 2594 warp instructions per 32 particles, 59 % in the candidate-pair loop at 68
// instructions per pair, 250 in the per-row window setup, 520 in prologue + epilogue):
//   * the cell table is PADDED by one empty cell on either side of the two fast key axes (DevParams::ga/gb include the
//     border, cell_coords() returns border-relative coordinates), so the nine stencil rows of a particle always exist:
//     no clamps, no per-row range tests, and the two bounds of a row are one address apart (`row[0]`, `row[3]`);
//   * a candidate pair (j, j+1) is one address computation per array (the second load is the first + one record; the
//     gathered arrays are allocated with a tail so that j+1 == n is readable) and the odd-length tail is masked;
//   * B_spline_2 (cpp:188-197) is concave piecewise linear: min(a1 r + b1, max(a2 r + b2, 0)) replaces the two range
//     tests and four selects; r comes from one MUFU.SQRT instead of select + MUFU.RSQ + multiply;
//   * the in-range list is addressed by a running shared-memory index (store + add per append);
//   * the velocity / position side of the per-particle maps uses reciprocals of mass and density instead of IEEE
//     divisions (the voltage side keeps the reference's exact operations, see integrate_fast).
// Neighbour-set membership stays bit-exact: r^2 without FMA against the same host-computed thresholds.
#pragma once
#include "sphsm_pass.cuh"
#include "sphsm_types.cuh"

namespace sphsm {

constexpr int LIST_K = 16;  // in-range list entries per lane between drains (12 and 14 measured slower: DESIGN.md §4)

__device__ __forceinline__ float rsqrt_ftz(float x) {
    float y;
    asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ float sqrt_ftz(float x) {
    float y;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_ftz(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// a / b rounded to nearest, identical to __fdiv_rn.  A zero numerator sends the compiler's division sequence down its slow path
// (FCHK flags it; ncu r01_v8: one CALL of ~50 instructions per warp in pass B for stim * dt / mass with stim == 0, the common
// case), so that case is answered directly: +-0 / b = +-0 for b > 0.
__device__ __forceinline__ float div_rn_z(float a, float b) { return (a == 0.0f && b > 0.0f) ? a : __fdiv_rn(a, b); }

// A launch covers the slots [begin, end) minus the hole [hole_begin, hole_begin + hole_len).  On one GPU the range is in the
// parameter block; in the slab step it is read from device memory (rng = {begin, end, hole_begin, hole_len}, written by the
// sort of the same step), the grid is sized for an upper bound and the surplus threads leave.
struct Range4 {
    int begin, end, hole_begin, hole_len;
};
__device__ __forceinline__ Range4 launch_range(const DevParams &p, const int *__restrict__ rng) {
    Range4 r = {p.own_begin, p.own_end, p.hole_begin, p.hole_len};
    if (rng) {
        const int4 v = __ldg(reinterpret_cast<const int4 *>(rng));
        r.begin = v.x; r.end = v.y; r.hole_begin = v.z; r.hole_len = v.w;
    }
    return r;
}
// the k-th target slot of the launch, or -1 past its end
__device__ __forceinline__ int launch_slot(const Range4 &r, int k) {
    int i = r.begin + k;
    if (i >= r.hole_begin) i += r.hole_len;
    return i < r.end ? i : -1;
}

// The in-range list lives at 32-bit shared-memory addresses held in a register (`lofs`, bytes): ptxas re-materialises the
// base of a __shared__ array at every use (S2R + MOV + LEA per append in the first build of this file), never an address
// that depends on a global load (DevParams::zero).
__device__ __forceinline__ void list_put(unsigned addr, int v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
__device__ __forceinline__ int list_get(unsigned addr) {
    int v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
// threads per block of the generation-4 passes, measured at 8M (pass A / pass B us): 64: 484 / 689, 128: 469 / 678, 256: 497 / 692, 512: 523 / 720
constexpr int PT4 = 128;
// resident blocks per SM pass A / pass B are compiled for: 56 / 64 registers (measured in round 2 against 8 / 7: see DESIGN.md)
constexpr int A_MINB = 9, B_MINB = 8;
constexpr unsigned LSTEP = 4u * PT4;  // bytes between consecutive entries of one lane
// Likewise a gathered array's base pointer: `pinned(ptr, zero)` is ptr + 0 with the zero coming from global memory, formed
// in PTX so that neither the front end (which would fold it into the index) nor ptxas (which would re-load the kernel
// parameter with LDC at every use) can take it apart; the gathers are then one IMAD.WIDE + LDG.
template <class T>
__device__ __forceinline__ const T *pinned(const T *ptr, int zero) {
    unsigned long long out;
    asm("add.u64 %0, %1, %2;" : "=l"(out) : "l"((unsigned long long)ptr), "l"((unsigned long long)(unsigned)zero));
    return reinterpret_cast<const T *>(out);
}

// r^2 with the x and y differences formed and squared on the packed FP32 pipe (FADD2 / FMUL2 round each element like
// the scalar instructions, and negation is exact, so r^2 is bit-identical to dist2_exact of the opposite differences)
__device__ __forceinline__ float dist2_packed(float2 dxy, float dz) {
    const float2 sq = __fmul2_rn(dxy, dxy);
    return __fadd_rn(__fadd_rn(sq.x, sq.y), __fmul_rn(dz, dz));
}

struct Rows3 {
    int s[3], e[3];
};
// `mid` points at cell (ca-1, cb, c2) of the padded table; the rows cb-1, cb, cb+1 are `ga` entries apart
__device__ __forceinline__ void load_rows3(const int *__restrict__ mid, int ga, bool plane_ok, Rows3 &r) {
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const int *q = mid + (k - 1) * ga;
        r.s[k] = plane_ok ? __ldg(q) : 0;
        r.e[k] = plane_ok ? __ldg(q + 3) : 0;
    }
}

// Sweep the nine stencil rows in the reference's order (cpp:462-464).  `pair(j, two, lofs)` evaluates the candidates j and
// j+1 (`two` false: j+1 is past the row) and appends the in-range ones at s_list[lofs], lofs += PT; `one(j, lofs)` is the
// single-candidate form for rows that could overflow the list (dense meshes); `drain(lofs)` consumes the list.
template <int STEP = 2, class Pair, class One, class Drain>
__device__ __forceinline__ void sweep4(const DevParams &p, const int *__restrict__ cell_start, int ga, int gagb, int key0, unsigned lbase,
                                       unsigned &lofs, Pair &&pair, One &&one, Drain &&drain) {
    const int *center = cell_start + (key0 - 1);
    const unsigned lmax = lbase + LIST_K * LSTEP;
    // plane validity from the key alone: a lower plane exists iff key >= ga*gb, an upper one iff key + ga*gb < num_cells
    Rows3 cur, nxt;
    load_rows3(center - gagb, ga, key0 >= gagb, cur);
#pragma unroll 1
    for (int dc = -1; dc <= 1; dc++) {
        if (dc < 1) load_rows3(center + (dc + 1) * gagb, ga, dc < 0 || key0 + gagb < p.num_cells, nxt);
#pragma unroll
        for (int k = 0; k < 3; k++) {
            int j = cur.s[k];
            const int e = cur.e[k];
            if (lofs + (unsigned)(e - j) * LSTEP <= lmax) {
#pragma unroll 1
                for (; j < e; j += STEP) {
                    if constexpr (STEP == 2) pair(j, j + 1 < e, lofs);
                    else pair(j, e, lofs);  // the body masks j+1 .. j+STEP-1 against the row end itself
                }
            } else {
                if (lofs == lmax) drain(lofs);  // the unchecked path may have filled the list exactly
#pragma unroll 1
                for (; j < e; j++) {
                    one(j, lofs);
                    if (lofs == lmax) drain(lofs);
                }
            }
        }
        cur = nxt;
    }
    drain(lofs);
}

// pass A's per-particle tail, shared by every fast-path kernel: the extra self term, pressure (cpp:483-503) and the records pass B
// reads.  S = (pres, dens): pass B takes its own density from here, so VEL is neither read nor rewritten between the gather
// and pass B's final store.
__device__ __forceinline__ void pass_a_finish(const DevParams &p, const Arrays &a, int i, const float4 pi, const float4 ci, float dens, float pvx,
                                              float pvy, float pvz) {
    const float4 e4 = a.E[i];
    dens = fmaf(pi.w, p.poly6_self, dens);                           // the extra self term, cpp:483 (Q1)
    float pres = p.K * (dens - p.rho0) - e4.x * p.voltage_constant;  // cpp:486-491
    if (e4.w > 0.0f) pres = fminf(fmaxf(pres, -p.max_pressure), p.max_pressure);
    else pres = -0.0f;  // cpp:493-503 (Q2)
    a.S[i] = make_float2(pres, dens);
    const float vol = __fdiv_rn(pi.w, dens);  // np->mass / np->dens as pass B reads it, cpp:551
    a.V[i] = make_float4(fmaf(pvx, p.mix, ci.x), fmaf(pvy, p.mix, ci.y), fmaf(pvz, p.mix, ci.z), vol);
    a.VN[i] = vol;
}

// ---------------------------------------------------------------------------------------------------
// pass A: density / pressure + XSPH intermediate velocity (reference cpp:448-513, 669-701)
// one target of pass A: slot i, in-range list of this lane at shared-memory address slist (stride LSTEP)
__device__ __forceinline__ void pass_a4_one(const DevParams &p, const DevParams *__restrict__ g, const Arrays &a, const int *__restrict__ cell_start,
                                            const uint32_t *__restrict__ skey, const int i, const unsigned slist) {
    const float4 pi = a.P[i];
    const float4 ci = a.C[i];
    const int z0 = g->zero;  // == 0, loaded from global: what is derived from it stays in registers (see list_put)
    const float4 *__restrict__ P = pinned(a.P, z0);
    const float4 *__restrict__ C = a.C;
    const float h2 = g->h2, c6 = g->c_poly6;
    const int ga = g->ga, gagb = g->ga * g->gb;
    const unsigned lbase = slist + 4u * (unsigned)z0;
    const float2 nxy = make_float2(-pi.x, -pi.y);
    const float nz = -pi.z;
    float dens = 0.0f, pvx = 0.0f, pvy = 0.0f, pvz = 0.0f;
    unsigned lofs = lbase;
    const int key = (int)skey[i];  // the sorted cell key of this slot (the limbo bucket = num_cells: no cell, no neighbours)
    if (key < p.num_cells) {
        auto r2_of = [&](const float4 pj) { return dist2_packed(__fadd2_rn(make_float2(pj.x, pj.y), nxy), pj.z + nz); };
        // four candidates per iteration: a lattice row (3-4 candidates) has all its loads in flight at once — the pair loop
        // left the kernel waiting on L1 (long-scoreboard 9 warps per issue at 87 % L1 data-path utilisation, ncu r01_v7)
        sweep4<4>(
            p, cell_start, ga, gagb, key, lbase, lofs,
            [&](int j, int e, unsigned &lo) {
                const float4 p0 = __ldg(P + j), p1 = __ldg(P + j + 1), p2 = __ldg(P + j + 2), p3 = __ldg(P + j + 3);
                const float r0 = r2_of(p0), r1 = r2_of(p1), r2 = r2_of(p2), r3 = r2_of(p3);
                if (r0 <= h2) {  // Poly6 support, cpp:151
                    list_put(lo, j);
                    lo += LSTEP;
                }
                if ((j + 1 < e) & (r1 <= h2)) {
                    list_put(lo, j + 1);
                    lo += LSTEP;
                }
                if ((j + 2 < e) & (r2 <= h2)) {
                    list_put(lo, j + 2);
                    lo += LSTEP;
                }
                if ((j + 3 < e) & (r3 <= h2)) {
                    list_put(lo, j + 3);
                    lo += LSTEP;
                }
            },
            [&](int j, unsigned &lo) {
                if (r2_of(__ldg(P + j)) <= h2) {
                    list_put(lo, j);
                    lo += LSTEP;
                }
            },
            [&](unsigned &lo) {
                for (unsigned q = lbase; q < lo; q += LSTEP) {
                    const int jj = list_get(q);
                    const float4 pj = __ldg(P + jj);
                    const float4 cj = __ldg(C + jj);
                    const float x = h2 - r2_of(pj);
                    const float w = c6 * x * x * x;  // Poly6, cpp:151 (float on the fast path)
                    dens = fmaf(pj.w, w, dens);
                    const float t = w * cj.w;
                    pvx = fmaf(cj.x - ci.x, t, pvx);
                    pvy = fmaf(cj.y - ci.y, t, pvy);
                    pvz = fmaf(cj.z - ci.z, t, pvz);
                }
                lo = lbase;
            });
    }
    pass_a_finish(p, a, i, pi, ci, dens, pvx, pvy, pvz);
}
// RNG: the launch range comes from device memory (slab step).  A template parameter, not a run-time test: with the test compiled
// in, the single-GPU kernel kept 48 bytes of spills at its 56 registers and lost 10 % (ncu r02: 520 us against 470).
template <bool RNG>
__global__ void __launch_bounds__(PT4, A_MINB) k_pass_a4(const __grid_constant__ DevParams p, const DevParams *__restrict__ g, Arrays a,
                                                const int *__restrict__ cell_start, const uint32_t *__restrict__ skey, const int *__restrict__ rng) {
    __shared__ int s_list[LIST_K * PT4];
    int i;
    if (RNG) {
        const int4 v = __ldg(reinterpret_cast<const int4 *>(rng));  // {begin, end, hole_begin, hole_len}
        i = v.x + blockIdx.x * PT4 + threadIdx.x;
        if (i >= v.z) i += v.w;
        if (i >= v.y) return;
    } else {
        i = p.own_begin + blockIdx.x * PT4 + threadIdx.x;
        if (i >= p.hole_begin) i += p.hole_len;
        if (i >= p.own_end) return;
    }
    pass_a4_one(p, g, a, cell_start, skey, i, (unsigned)__cvta_generic_to_shared(s_list) + 4u * threadIdx.x);
}

// ---------------------------------------------------------------------------------------------------
// Update_Properties (cpp:602-649) with reciprocals on the velocity / position side.  The voltage side of the step (ionic
// model with its double promotions, Inter_Vm, the Vm update) keeps the reference's exact operations: Vm then stays
// BIT-IDENTICAL to the reference wherever the Laplacian vanishes (both Resources/*.csv configs as main.cpp runs them), and
// the excitable dynamics amplify rounding differences (cfg2 wave, |dVm| max at step 200: 2.8e-2 exact, 6.7e-2 with a float
// ionic model, which saved 22 us of 717 at 8M: DESIGN.md §4).
__device__ __forceinline__ void integrate_fast(const DevParams &p, bool fixed, float dtm, float ivx, float ivy, float ivz, float ax, float ay, float az,
                                               float inter_vm, float mass, float &x, float &y, float &z, float &vx, float &vy, float &vz, float &Vm) {
    if (!fixed) {
        vx = fmaf(ax, dtm, ivx);
        vy = fmaf(ay, dtm, ivy);
        vz = fmaf(az, dtm, ivz);
        x = fmaf(vx, p.dt, x);
        y = fmaf(vy, p.dt, y);
        z = fmaf(vz, p.dt, z);
    }
    Vm = Vm + div_rn_z(inter_vm * p.dt, mass);  // cpp:612
    Vm = fminf(fmaxf(Vm, -p.max_voltage), p.max_voltage);
    // walls (cpp:620-646); the final bounds.clamp (m3Bounds.h:84-88) cannot move a position that passed them
    if (x < 0.0f) { vx *= p.wall_hit; x = 0.0f; }
    if (x >= p.world[0]) { vx *= p.wall_hit; x = __fsub_rn(p.world[0], 0.0001f); }
    if (y < 0.0f) { vy *= p.wall_hit; y = 0.0f; }
    if (y >= p.world[1]) { vy *= p.wall_hit; y = __fsub_rn(p.world[1], 0.0001f); }
    if (z < 0.0f) { vz *= p.wall_hit; z = 0.0f; }
    if (z >= p.world[2]) { vz *= p.wall_hit; z = __fsub_rn(p.world[2], 0.0001f); }
}

// pass B's per-particle tail, shared by the thread-per-particle and the warp-per-particle kernels: acceleration, Inter_Vm
// (cpp:568-571), Update_Properties (cpp:602-649), and — when cell_count is given — the next step's counting-sort input.
// e4 = (Vm, Iion, w, stim) AFTER the ionic model; L = the SPH Laplacian sum of Vm.
// EGM: also stores the electrogram source vol * L (vi.w = m / dens_new) into a.Q (sphsm_egm.cuh).
// dens = this particle's new density (S.y, written by pass A); the old velocity is not an input of the step's last stage
// (cpp:605: vel = inter_vel + acc * dt / mass), so VEL is written here without having been read.
template <bool DIAG, bool EGM>
__device__ __forceinline__ void pass_b_finish(const DevParams &p, const Arrays &a, float4 *__restrict__ Pout, const int i, const float4 pi,
                                              const float4 vi, float4 e4, const float dens, const bool fixed, float ax, float ay, float az,
                                              const float L, const float inv_mass, uint32_t *__restrict__ next_keys,
                                              uint32_t *__restrict__ next_rank, uint32_t *__restrict__ cell_count) {
    float4 v4 = fixed ? a.VEL[i] : make_float4(0.0f, 0.0f, 0.0f, 0.0f);  // a fixed particle keeps its velocity (cpp:603)
    v4.w = dens;
    const float inv_dens = rcp_ftz(dens);
    ax *= inv_dens;  // cpp:568
    ay *= inv_dens;
    az *= inv_dens;
    // cpp:571: Inter_Vm += (sigma/(Beta*Cm))*Inter_Vm - ((Iion - stim*dt/mass)/Cm)   (the += form, Q9)
    const float dtm = p.dt * inv_mass;
    const float ivm = L + (p.diff_coef * L - (e4.y - div_rn_z(e4.w * p.dt, pi.w)) / p.Cm);
    if (DIAG) a.ACC[i] = make_float4(ax, ay, az, ivm);
    if (EGM) a.Q[i] = vi.w * L;
    float x = pi.x, y = pi.y, z = pi.z;
    integrate_fast(p, fixed, dtm, vi.x, vi.y, vi.z, ax, ay, az, ivm, pi.w, x, y, z, v4.x, v4.y, v4.z, e4.x);
    Pout[i] = make_float4(x, y, z, pi.w);
    a.VEL[i] = v4;
    a.E[i] = e4;
    if (cell_count) {
        int ca, cb, cc;
        const uint32_t key = cell_coords(p, x, y, z, ca, cb, cc) ? (uint32_t)cell_key(p, ca, cb, cc) : (uint32_t)p.num_cells;
        next_keys[i] = key;
        next_rank[i] = atomicAdd(&cell_count[key], 1u);
    }
}

// pass B: ionic cell model + pressure / viscosity force + SPH Laplacian of Vm + integration and walls
// (reference cpp:575-593, 515-573, 598-651).  PB = (pos.xyz, Vm) is the neighbour record of this pass.
// cell_count != nullptr: the thread also files its particle's NEW position for the next step's counting sort (key, provisional
// rank in the cell, per-cell count — what k_cell_count does, without re-reading the positions)
template <bool DIAG, bool EGM>
__device__ __forceinline__ void pass_b4_one(const DevParams &p, const DevParams *__restrict__ g, const Arrays &a, float4 *__restrict__ Pout,
                                            const int *__restrict__ cell_start, const uint32_t *__restrict__ skey, uint32_t *__restrict__ next_keys,
                                            uint32_t *__restrict__ next_rank, uint32_t *__restrict__ cell_count, const int i, const unsigned slist) {
    const float4 pi = a.P[i];
    const float4 vi = a.V[i];
    float4 e4 = a.E[i];
    const float2 si = a.S[i];  // (pres, dens)
    const bool fixed = __float_as_int(a.O[i].w) != 0;  // (loaded with the other records: the epilogue does not wait for it)
    const float pres_i = si.x;
    const float Vm_i = e4.x;
    const float inv_mass = rcp_ftz(pi.w);
    cell_model<false>(p, e4.x, pi.w, e4.y, e4.z);

    const int z0 = g->zero;  // == 0, loaded from global: what is derived from it stays in registers (see list_put)
    const float4 *__restrict__ PB = pinned(a.PB, z0);
    const float4 *__restrict__ V = a.V;
    const float2 *__restrict__ S = a.S;
    const float *__restrict__ VN = pinned(a.VN, z0);
    const float sp2 = g->r2_spiky;
    const float a1 = g->bs_a1, b1 = g->bs_b1, a2 = g->bs_a2, b2 = g->bs_b2;
    const int ga = g->ga, gagb = g->ga * g->gb;
    const unsigned lbase = slist + 4u * (unsigned)z0;
    const float2 nxy = make_float2(-pi.x, -pi.y), nzv = make_float2(-pi.z, -Vm_i);
    float ax = 0.0f, ay = 0.0f, az = 0.0f, L = 0.0f, L1 = 0.0f;  // two Laplacian accumulators: the pair's terms are independent
    unsigned lofs = lbase;
    const int key = (int)skey[i];  // the sorted cell key of this slot (the limbo bucket = num_cells: no cell, no neighbours)
    if (key < p.num_cells) {
        // one candidate of phase 1: the 2h-support Laplacian term (cpp:563), and whether it is inside the Spiky / Visco
        // support r <= h (cpp:157,163).  r2 <= 1e-12 (INF, SPH_SM_monodomain.h:24, cpp:546) skips the pair.
        // (x, y) and (z, Vm) of the record are differenced as packed pairs: (dx, dy), (dz, Vm_j - Vm_i).
        auto cand = [&](const float4 pj, float vol, bool live, float &acc) -> bool {
            const float2 dxy = __fadd2_rn(make_float2(pj.x, pj.y), nxy);
            const float2 dzv = __fadd2_rn(make_float2(pj.z, pj.w), nzv);
            const float r2 = dist2_packed(dxy, dzv.x);
            const bool on = live && r2 > 1e-12f;
            const float r = sqrt_ftz(r2);
            const float bs = fminf(fmaf(a1, r, b1), fmaxf(fmaf(a2, r, b2), 0.0f));  // B_spline_2, cpp:188-197 (negative for q < 2/3)
            const float t = fmaf(dzv.y * vol, bs, acc);
            acc = on ? t : acc;
            return on && r2 <= sp2;
        };
        // two candidates per iteration (four, as in pass A, need 72 registers and measured 686 us against 678: DESIGN.md §4)
        sweep4<2>(
            p, cell_start, ga, gagb, key, lbase, lofs,
            [&](int j, bool two, unsigned &lo) {
                const float4 p0 = __ldg(PB + j), p1 = __ldg(PB + j + 1);
                const float v0 = __ldg(VN + j), v1 = __ldg(VN + j + 1);
                if (cand(p0, v0, true, L)) {
                    list_put(lo, j);
                    lo += LSTEP;
                }
                if (cand(p1, v1, two, L1)) {
                    list_put(lo, j + 1);
                    lo += LSTEP;
                }
            },
            [&](int j, unsigned &lo) {
                if (cand(__ldg(PB + j), __ldg(VN + j), true, L)) {
                    list_put(lo, j);
                    lo += LSTEP;
                }
            },
            [&](unsigned &lo) {
                const float hh = g->h, cs_half = 0.5f * g->c_spiky, cs_mu = g->c_spiky * g->mu;
                for (unsigned q = lbase; q < lo; q += LSTEP) {
                    const int jj = list_get(q);
                    const float4 pj = __ldg(PB + jj);
                    const float4 vj = __ldg(V + jj);
                    const float pres_j = __ldg(&S[jj].x);
                    const float dx = pi.x - pj.x, dy = pi.y - pj.y, dz = pi.z - pj.z;
                    const float r2 = dist2_exact(dx, dy, dz);
                    const float inv_r = rsqrt_ftz(r2);
                    const float hr = fmaf(-r2, inv_r, hh);
                    const float t = vj.w * hr;
                    const float fpr = (t * hr) * (inv_r * cs_half) * (pres_i + pres_j);  // = -(Force_pressure / dis), cpp:553-554
                    const float fv = t * cs_mu;                                           // Force_viscosity, cpp:559
                    ax = fmaf(dx, fpr, ax);
                    ay = fmaf(dy, fpr, ay);
                    az = fmaf(dz, fpr, az);
                    ax = fmaf(vj.x - vi.x, fv, ax);
                    ay = fmaf(vj.y - vi.y, fv, ay);
                    az = fmaf(vj.z - vi.z, fv, az);
                }
                lo = lbase;
            });
    }
    pass_b_finish<DIAG, EGM>(p, a, Pout, i, pi, vi, e4, si.y, fixed, ax, ay, az, L + L1, inv_mass, next_keys, next_rank, cell_count);
}
template <bool DIAG, bool RNG, bool EGM>
__global__ void __launch_bounds__(PT4, B_MINB) k_pass_b4(const __grid_constant__ DevParams p, const DevParams *__restrict__ g, Arrays a,
                                                float4 *__restrict__ Pout, const int *__restrict__ cell_start, const uint32_t *__restrict__ skey,
                                                uint32_t *__restrict__ next_keys, uint32_t *__restrict__ next_rank, uint32_t *__restrict__ cell_count,
                                                const int *__restrict__ rng) {
    __shared__ int s_list[LIST_K * PT4];
    int i;
    if (RNG) {
        const int4 v = __ldg(reinterpret_cast<const int4 *>(rng));  // {begin, end, hole_begin, hole_len}
        i = v.x + blockIdx.x * PT4 + threadIdx.x;
        if (i >= v.z) i += v.w;
        if (i >= v.y) return;
    } else {
        i = p.own_begin + blockIdx.x * PT4 + threadIdx.x;
        if (i >= p.hole_begin) i += p.hole_len;
        if (i >= p.own_end) return;
    }
    pass_b4_one<DIAG, EGM>(p, g, a, Pout, cell_start, skey, next_keys, next_rank, cell_count, i, (unsigned)__cvta_generic_to_shared(s_list) + 4u * threadIdx.x);
}

}  // namespace sphsm
