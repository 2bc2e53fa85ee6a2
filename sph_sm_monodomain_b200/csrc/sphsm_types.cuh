// sphsm_types.cuh — device-side parameter block, HBM data layout and the arithmetic policy.
//
// HBM layout (all arrays are SoA, length = capacity, kept in CELL-SORTED slot order; see DESIGN.md §3):
//   P    float4  (pos.xyz, mass)              persistent   — the only array both neighbour passes gather
//   VEL  float4  (vel.xyz, dens)              persistent
//   O    float4  (orig.xyz, bits(flags))      persistent   — flags: 0 = free, k>0 = fixed, cold index k-1
//   E    float4  (Vm, Iion, w, stim)          persistent
//   ID   int32   original particle index      persistent
//   C    float4  (corrected_vel.xyz, m/dens_old)   written by stage 2, gathered by pass A
//   V    float4  (inter_vel.xyz,     m/dens_new)   written by pass A, gathered by pass B
//   S    float2  (pres, Vm)                        written by pass A, gathered by pass B
//   PB   float4  (pos.xyz, Vm)                     written by the reorder, gathered by pass B (fast path)
//   VN   float   m/dens_new (= V.w), dense         written by pass A, gathered by pass B's phase 1 (fast path)
//   ACC  float4  (acc.xyz, Inter_Vm)               staged / diagnostics mode only
//   Q    float   vol * L, pass B's source strength  electrograms only (sphsm_egm.cuh); null while they are off
//   GOAL float4  (goal.xyz, -)  PV float4 (predicted_vel.xyz, -)   diagnostics mode only
//   COLD_GOAL / COLD_PV float4 by ORIGINAL index: the frozen mGoalPos / predicted_vel of fixed particles
//        (the reference never updates them for mFixed particles, cpp:228,326,431)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace sphsm {

struct DevParams {
    int n;
    int g[3];        // Grid_Size (x,y,z), cpp:32-35
    int perm[3];     // key = c[perm0] + G[perm0]*(c[perm1] + G[perm1]*c[perm2]); (0,1,2) = the reference hash
    int ga, gb, gc;  // G[perm0] + 2, G[perm1] + 2 (one empty border cell on either side, see cell_coords), G[perm2]
    int num_cells;   // ga*gb*gcl; key num_cells is the limbo bucket (outside the grid / NaN)
    float cell_size, h, h2;
    float world[3];
    float gravity[3];
    float K, rho0, dt, inv_dt, wall_hit, mu, mix;
    float c_poly6, c_spiky, c_bspline;
    float alpha, beta;
    int quadratic, volume, allow_flip;
    float Cm, Beta, sigma, diff_coef;  // diff_coef = sigma / (Beta * Cm), cpp:571
    float Vr, fh_denom, fh_asd, C1, C2, C3, C4;
    float voltage_constant, max_pressure, max_voltage;
    // exact r^2 thresholds (host-computed, see sphsm_capi.cu:compute_thresholds): the largest float r2 with
    //   sqrt_rn(r2) <= h            (Spiky/Visco support, cpp:157,163)
    //   div_rn(sqrt_rn(r2), h) < 1  (B_spline_2 inner branch, cpp:191)
    //   div_rn(sqrt_rn(r2), h) < 2  (B_spline_2 outer branch, cpp:193)
    float r2_spiky, r2_q1, r2_q2;
    // fast-path folded constants
    float bs_a1, bs_b1, bs_a2, bs_b2;  // B2(r) = bs_a*r + bs_b on the two branches
    float poly6_self;                  // Poly6(0), cpp:483
    // slab decomposition (multi-GPU): this rank's grid holds the planes [c_off, c_off + gcl) along perm[2]
    // (owned planes [slab_lo, slab_hi) plus one halo plane per interior side); single GPU: c_off = 0, gcl = gc.
    int c_off, gcl, slab_lo, slab_hi;
    int slab_on;              // 1: multi-GPU slab mode (sums and outputs cover owned particles only)
    int own_begin, own_end;   // slot range the neighbour passes compute ([0, n) on a single GPU)
    int hole_begin, hole_len; // ... minus [hole_begin, hole_begin + hole_len): one launch over the two boundary planes of a slab
    int zero;  // always 0; read from the global-memory copy of this block to build values ptxas cannot re-materialise
};

struct Arrays {
    float4 *P, *VEL, *O, *E;
    int *ID;
    float4 *C, *V;
    float2 *S;
    float4 *ACC, *GOAL, *PV;
    float4 *PB;  // (pos.xyz, Vm): pass B's neighbour record, written by the reorder
    float *VN;   // m/dens_new again, as a DENSE float array: pass B's phase 1 reads it for every candidate, and a 4-byte
                 // gather from the 16-byte-strided V.w costs four L1 wavefronts per warp where this costs one
    float4 *COLD_GOAL, *COLD_PV;
    float *Q;    // electrograms only: the same buffer in both ping-pong sets (written and read within one step)
};

// Shape-matching results shared between the solve and the per-particle goal kernel.
struct SmState {
    // rest-state (cached until orig/mass/fixed change)
    double Mfix;        // sum m' (fixed x100), cpp:244-251
    double M;           // sum m
    double SmpX[3];     // sum m' X
    double Smq9[9];     // sum m q9  (q = X - ocm)
    float ocm[3];
    float Aqq[9], AqqInv[9];
    int aqq_inv_ok;
    float A9qq[81], A9qqInv[81];
    // per step
    float cm[3];
    float xform[27];    // linear: T in [0..8]; quadratic: the 3x9 matrix, cpp:390-427
    float R[9];
};

// ---------------------------------------------------------------------------------------------------
// Arithmetic policy.  STRICT = the reference's x86-64 evaluation: every float op rounded separately
// (no FMA contraction), IEEE sqrt/div.  FAST = plain operators (nvcc may contract to FMA).
template <bool STRICT>
struct Ar {
    static __device__ __forceinline__ float mul(float a, float b) { return STRICT ? __fmul_rn(a, b) : a * b; }
    static __device__ __forceinline__ float add(float a, float b) { return STRICT ? __fadd_rn(a, b) : a + b; }
    static __device__ __forceinline__ float sub(float a, float b) { return STRICT ? __fsub_rn(a, b) : a - b; }
    static __device__ __forceinline__ float div(float a, float b) { return STRICT ? __fdiv_rn(a, b) : a / b; }
    static __device__ __forceinline__ float sqrt(float a) { return STRICT ? __fsqrt_rn(a) : sqrtf(a); }
    static __device__ __forceinline__ double dmul(double a, double b) { return STRICT ? __dmul_rn(a, b) : a * b; }
    static __device__ __forceinline__ double dadd(double a, double b) { return STRICT ? __dadd_rn(a, b) : a + b; }
    static __device__ __forceinline__ double ddiv(double a, double b) { return STRICT ? __ddiv_rn(a, b) : a / b; }
};

// r^2 exactly as m3Vector::magnitudeSquared evaluates it on x86-64 (m3Vector.h:93): separate mul/add in
// both modes — neighbour-set membership must be bit-exact even on the fast path.
__device__ __forceinline__ float dist2_exact(float dx, float dy, float dz) {
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// Calculate_Cell_Position + the range test of Calculate_Cell_Hash (cpp:127-141): float division by
// Cell_Size and C truncation.  Returns false for positions outside the grid (or NaN): the limbo bucket.
// ca and cb are returned BORDER-RELATIVE (+1): the cell table carries one empty cell on either side of the two fast key
// axes, so the 3x3 rows x 3 cells around any particle exist and the sweeps need neither clamps nor range tests.
__device__ __forceinline__ bool cell_coords(const DevParams &p, float x, float y, float z, int &ca, int &cb, int &cc) {
    int cx = __float2int_rz(__fdiv_rn(x, p.cell_size));
    int cy = __float2int_rz(__fdiv_rn(y, p.cell_size));
    int cz = __float2int_rz(__fdiv_rn(z, p.cell_size));
    bool ok = (x == x) && (y == y) && (z == z) && cx >= 0 && cx < p.g[0] && cy >= 0 && cy < p.g[1] && cz >= 0 && cz < p.g[2];
    ca = (p.perm[0] == 0 ? cx : (p.perm[0] == 1 ? cy : cz)) + 1;
    cb = (p.perm[1] == 0 ? cx : (p.perm[1] == 1 ? cy : cz)) + 1;
    cc = p.perm[2] == 0 ? cx : (p.perm[2] == 1 ? cy : cz);
    if (ok && (cc < p.c_off || cc >= p.c_off + p.gcl)) ok = false;  // outside this rank's slab + halo
    return ok;
}
__device__ __forceinline__ int cell_key(const DevParams &p, int ca, int cb, int cc) {
    return ca + p.ga * (cb + p.gb * (cc - p.c_off));
}

// Visit the 27-cell stencil in the reference's order (outer perm2, middle perm1, inner perm0 — k,j,i for the
// reference key, cpp:462-464).  The three perm0-neighbours of a row are contiguous in the sorted arrays, so a row
// is ONE run [cell_start[first], cell_start[last+1]).
template <class F>
__device__ __forceinline__ void for_each_candidate(const DevParams &p, const int *__restrict__ cell_start, int ca, int cb, int cc, F &&f) {
    const int a_lo = max(ca - 1, 0), a_hi = min(ca + 1, p.ga - 1);
#pragma unroll 1
    for (int dc = -1; dc <= 1; dc++) {
        int c2 = cc + dc;
        if (c2 < p.c_off || c2 >= p.c_off + p.gcl) continue;
#pragma unroll 1
        for (int db = -1; db <= 1; db++) {
            int b2 = cb + db;
            if (b2 < 0 || b2 >= p.gb) continue;
            int row = p.ga * (b2 + p.gb * (c2 - p.c_off));
            int s = __ldg(cell_start + row + a_lo);
            int e = __ldg(cell_start + row + a_hi + 1);
#pragma unroll 1
            for (int j = s; j < e; j++) f(j);
        }
    }
}

}  // namespace sphsm
