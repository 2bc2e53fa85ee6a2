// sphsm_pass6.cuh — the neighbour passes with the stencil rows of a whole block of targets staged in shared memory by 1-D bulk
// copies (cp.async.bulk + mbarrier, the TMA engine); phase 1 reads shared memory.  Selected with SPHSM_PASS=6 /
// sphsm_tune("pass", 6); NOT the default: measured at 8M on one B200 it is slower than the gathered passes of sphsm_pass4.cuh
// (pass A 548 us against 469, pass B 859 against 716; ncu profiles/r02_gen6_pass_{a,b}.json, SASS excerpt
// profiles/r02_gen6_sass_excerpt.txt).  The staging itself does what it was built for — the candidate-pair loops drop to 18 % of the
// warp samples while issuing 48 % of the instructions — but nine spans of ~T records are 280 B of shared memory per target: 5 blocks
// = 20 warps per SM (gathered: 32), and with so few warps the block start-up chain (keys -> cell table -> copies), phase 2's L2
// gathers and the epilogue's atomics are exposed (12 % of the samples wait at the block barrier alone).  Sharing the spans between
// four adjacent cell rows (multi-row tiles, 100 B per target) was built as well and lost to register pressure (two sweeps plus
// the tile bookkeeping need 80-96 registers; 64-72 spill: 1124-1579 us) — DESIGN.md section 4.
//
// What generation 4 left on the table (ncu profiles/r01_v8_pass_{a,b}.json and their source pages): both passes are issue / L1
// bound with HALF of the pair loop's stall samples on one instruction, the first use of the gathered candidate records
// (long scoreboard: 64 % L1 hit rate, the rest pays L2 latency), and 800 of pass B's 2075 warp instructions per 32 particles
// sit outside the candidate loops (cell coordinates by three IEEE divisions, 64-bit address arithmetic for 18 row bounds, a
// division slow path taken by every warp).
//
// The slots are sorted by cell key, so the T consecutive targets of a block cover one contiguous KEY range [kf, kl], and for
// each of the nine stencil rows (db, dc) the union of their candidate windows is the contiguous key range
// [kf + off - 1, kl + off + 1] (off = dc * ga * gb + db * ga; the padded cell table makes this true across row ends as well), i.e.
// ONE contiguous slot range.  Nine spans per block, each fetched by one bulk copy per record array straight from L2 into
// shared memory (no L1 tags, no registers, no per-lane address arithmetic) while the threads run their prologue (own
// records, ionic model).  The candidate loops are those of generation 4 with LDS in place of LDG: same candidates, same
// order, same arithmetic, so the results are BIT-IDENTICAL to generation 4 (tests/test_gpu_api.py::test_staged_matches_gathered).
//
// A block whose spans do not fit the staging area (dense meshes: the reference's own inputs hold up to 75 particles per cell;
// sparse sets: key ranges of thousands of cells) takes the gathered path of generation 4 inside the same kernel — the
// choice is per block and changes no result.
//
// Also new here: the sorted cell key of every slot is kept (SKEY, written by the sort), so neither pass recomputes cell
// coordinates; plane validity follows from the key alone (key >= ga*gb: a lower plane exists; key + ga*gb < num_cells: an upper
// one does).
#pragma once
#include "sphsm_pass4.cuh"

namespace sphsm {

constexpr int SPAN_TAIL = 4;  // records staged behind each span: the pair / quad loops read up to j + 3 (masked) past a row end

// ---- PTX: shared-memory loads by 32-bit address, mbarrier, bulk copy -------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *ptr) { return (unsigned)__cvta_generic_to_shared(ptr); }
__device__ __forceinline__ float4 lds_f4(unsigned addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float lds_f32(unsigned addr) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ unsigned lds_u32(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void mbar_init(unsigned mbar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(mbar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {  // makes the initialised barrier visible to the async proxy (the TMA engine)
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned mbar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned mbar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SPHSM_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra SPHSM_DONE;\n"
        "bra SPHSM_WAIT;\n"
        "SPHSM_DONE:\n"
        "}\n" ::"r"(mbar),
        "r"(parity)
        : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completion is counted on the mbarrier
__device__ __forceinline__ void bulk_g2s(unsigned dst, const void *src, unsigned bytes, unsigned mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes), "r"(mbar)
                 : "memory");
}

// ---- shared-memory layout of one block of T targets ------------------------------------------------------------------------
//   [0, 8)      the mbarrier
//   [16, 52)    c16[9]: per span, (shared address of its first staged 16-byte record) - 16 * (its first global slot), so that the
//               record of global slot j sits at c16[r] + 16 * j (unsigned wrap-around arithmetic)
//   [52, 88)    c4[9]: the same for the 4-byte array (pass B's VN)
//   [96, 100)   staged flag of the block
//   [128, ...)  the in-range lists (LIST_K entries per lane), the 16-byte stage, the 4-byte stage
template <int T, bool WITH4>
struct Lay6 {
    static constexpr int SLOTS = 14 * T;  // 16-byte records staged per block: a lattice block needs 9-16 lattice lines of ~T + 4 (see DESIGN.md)
    static constexpr int SLOTS4 = SLOTS + 9 * 8;
    static constexpr int LISTK = LIST_K;  // in-range list entries per lane between drains
    static constexpr unsigned OFF_MBAR = 0, OFF_C16 = 16, OFF_C4 = 52, OFF_FLAG = 96, OFF_LIST = 128;
    static constexpr unsigned OFF_ST16 = OFF_LIST + 4u * LIST_K * T;
    static constexpr unsigned OFF_ST4 = OFF_ST16 + 16u * SLOTS;
    static constexpr unsigned BYTES = WITH4 ? OFF_ST4 + 4u * SLOTS4 : OFF_ST4;
};

// the slot range of block `b` of a launch over [own_begin, own_end) minus the hole: blocks never straddle the hole, so a block's
// targets are consecutive slots.  Host side: grid6() gives the matching block count.
template <int T>
__device__ __forceinline__ void block_range6(const Range4 &r, int b, int &base, int &end) {
    const int len1 = r.hole_len > 0 ? r.hole_begin - r.begin : r.end - r.begin;
    const int nb1 = (len1 + T - 1) / T;
    if (b < nb1) {
        base = r.begin + b * T;
        end = r.begin + len1;
    } else {
        base = r.hole_begin + r.hole_len + (b - nb1) * T;
        end = r.end;
    }
}

// Warp 0 of the block: slot ranges of the nine spans, the staging decision, the bulk copies, the address tables.
//   kf, kl      keys of the first and of the last target of the block that has a cell (nv > 0 of them)
//   A16 / A4    the global arrays staged as 16-byte / 4-byte records (A4 == nullptr: none)
// Returns (to every lane of warp 0) whether the block is staged.
template <int T, bool WITH4>
__device__ __forceinline__ bool stage_spans6(const DevParams &p, const int *__restrict__ cell_start, const int ga, const int gagb, const int nv,
                                             const int kf, const int kl, const float4 *__restrict__ A16, const float *__restrict__ A4,
                                             const unsigned smem0, const bool enabled) {
    using L = Lay6<T, WITH4>;
    const int lane = threadIdx.x & 31;
    int slo = 0, len = 0;
    if (lane < 9 && nv > 0) {
        const int off = (lane / 3 - 1) * gagb + (lane % 3 - 1) * ga;
        const int kmin = max(kf + off - 1, 0), kmax = min(kl + off + 2, p.num_cells);  // clamps: planes / rows that do not exist
        if (kmin < kmax) {
            slo = __ldg(cell_start + kmin);
            len = __ldg(cell_start + kmax) - slo;
        }
    }
    const int n16 = len > 0 ? len + SPAN_TAIL : 0;
    const int lo4 = slo & ~3;  // 16-byte alignment of the 4-byte array's source address
    const int n4 = (WITH4 && len > 0) ? ((slo + len + SPAN_TAIL + 3) & ~3) - lo4 : 0;
    int o16 = n16, o4 = n4;  // inclusive prefix sums over the lanes
#pragma unroll
    for (int d = 1; d < 16; d <<= 1) {
        const int t16 = __shfl_up_sync(0xffffffffu, o16, d), t4 = __shfl_up_sync(0xffffffffu, o4, d);
        if (lane >= d) { o16 += t16; o4 += t4; }
    }
    const int tot16 = __shfl_sync(0xffffffffu, o16, 8), tot4 = __shfl_sync(0xffffffffu, o4, 8);
    o16 -= n16;
    o4 -= n4;
    const bool staged = enabled && tot16 <= L::SLOTS && tot4 <= L::SLOTS4;
    const unsigned mbar = smem0 + L::OFF_MBAR;
    const unsigned st16 = smem0 + L::OFF_ST16 + 16u * (unsigned)o16, st4 = smem0 + L::OFF_ST4 + 4u * (unsigned)o4;
    if (staged) {
        if (lane == 0) mbar_arrive_expect_tx(mbar, 16u * (unsigned)tot16 + 4u * (unsigned)tot4);
        __syncwarp();
        if (n16 > 0) {
            bulk_g2s(st16, A16 + slo, 16u * (unsigned)n16, mbar);
            if (WITH4) bulk_g2s(st4, A4 + lo4, 4u * (unsigned)n4, mbar);
        }
    }
    if (lane < 9) {
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(smem0 + L::OFF_C16 + 4u * lane), "r"(st16 - 16u * (unsigned)slo) : "memory");
        if (WITH4) asm volatile("st.shared.u32 [%0], %1;" ::"r"(smem0 + L::OFF_C4 + 4u * lane), "r"(st4 - 4u * (unsigned)lo4) : "memory");
    }
    if (lane == 0) asm volatile("st.shared.u32 [%0], %1;" ::"r"(smem0 + L::OFF_FLAG), "r"(staged ? 1u : 0u) : "memory");
    return staged;
}

// Sweep the nine stencil rows in the reference's order (cpp:462-464), as sweep4 does; `row(r)` is called before each row with its
// plane (0..2) and row (0..2) indices, so that the staged variant can fetch the row's shared-memory address constants.
template <int T, int STEP, int LISTK, class Row, class Pair, class One, class Drain>
__device__ __forceinline__ void sweep6(const int *__restrict__ cell_start, const int ga, const int gagb, const int num_cells, const int key,
                                       const unsigned lbase, unsigned &lofs, Row &&row, Pair &&pair, One &&one, Drain &&drain) {
    constexpr unsigned LSTEP6 = 4u * T;
    const int *center = cell_start + (key - 1);
    const unsigned lmax = lbase + LISTK * LSTEP6;
    Rows3 cur, nxt;
    load_rows3(center - gagb, ga, key >= gagb, cur);
#pragma unroll 1
    for (int dc = 0; dc < 3; dc++) {
        if (dc == 0) load_rows3(center, ga, true, nxt);
        else if (dc == 1) load_rows3(center + gagb, ga, key + gagb < num_cells, nxt);
#pragma unroll
        for (int k = 0; k < 3; k++) {
            int j = cur.s[k];
            const int e = cur.e[k];
            row(dc, k);
            if (lofs + (unsigned)(e - j) * LSTEP6 <= lmax) {
#pragma unroll 1
                for (; j < e; j += STEP) pair(j, e, lofs);  // the body masks j+1 .. j+STEP-1 against the row end itself
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

// ---------------------------------------------------------------------------------------------------
// pass A: density / pressure + XSPH intermediate velocity (reference cpp:448-513, 669-701)
// L = the shared-memory layout; tstride / trow: the address tables hold `tstride` spans per plane and this target's three stencil
// rows are entries trow, trow + 1, trow + 2 of each plane (generation 6: 3 and 0; the multi-row tiles of generation 7: R + 2 and
// the target's row inside the tile)
template <class L, int T, bool STAGED>
__device__ __forceinline__ void pass_a6_neighbours(const DevParams *__restrict__ g, const Arrays &a, const int *__restrict__ cell_start, const int key,
                                                   const unsigned smem0, const int tstride, const int trow, const float4 pi, const float4 ci,
                                                   float &dens, float &pvx, float &pvy, float &pvz) {
    constexpr unsigned LSTEP6 = 4u * T;
    const int z0 = g->zero;  // == 0, loaded from global: what is derived from it stays in registers (see list_put)
    const float4 *__restrict__ P = pinned(a.P, z0);
    const float4 *__restrict__ C = a.C;
    const float h2 = g->h2, c6 = g->c_poly6;
    const int ga = g->ga, gagb = g->ga * g->gb, num_cells = g->num_cells;
    const unsigned lbase = smem0 + L::OFF_LIST + 4u * (unsigned)(threadIdx.x + z0);
    const unsigned tab = smem0 + L::OFF_C16 + 4u * (unsigned)(trow + z0);
    const float2 nxy = make_float2(-pi.x, -pi.y);
    const float nz = -pi.z;
    unsigned lofs = lbase, c16 = 0;
    auto r2_of = [&](const float4 pj) { return dist2_packed(__fadd2_rn(make_float2(pj.x, pj.y), nxy), pj.z + nz); };
    auto ld = [&](int j) -> float4 {
        if constexpr (STAGED) return lds_f4(c16 + 16u * (unsigned)j);
        else return __ldg(P + j);
    };
    sweep6<T, 4, L::LISTK>(
        cell_start, ga, gagb, num_cells, key, lbase, lofs,
        [&](int dc, int k) {
            if constexpr (STAGED) c16 = lds_u32(tab + 4u * (unsigned)(dc * tstride + k));
        },
        [&](int j, int e, unsigned &lo) {
            const float4 p0 = ld(j), p1 = ld(j + 1), p2 = ld(j + 2), p3 = ld(j + 3);
            const float r0 = r2_of(p0), r1 = r2_of(p1), r2 = r2_of(p2), r3 = r2_of(p3);
            if (r0 <= h2) {  // Poly6 support, cpp:151
                list_put(lo, j);
                lo += LSTEP6;
            }
            if ((j + 1 < e) & (r1 <= h2)) {
                list_put(lo, j + 1);
                lo += LSTEP6;
            }
            if ((j + 2 < e) & (r2 <= h2)) {
                list_put(lo, j + 2);
                lo += LSTEP6;
            }
            if ((j + 3 < e) & (r3 <= h2)) {
                list_put(lo, j + 3);
                lo += LSTEP6;
            }
        },
        [&](int j, unsigned &lo) {
            if (r2_of(ld(j)) <= h2) {
                list_put(lo, j);
                lo += LSTEP6;
            }
        },
        [&](unsigned &lo) {
            for (unsigned q = lbase; q < lo; q += LSTEP6) {
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

template <int T>
__global__ void __launch_bounds__(T, 768 / T) k_pass_a6(const __grid_constant__ DevParams p, const DevParams *__restrict__ g, Arrays a,
                                               const int *__restrict__ cell_start, const uint32_t *__restrict__ skey, int stage_on,
                                               const int *__restrict__ rng) {
    using L = Lay6<T, false>;
    extern __shared__ __align__(128) uint8_t smem6[];
    const unsigned smem0 = smem_u32(smem6);
    int base, end;
    block_range6<T>(launch_range(p, rng), blockIdx.x, base, end);
    const int i = base + threadIdx.x;
    const bool live = i < end;
    const int key = live ? (int)skey[i] : p.num_cells;
    const bool valid = key < p.num_cells;  // has a cell (the limbo bucket sorts last: the valid targets of a block are a prefix)
    if (threadIdx.x == 0) {
        mbar_init(smem0 + L::OFF_MBAR, 1);
        mbar_fence_init();
    }
    const int nv = __syncthreads_count(valid);
    if (threadIdx.x < 32) {
        const int kf = (int)skey[base], kl = nv > 0 ? (int)skey[base + nv - 1] : 0;
        stage_spans6<T, false>(p, cell_start, p.ga, p.ga * p.gb, nv, kf, kl, a.P, nullptr, smem0, stage_on != 0);
    }
    float4 pi = make_float4(0.f, 0.f, 0.f, 0.f), ci = pi;
    if (live) {
        pi = a.P[i];
        ci = a.C[i];
    }
    __syncthreads();
    const bool staged = lds_u32(smem0 + L::OFF_FLAG) != 0;
    float dens = 0.0f, pvx = 0.0f, pvy = 0.0f, pvz = 0.0f;
    if (staged) {
        mbar_wait(smem0 + L::OFF_MBAR, 0);
        if (valid) pass_a6_neighbours<L, T, true>(g, a, cell_start, key, smem0, 3, 0, pi, ci, dens, pvx, pvy, pvz);
    } else if (valid) {
        pass_a6_neighbours<L, T, false>(g, a, cell_start, key, smem0, 3, 0, pi, ci, dens, pvx, pvy, pvz);
    }
    if (live) pass_a_finish(p, a, i, pi, ci, dens, pvx, pvy, pvz);
}

// ---------------------------------------------------------------------------------------------------
// pass B: ionic cell model + pressure / viscosity force + SPH Laplacian of Vm + integration and walls
// (reference cpp:575-593, 515-573, 598-651).  PB = (pos.xyz, Vm) and VN = m/dens are the neighbour records of phase 1.
template <class L, int T, int STEP, bool STAGED>
__device__ __forceinline__ void pass_b6_neighbours(const DevParams *__restrict__ g, const Arrays &a, const int *__restrict__ cell_start, const int key,
                                                   const unsigned smem0, const int tstride, const int trow, const float4 pi, const float4 vi,
                                                   const float Vm_i, const float pres_i, float &ax, float &ay, float &az, float &Lsum) {
    constexpr unsigned LSTEP6 = 4u * T;
    const int z0 = g->zero;  // == 0, loaded from global: what is derived from it stays in registers (see list_put)
    const float4 *__restrict__ PB = pinned(a.PB, z0);
    const float4 *__restrict__ V = a.V;
    const float2 *__restrict__ S = a.S;
    const float *__restrict__ VN = pinned(a.VN, z0);
    const float sp2 = g->r2_spiky;
    const float a1 = g->bs_a1, b1 = g->bs_b1, a2 = g->bs_a2, b2 = g->bs_b2;
    const int ga = g->ga, gagb = g->ga * g->gb, num_cells = g->num_cells;
    const unsigned lbase = smem0 + L::OFF_LIST + 4u * (unsigned)(threadIdx.x + z0);
    const unsigned tab = smem0 + L::OFF_C16 + 4u * (unsigned)(trow + z0);
    const float2 nxy = make_float2(-pi.x, -pi.y), nzv = make_float2(-pi.z, -Vm_i);
    float L0 = 0.0f, L1 = 0.0f;  // two Laplacian accumulators: even / odd candidates of a row (as generation 4)
    unsigned lofs = lbase, c16 = 0, c4 = 0;
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
    auto ld16 = [&](int j) -> float4 {
        if constexpr (STAGED) return lds_f4(c16 + 16u * (unsigned)j);
        else return __ldg(PB + j);
    };
    auto ld4 = [&](int j) -> float {
        if constexpr (STAGED) return lds_f32(c4 + 4u * (unsigned)j);
        else return __ldg(VN + j);
    };
    sweep6<T, STEP, L::LISTK>(
        cell_start, ga, gagb, num_cells, key, lbase, lofs,
        [&](int dc, int k) {
            if constexpr (STAGED) {
                const unsigned q = tab + 4u * (unsigned)(dc * tstride + k);
                c16 = lds_u32(q);
                c4 = lds_u32(q + (L::OFF_C4 - L::OFF_C16));
            }
        },
        [&](int j, int e, unsigned &lo) {
            if constexpr (STEP == 4) {
                const float4 p0 = ld16(j), p1 = ld16(j + 1), p2 = ld16(j + 2), p3 = ld16(j + 3);
                const float v0 = ld4(j), v1 = ld4(j + 1), v2 = ld4(j + 2), v3 = ld4(j + 3);
                const bool i0 = cand(p0, v0, true, L0), i1 = cand(p1, v1, j + 1 < e, L1);
                const bool i2 = cand(p2, v2, j + 2 < e, L0), i3 = cand(p3, v3, j + 3 < e, L1);
                if (i0) { list_put(lo, j); lo += LSTEP6; }
                if (i1) { list_put(lo, j + 1); lo += LSTEP6; }
                if (i2) { list_put(lo, j + 2); lo += LSTEP6; }
                if (i3) { list_put(lo, j + 3); lo += LSTEP6; }
            } else {
                const float4 p0 = ld16(j), p1 = ld16(j + 1);
                const float v0 = ld4(j), v1 = ld4(j + 1);
                if (cand(p0, v0, true, L0)) { list_put(lo, j); lo += LSTEP6; }
                if (cand(p1, v1, j + 1 < e, L1)) { list_put(lo, j + 1); lo += LSTEP6; }
            }
        },
        [&](int j, unsigned &lo) {
            if (cand(ld16(j), ld4(j), true, L0)) {
                list_put(lo, j);
                lo += LSTEP6;
            }
        },
        [&](unsigned &lo) {
            const float hh = g->h, cs_half = 0.5f * g->c_spiky, cs_mu = g->c_spiky * g->mu;
            for (unsigned q = lbase; q < lo; q += LSTEP6) {
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
    Lsum = L0 + L1;
}

// cell_count != nullptr: the thread also files its particle's NEW position for the next step's counting sort (key, provisional
// rank in the cell, per-cell count — what k_cell_count does, without re-reading the positions)
template <int T, int STEP, bool DIAG, bool EGM>
__global__ void __launch_bounds__(T, 640 / T) k_pass_b6(const __grid_constant__ DevParams p, const DevParams *__restrict__ g, Arrays a,
                                               float4 *__restrict__ Pout, const int *__restrict__ cell_start, const uint32_t *__restrict__ skey,
                                               uint32_t *__restrict__ next_keys, uint32_t *__restrict__ next_rank, uint32_t *__restrict__ cell_count,
                                               int stage_on, const int *__restrict__ rng) {
    using L = Lay6<T, true>;
    extern __shared__ __align__(128) uint8_t smem6[];
    const unsigned smem0 = smem_u32(smem6);
    int base, end;
    block_range6<T>(launch_range(p, rng), blockIdx.x, base, end);
    const int i = base + threadIdx.x;
    const bool live = i < end;
    const int key = live ? (int)skey[i] : p.num_cells;
    const bool valid = key < p.num_cells;
    if (threadIdx.x == 0) {
        mbar_init(smem0 + L::OFF_MBAR, 1);
        mbar_fence_init();
    }
    const int nv = __syncthreads_count(valid);
    if (threadIdx.x < 32) {
        const int kf = (int)skey[base], kl = nv > 0 ? (int)skey[base + nv - 1] : 0;
        stage_spans6<T, true>(p, cell_start, p.ga, p.ga * p.gb, nv, kf, kl, a.PB, a.VN, smem0, stage_on != 0);
    }
    // the block's own records and the ionic model run while the spans are in flight
    float4 pi = make_float4(0.f, 0.f, 0.f, 1.f), vi = make_float4(0.f, 0.f, 0.f, 0.f), e4 = vi;
    float2 si = make_float2(0.f, 1.f);
    bool fixed = false;
    if (live) {
        pi = a.P[i];
        vi = a.V[i];
        e4 = a.E[i];
        si = a.S[i];  // (pres, dens)
        fixed = __float_as_int(a.O[i].w) != 0;
    }
    const float Vm_i = e4.x;
    const float inv_mass = rcp_ftz(pi.w);
    if (live) {
        if (SPHSM_FAST_ODE) cell_model_fast(p, e4.x, inv_mass, e4.y, e4.z);
        else cell_model<false>(p, e4.x, pi.w, e4.y, e4.z);
    }
    __syncthreads();
    const bool staged = lds_u32(smem0 + L::OFF_FLAG) != 0;
    float ax = 0.0f, ay = 0.0f, az = 0.0f, Lsum = 0.0f;
    if (staged) {
        mbar_wait(smem0 + L::OFF_MBAR, 0);
        if (valid) pass_b6_neighbours<L, T, STEP, true>(g, a, cell_start, key, smem0, 3, 0, pi, vi, Vm_i, si.x, ax, ay, az, Lsum);
    } else if (valid) {
        pass_b6_neighbours<L, T, STEP, false>(g, a, cell_start, key, smem0, 3, 0, pi, vi, Vm_i, si.x, ax, ay, az, Lsum);
    }
    if (live) pass_b_finish<DIAG, EGM>(p, a, Pout, i, pi, vi, e4, si.y, fixed, ax, ay, az, Lsum, inv_mass, next_keys, next_rank, cell_count);
}

}  // namespace sphsm
