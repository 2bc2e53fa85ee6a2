// sphsm_egm.cuh — extracellular electrograms (pseudo-ECG / surface EMG) at fixed virtual electrodes, reduced on the device.
//
// For every step s, every particle i the step integrated and every electrode e (a fixed point in world coordinates):
//   q_i      = vol_i * L_i                        source strength: L_i is the SPH Laplacian sum of Vm that pass B adds into
//                                                 Inter_Vm (cpp:563), vol_i = m_i / dens_i with the step's new density
//   phi_e(s) = gain * sum_i q_i / sqrt(|x_i - e|^2 + eps^2)
// with x_i = PB.xyz, the configuration L_i was evaluated on.  This is the discrete pseudo-ECG integral (Plonsey; Gima & Rudy),
// phi = 1/(4 pi sigma_e) * integral of div(sigma_i grad Vm) / r dV, up to the caller's constant `gain`; eps > 0 keeps an
// electrode inside the tissue finite.
//
// Pass B stores q_i into the dense array Arrays::Q while electrograms are on (its EGM variants); k_egm runs once per step
// after the kernel that integrated the step, over the same slots ([0, n) on one GPU, SlabMeta::rng_all in the slab step), and
// reads 20 bytes per particle (PB.xyz, Q).  Its design, for bandwidth and a fixed summation order:
//   - a persistent grid (EGM_BLOCKS_PER_SM blocks per SM, grid-stride); each thread loads EGM_SLOTS slots before using any of them
//   - the electrodes are staged in shared memory
//   - per electrode, a thread's float terms over its slots are summed by a fixed xor-butterfly across the warp and added into the
//     warp's double row in shared memory (one row per warp, chunks in grid-stride order)
//   - the rows are summed in warp order into partial[block][e]; the last block to finish (ticket) sums the partials in block
//     order into the ring row of step s.
// No float atomics: the result is bit-reproducible for a given grid, which the host fixes from the handle's state.  In slab mode
// each rank holds the partial sum over the particles it integrated (merged by summation in rank order on the host).
//
// The step number comes from the device step counter shared with the recorder (sphsm_record.cuh): ctl[0] is total_time_steps
// before the step; k_egm runs last in the step's hook and its last block advances it.
#pragma once
#include "sphsm_pass4.cuh"
#include "sphsm_pass4w.cuh"
#include "sphsm_types.cuh"

namespace sphsm {

constexpr int EGM_MAX_ELECTRODES = 256;  // SPHSM_EGM_MAX_ELECTRODES
constexpr int EGM_THREADS = 256;
constexpr int EGM_WARPS = EGM_THREADS / 32;
constexpr int EGM_SLOTS = 8;  // slots per thread loaded before use (8 x 20 B in flight per thread)
constexpr int EGM_BLOCKS_PER_SM = 2;

struct EgmArgs {
    const float4 *el;  // n_el electrodes (x, y, z, -)
    int n_el, rows;
    float gain, eps2;  // eps2 = softening^2
    double *partial;   // grid x n_el: per-block sums of the current step
    double *ring;      // rows x n_el: phi of step s in row s % rows
    unsigned *ctl;     // [0] the step counter (total_time_steps before the step), [1] ticket
};

// rng != nullptr: slot range from device memory (slab step), `count` bounds it; otherwise p.own_begin .. p.own_end
__global__ void __launch_bounds__(EGM_THREADS, EGM_BLOCKS_PER_SM) k_egm(const __grid_constant__ DevParams p, const int *__restrict__ rng, int count,
                                                                        const float4 *__restrict__ PB, const float *__restrict__ Q, EgmArgs g) {
    __shared__ float4 s_el[EGM_MAX_ELECTRODES];
    __shared__ double s_acc[EGM_WARPS][EGM_MAX_ELECTRODES];
    __shared__ bool last;
    const int E = g.n_el, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int e = threadIdx.x; e < E; e += EGM_THREADS) s_el[e] = g.el[e];
    for (int e = threadIdx.x; e < EGM_WARPS * EGM_MAX_ELECTRODES; e += EGM_THREADS) (&s_acc[0][0])[e] = 0.0;
    __syncthreads();
    const Range4 r = launch_range(p, rng);
    const int chunk = EGM_THREADS * EGM_SLOTS;
    for (int base = blockIdx.x * chunk; base < count; base += gridDim.x * chunk) {
        float x[EGM_SLOTS], y[EGM_SLOTS], z[EGM_SLOTS], q[EGM_SLOTS];
#pragma unroll
        for (int s = 0; s < EGM_SLOTS; s++) {
            const int k = base + s * EGM_THREADS + threadIdx.x;
            const int i = k < count ? launch_slot(r, k) : -1;
            float4 pb = make_float4(0.f, 0.f, 0.f, 0.f);
            float qi = 0.f;
            if (i >= 0) {
                pb = __ldcs(PB + i);
                qi = __ldcs(Q + i);
            }
            const bool src = qi != 0.f;  // (a slot without source adds nothing, whatever its position: limbo slots hold NaN)
            x[s] = src ? pb.x : 0.f;
            y[s] = src ? pb.y : 0.f;
            z[s] = src ? pb.z : 0.f;
            q[s] = qi;
        }
#pragma unroll 1
        for (int e = 0; e < E; e++) {
            const float4 el = s_el[e];
            float t = 0.f;
#pragma unroll
            for (int s = 0; s < EGM_SLOTS; s++) {
                const float dx = x[s] - el.x, dy = y[s] - el.y, dz = z[s] - el.z;
                const float d2 = fmaf(dx, dx, fmaf(dy, dy, fmaf(dz, dz, g.eps2)));
                t = fmaf(q[s], rsqrtf(d2), t);
            }
            t = warp_sum(t);
            if (lane == 0) s_acc[warp][e] += (double)t;
        }
    }
    __syncthreads();
    for (int e = threadIdx.x; e < E; e += EGM_THREADS) {
        double b = 0.0;
#pragma unroll
        for (int w = 0; w < EGM_WARPS; w++) b += s_acc[w][e];
        g.partial[(size_t)blockIdx.x * E + e] = b;
    }
    // the last block out sums the partials in block order and advances the step counter (every block has read it by then)
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = atomicAdd(&g.ctl[1], 1u) == gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    const int step = (int)__ldcg(g.ctl) + 1;
    for (int e = threadIdx.x; e < E; e += EGM_THREADS) {
        double s = 0.0;
        for (int b = 0; b < (int)gridDim.x; b++) s += __ldcg(g.partial + (size_t)b * E + e);
        g.ring[(size_t)(step % g.rows) * E + e] = (double)g.gain * s;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        g.ctl[0] = (unsigned)step;
        g.ctl[1] = 0u;
    }
}

}  // namespace sphsm
