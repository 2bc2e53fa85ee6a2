// sphsm_record.cuh — on-device recorder of the membrane-potential wave: activation / recovery time maps and probe traces.
//
// k_record runs once per step, on the compute stream right after the kernel that integrated the particles (pass B, or k_update
// of the staged step), over the slots this rank integrated: [0, n) on one GPU, the owned range of SlabMeta::rng_all in the slab
// step.  At that point every such slot holds both values of its particle's Vm:
//   PB.w  the Vm the step started from (written by the gather of this step: k_reorder / k_reorder_goal, or k_refresh_derived
//         in stage 6 of the staged step), i.e. after any call made between steps (turnOffStim, uploads, masks)
//   E.x   the Vm the step produced
// and nothing moves the slots again before the step ends.  The crossing rule needs only that pair:
//   upstroke    pre <  vm_up   && post >= vm_up    -> first_up (if unset), last_up = step, n_up += 1
//   downstroke  pre >= vm_down && post <  vm_down  -> last_down = step
// with step = total_time_steps after the step (the first recorded step of a fresh handle is 1).  The rule is stateless, so in
// slab mode each crossing is seen by exactly one rank (the one that integrated the particle in that step), nothing travels with
// migrants, and per-rank maps merge exactly (first_up: min over set values, last_up / last_down: max, n_up: sum).  A change of
// Vm made between steps is not a crossing.
//
// Probes: probe_of[id] = k for the k-th probe, -1 otherwise.  The entry of probe k at step s is trace[(s % rows) * K + k] =
// (pos.xyz, Vm) after the step, and stamp[...] = s marks it as written by this rank for that step (a ring row holds data of
// step s only where its stamp says s, so ranks merge exactly and nothing needs clearing between steps).
//
// The step number comes from device memory, not from a kernel argument (a replayed CUDA graph reuses its captured arguments):
// ctl[0] is total_time_steps before the step (set by the host when recording starts or the host counter changes outside a
// step).  The counter is shared with the electrograms (sphsm_egm.cuh) and advanced once per step by the last kernel of the
// step's hook: here (advance = 1) when electrograms are off, the last block to finish (ticket in ctl[1]) advancing it; k_egm
// otherwise.  One launch per step.
#pragma once
#include "sphsm_pass4.cuh"
#include "sphsm_types.cuh"

namespace sphsm {

struct RecArgs {
    int *first_up, *last_up, *last_down, *n_up;  // by original id; steps unset = -1
    const int *probe_of;                          // nullptr: no probes
    float4 *trace;                                // rows x n_probes
    int *stamp;                                   // rows x n_probes: the step that wrote the entry
    int n_probes, rows;
    float vm_up, vm_down;
    unsigned *ctl;                                // [0] steps recorded up to (= total_time_steps), [1] ticket
    int advance;                                  // 1: this launch advances ctl[0] (0: k_egm follows and does)
};

constexpr int REC_THREADS = 256;

// rng != nullptr: slot range from device memory (slab step), `count` bounds it; otherwise p.own_begin .. p.own_end
__global__ void __launch_bounds__(REC_THREADS) k_record(const __grid_constant__ DevParams p, const int *__restrict__ rng, int count,
                                                        const int *__restrict__ ID, const float4 *__restrict__ PB,
                                                        const float4 *__restrict__ E, const float4 *__restrict__ P, RecArgs r) {
    const int step = (int)r.ctl[0] + 1;
    const int k = blockIdx.x * REC_THREADS + threadIdx.x;
    const int i = k < count ? launch_slot(launch_range(p, rng), k) : -1;
    if (i >= 0) {
        const int id = ID[i];
        if (id >= 0) {
            const float pre = PB[i].w, post = E[i].x;
            if (pre < r.vm_up && post >= r.vm_up) {
                if (r.first_up[id] < 0) r.first_up[id] = step;
                r.last_up[id] = step;
                r.n_up[id] += 1;
            }
            if (pre >= r.vm_down && post < r.vm_down) r.last_down[id] = step;
            if (r.probe_of) {
                const int q = r.probe_of[id];
                if (q >= 0) {
                    const float4 x = P[i];
                    const size_t e = (size_t)(step % r.rows) * r.n_probes + q;
                    r.trace[e] = make_float4(x.x, x.y, x.z, post);
                    r.stamp[e] = step;
                }
            }
        }
    }
    // last block out advances the step counter (every block has read it by then)
    if (!r.advance) return;
    __shared__ bool last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        last = atomicAdd(&r.ctl[1], 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        r.ctl[0] = (unsigned)step;
        r.ctl[1] = 0u;
    }
}

// probe_of[ids[k]] = k (the rest of probe_of was set to -1)
__global__ void k_record_probes(const int *__restrict__ ids, int n, int *__restrict__ probe_of) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k < n) probe_of[ids[k]] = k;
}

}  // namespace sphsm
