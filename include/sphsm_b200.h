/* sphsm_b200.h — the C-ABI of libsphsm_b200.so: the B200 (sm_100a) implementation of the
 * SPH_SM_monodomain per-timestep particle pipeline.
 *
 * This is the ONLY boundary between host code and CUDA: the drop-in C++ class in
 * include/SPH_SM_monodomain.h, the ctypes binding in sph_sm_monodomain_b200/_capi.py, the tests and
 * bench.py all call exactly these entry points; nothing else touches the device.  Plain pointers and
 * sizes, no C++/torch types.  Each entry point cites the reference interface it replaces ("h" =
 * SPH_SM_monodomain/SPH_SM_monodomain.h, "cpp" = SPH_SM_monodomain/SPH_SM_monodomain.cpp of
 * Hagen23/SPH-SM-Monodomain).
 *
 * Conventions: every function returns 0 (SPHSM_OK) or a negative sphsm_status and never throws or aborts
 * across the ABI; sphsm_last_error() gives the message of the last failure on that handle (or of the last
 * failed sphsm_create when h == NULL).  A handle owns its device memory, stream and CUDA graph; calls are
 * asynchronous on the handle's stream except download / get_* / sync, which synchronise.  One host thread
 * per handle.  There is NO CPU fallback: without a usable CUDA device sphsm_create fails with
 * SPHSM_ERR_CUDA.
 */
#ifndef SPHSM_B200_H
#define SPHSM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPHSM_ABI_VERSION 1

typedef enum {
    SPHSM_OK = 0,
    SPHSM_ERR_INVALID = -1,  /* bad argument / bad state */
    SPHSM_ERR_CUDA = -2,     /* CUDA runtime error (message in sphsm_last_error) */
    SPHSM_ERR_CAPACITY = -3, /* more particles than params.capacity */
    SPHSM_ERR_COMM = -4      /* NCCL / multi-GPU error */
} sphsm_status;

/* Stage ids: the call order of compute_SPH_SM_monodomain, cpp:794-824. */
typedef enum {
    SPHSM_STAGE_STEP = 0,                   /* Animation(), cpp:826-829 */
    SPHSM_STAGE_FIND_NEIGHBORS = 1,         /* Find_neighbors, cpp:199-213 */
    SPHSM_STAGE_CORRECTED_VELOCITY = 2,     /* calculate_corrected_velocity, cpp:653-667 (+215-446) */
    SPHSM_STAGE_INTERMEDIATE_VELOCITY = 3,  /* calculate_intermediate_velocity, cpp:669-701 */
    SPHSM_STAGE_DENSITY_PRESSURE = 4,       /* Compute_Density_SingPressure, cpp:448-513 */
    SPHSM_STAGE_CELL_MODEL = 5,             /* calculate_cell_model, cpp:575-593 */
    SPHSM_STAGE_FORCE = 6,                  /* Compute_Force, cpp:515-573 */
    SPHSM_STAGE_UPDATE = 7,                 /* Update_Properties, cpp:598-651 */
    /* the two public sub-steps of stage 2 (h:127-129); sphsm_step never issues them separately */
    SPHSM_STAGE_EXTERNAL_FORCES = 8,        /* apply_external_forces, cpp:215-232: predicted_vel only */
    SPHSM_STAGE_PROJECT_POSITIONS = 9       /* projectPositions, cpp:234-446: mGoalPos only */
} sphsm_stage_id;

/* Every tunable the reference hard-codes in its ctor (cpp:13-69) or in-class initialisers (h:72-94).
 * sphsm_default_params() fills in the reference's values bit-for-bit. */
typedef struct {
    uint32_t struct_size;   /* = sizeof(sphsm_params); checked by sphsm_create */
    int32_t device;         /* CUDA device ordinal */
    int32_t capacity;       /* Max_Number_Paticles, cpp:19 (50000) */
    float world[3];         /* World_Size, cpp:29 (1.5,1.5,1.5); also the SM bounds max, cpp:61 */
    float kernel_h;         /* kernel == Cell_Size, cpp:17,31 (0.04f) */
    float gravity[3];       /* cpp:39 */
    float K;                /* cpp:40 */
    float stand_density;    /* cpp:41 */
    float time_delta;       /* cpp:47 */
    float wall_hit;         /* cpp:48 */
    float mu;               /* cpp:49 */
    float velocity_mixing;  /* cpp:43 */
    float poly6_constant;   /* cpp:54 */
    float spiky_constant;   /* cpp:55 */
    float bspline_constant; /* cpp:57 */
    float alpha, beta;      /* cpp:64-65 */
    int32_t quadratic_match;     /* cpp:67 */
    int32_t volume_conservation; /* cpp:68 */
    int32_t allow_flip;          /* cpp:69 */
    float Cm, Beta, sigma;  /* cpp:23-26 */
    float stim_strength;    /* cpp:27 */
    float FH_Vt, FH_Vp, FH_Vr, C1, C2, C3, C4; /* h:72-80 */
    float voltage_constant, max_pressure, max_voltage; /* h:92-94 */
    float particle_mass;    /* Init_Particle, cpp:116 (0.2f) */
    /* --- implementation controls (no reference counterpart) --- */
    int32_t diagnostics;    /* 1: every step also materialises the reference's intermediate Particle fields
                               (predicted_vel, goal, corrected_vel, inter_vel, acc, pres, Inter_Vm) so that
                               sphsm_download_aos returns all 33 fields exactly as Get_Paticles() would show
                               them; 0: only persistent state is kept current (fused fast path). */
    int32_t strict;         /* 1: reference-order arithmetic (no FMA contraction, sequential float moment sums,
                               double where the reference promotes) for bit-level validation at small N;
                               0: the production path. */
    int32_t slab_axis;      /* multi-GPU: axis (0,1,2) the domain is cut along; also the slowest-varying axis of
                               the internal cell key. -1: single-GPU reference key order (x fastest). */
    int32_t reserved[8];    /* tuning / validation switches, 0 = default everywhere:
                               [0] multi-GPU: particles per halo / migrant message (default: 2.5 x the mean cell-plane
                                   population at capacity + 4096)
                               [1] 1: canonical in-cell order (ascending original index) in EVERY cell of a slab rank, not
                                   only next to the slab faces (bit-level comparison against the single-GPU run)
                               [2] neighbour-grid sort: 1 = LSD radix sort, 2 = counting sort (default: by grid size)
                               [3] unused
                               [4] 1: no CUDA-graph replay of small single-GPU steps
                               [5..7] unused */
} sphsm_params;

typedef struct sphsm_handle sphsm_handle;

/* Same field order/size/padding as the reference's `Particle` (Particle.h:7-35): 132 bytes. */
#define SPHSM_PARTICLE_STRIDE 132

int sphsm_abi_version(void);

/* ctor defaults, cpp:13-79 + h:72-94.  world/capacity may then be changed before sphsm_create (the derived
 * Grid_Size / Number_Cells, cpp:32-37, follow from world and kernel_h). */
int sphsm_default_params(sphsm_params *p);

/* SPH_SM_monodomain::SPH_SM_monodomain() / ~SPH_SM_monodomain(), cpp:13-85 */
int sphsm_create(const sphsm_params *p, sphsm_handle **out);
int sphsm_destroy(sphsm_handle *h);

/* Live parameter changes: add_viscosity (cpp:87-91), flip_quadratic / flip_volume (h:154-155), the public
 * voltage_constant / max_pressure / max_voltage (h:92-94).  world, kernel_h, capacity, device are fixed at create. */
int sphsm_get_params(sphsm_handle *h, sphsm_params *out);
int sphsm_set_params(sphsm_handle *h, const sphsm_params *p);

/* Init_Fluid(std::vector<m3Vector>) / Init_Particle, cpp:93-125: APPENDS n particles (pos = orig = goal,
 * vel = 0, dens = Stand_Density, mass = particle_mass, Vm = Iion = stim = w = 0); particles beyond capacity are
 * silently dropped exactly as cpp:103 does (the return value stays SPHSM_OK). xyz: n*3 floats. */
int sphsm_init_fluid(sphsm_handle *h, const float *xyz, int n);

/* Whole-array state exchange with the caller's Particle[] (Get_Paticles(), h:150).  `stride` is the byte
 * distance between consecutive particles (SPHSM_PARTICLE_STRIDE for the reference layout).  upload replaces the
 * simulation state with n particles; download writes all 33 fields of the first n particles in the caller's
 * (original) particle order. */
int sphsm_upload_aos(sphsm_handle *h, const void *particles, int n, int stride);
int sphsm_download_aos(sphsm_handle *h, void *particles, int n, int stride);
/* pos (3 floats per particle, original order) only — what main.cpp's display_points reads every frame. */
int sphsm_download_positions(sphsm_handle *h, float *xyz, int n);

/* set_stim(center, radius, strength), cpp:704-717 — NB squared distance is compared with `radius`. */
int sphsm_set_stim(sphsm_handle *h, float cx, float cy, float cz, float radius, float strength);
/* turnOnStim_Mesh / turnOnStim_Cube, cpp:745-762 / 719-743 (one fused device pass over positions x particles
 * instead of the reference's per-position set_stim loop; same result). xyz: n*3 floats. */
int sphsm_stim_mesh(sphsm_handle *h, const float *xyz, int n);
int sphsm_stim_cube(sphsm_handle *h, const float *xyz, int n);
/* turnOffStim, cpp:764-783 */
int sphsm_stim_off(sphsm_handle *h);
/* set_stim (cpp:704-717) for every particle inside the axis-aligned box [lo, hi]: what turnOnStim_Cube's loop of set_stim calls
 * over a block of positions amounts to, as one O(N) kernel (pacing protocols stimulate an end slab every few steps). */
int sphsm_set_stim_box(sphsm_handle *h, const float lo[3], const float hi[3], float strength);
/* Overwrite the per-particle fixed flags / stimulation values (original particle order, n entries each; either
 * pointer may be NULL).  The reference's callers do this by writing through Get_Paticles(). */
int sphsm_set_masks(sphsm_handle *h, const uint8_t *fixed, const float *stim, int n);

/* Animation() x nsteps, cpp:826-829 */
int sphsm_step(sphsm_handle *h, int nsteps);
/* One stage of the step (the reference exposes them as public methods, h:120-143).  Stages 3, 4 and 6 rebuild
 * the neighbour grid first if the particle data changed since it was last built. */
int sphsm_stage(sphsm_handle *h, int stage);
int sphsm_sync(sphsm_handle *h);

/* Asynchronous forms of the per-frame I/O (what main.cpp does through Get_Paticles() every frame: write stim / fixed,
 * read pos).  They return once the work is queued: the host arrays should be page-locked (otherwise the copies do not
 * overlap) and must not be touched until sphsm_io_wait or sphsm_sync returns.  Copies run on dedicated streams in both
 * directions while the compute stream keeps stepping; each call orders itself after the previous call of its kind. */
int sphsm_set_masks_async(sphsm_handle *h, const uint8_t *fixed, const float *stim, int n);
int sphsm_download_positions_async(sphsm_handle *h, float *xyz, int n);
/* (multi-GPU: the owned range is only known on the device, so up to `cap` records cross and *count is written with them:
 * like the arrays it is valid once sphsm_io_wait or sphsm_sync has returned; `count` should point into page-locked memory) */
int sphsm_download_owned_async(sphsm_handle *h, int *ids, float *xyz, int cap, int *count);
/* Stimulation input for the particles this rank owns: stim[k] belongs to the k-th particle of the most recent
 * sphsm_download_owned_async on this handle (4 bytes per owned particle; the multi-GPU form of the per-step mask upload). */
int sphsm_set_stim_owned_async(sphsm_handle *h, const float *stim, int count);
int sphsm_io_wait(sphsm_handle *h);

/* Snapshot / restart (the reference has none).  The file holds the tunable parameters and every particle in the
 * reference's Particle layout (SPHSM_PARTICLE_STRIDE bytes, all 33 fields, original order) plus the step counter;
 * sphsm_load_state restores them into an existing handle of sufficient capacity and the same world / kernel size. */
int sphsm_save_state(sphsm_handle *h, const char *path);
int sphsm_load_state(sphsm_handle *h, const char *path);

int sphsm_num_particles(sphsm_handle *h);  /* Get_Particle_Number, h:148 */
int sphsm_num_cells(sphsm_handle *h);      /* Number_Cells, cpp:37 */
int sphsm_grid_size(sphsm_handle *h, int out3[3]); /* Grid_Size, cpp:32-35 */
int sphsm_total_time_steps(sphsm_handle *h);       /* total_time_steps, h:101 */

/* Accumulated device time (seconds) of the seven stages in the order of the d_* members (h:99):
 * find_neighbors, corrected_velocity, intermediate_velocity, Density_SingPressure, cell_model, compute_Force,
 * Update_Properties.  Only filled while stage timing is enabled (it serialises the step with CUDA events). */
int sphsm_enable_stage_timing(sphsm_handle *h, int on);
int sphsm_get_stage_times(sphsm_handle *h, double out7[7]);

/* Buckets after Find_neighbors as CSR in the REFERENCE's hash order (cpp:136-146): cell_start has
 * sphsm_num_cells()+1 entries, indices has sphsm_num_particles() entries of original particle indices
 * (ascending inside a bucket, as the reference's push_back order yields). */
int sphsm_get_cells_csr(sphsm_handle *h, int *cell_start, int *indices);
/* Neighbour sets computed ON THE DEVICE by the same traversal the passes use, for the first n_query original
 * particle indices in `query`: kind 0 = candidate set (27 cells); 1 = {r2 <= h*h} (Poly6); 2 = {r2 > 1e-12 &&
 * r <= h} (Spiky/Visco); 3 = {r2 > 1e-12 && r/h < 2} (B_spline_2).  counts[n_query]; indices[n_query*cap] holds
 * original particle indices sorted ascending. */
int sphsm_get_neighbor_sets(sphsm_handle *h, int kind, const int *query, int n_query, int cap, int *counts, int *indices);

/* Shape-matching internals of the last calculate_corrected_velocity: cm[3], original cm[3], and the transform
 * (27 floats: the linear T in [0..8], or the quadratic 3x9 matrix). */
int sphsm_get_sm_transform(sphsm_handle *h, float cm[3], float ocm[3], float xform[27]);

/* Counters for bench.py: kernels launched by this handle since creation / since the last reset. */
int sphsm_get_launch_count(sphsm_handle *h, long long *launches);
int sphsm_reset_launch_count(sphsm_handle *h);
/* Device time (ms, CUDA events on the handle's stream) of the last sphsm_step call's nsteps steps in total. */
int sphsm_last_step_ms(sphsm_handle *h, float *ms);
/* A device-side stopwatch over any sequence of calls: sphsm_timer_mark(h, 0) ... sphsm_timer_mark(h, 1), then sphsm_timer_ms
 * gives the device time of everything queued on the handle's stream between the two marks. */
int sphsm_timer_mark(sphsm_handle *h, int which);
int sphsm_timer_ms(sphsm_handle *h, float *ms);
/* Average device time (ms per launch) of each kernel group inside the last profiled step, see bench.py. */
#define SPHSM_NUM_KERNEL_GROUPS 8
int sphsm_profile_step(sphsm_handle *h, int nsteps, float out_ms[SPHSM_NUM_KERNEL_GROUPS]);
const char *sphsm_kernel_group_name(int group);

/* ---- multi-GPU (one process per GPU; slab decomposition along params.slab_axis; no reference counterpart) ------ */
/* Protocol: every rank creates its handle with the same GLOBAL capacity / world and slab_axis = the longest axis, uploads
 * the same global particle set (init_fluid / upload_aos / set_masks ...), then:
 *   rank 0: sphsm_comm_unique_id(id) -> share the 128 bytes by any means (bench.py: torch.distributed broadcast)
 *   all:    sphsm_comm_init(h, nranks, rank, id); sphsm_comm_set_slab(h, lo, hi)   (rank r owns cell planes [lo, hi))
 * From then on sphsm_step includes the halo / migrant exchange (ncclSend / ncclRecv with the two slab neighbours) and
 * the shape-matching moment allreduce, particle ids stay global, and download_aos / download_positions write only the
 * particles this rank owns (n = global count).  params.reserved[0] overrides the per-message halo capacity.
 * The step never waits for the host: a step error (halo message overflow, a particle crossing two cell planes) is returned by
 * sphsm_step on EVERY rank at the same step, two to three steps after it happened.  Calls that change particle state between
 * steps (set_masks*, stim_*, set_stim*, uploads) are COLLECTIVE in slab mode: all ranks issue the same calls in the same order
 * (the next step's halo exchange may already be under way and is repeated on every rank alike when such a call voids it).
 * NCCL is resolved at run time (dlopen "libnccl.so.2", or $SPHSM_NCCL_LIB). */
int sphsm_comm_unique_id(void *id128);
int sphsm_comm_init(sphsm_handle *h, int nranks, int rank, const void *id128);
int sphsm_comm_set_slab(sphsm_handle *h, int cell_lo, int cell_hi);
/* out: [0] comm mode (0 none, 1 NCCL, 2 local group) [1] nranks [2] rank [3] local slots (owned + halo)
 *      [4] first owned slot [5] end of owned slots [6] halo message capacity [7] slab mode on */
int sphsm_comm_info(sphsm_handle *h, int out8[8]);
/* Exchange-1 message capacities (particles) of the exchange packed last: [0] to left [1] to right [2] from left [3] from right.
 * The halo capacity, unless sphsm_tune("x1_dynamic", 1) / SPHSM_X1_DYNAMIC=1 (every rank alike) lets the ncclSend / ncclRecv messages
 * follow the face populations of three exchanges earlier (a quarter + 2048 particles of margin; full capacity after every upload /
 * new slab): for particle sets whose face populations change smoothly — a regular lattice moves whole planes at once. */
int sphsm_comm_x1_sizes(sphsm_handle *h, int out4[4]);
/* Bit 0: exchange 1 of the NCCL mode runs as the push exchange — the packing kernel stores the halo / migrant records straight into
 * the neighbour's receive slot (CUDA IPC mapping over NVLink) and a flag word publishes them.  Bit 1: the small allreduces of the
 * step (moment sums + error flag) run as the push allreduce — one kernel stores the rank's values into every rank's landing area,
 * waits for the others' and adds them in rank order.  0: ncclSend / ncclRecv / ncclAllReduce (a peer could not be mapped, more than
 * 32 ranks, or some rank runs with SPHSM_P2P=0 / SPHSM_P2P_RED=0 — decided once, for all ranks, inside sphsm_comm_init). */
int sphsm_comm_p2p(sphsm_handle *h);
/* Compact read-back of the owned particles: original ids and positions (3 floats each); *count = owned particles. */
int sphsm_download_owned(sphsm_handle *h, int *ids, float *xyz, int cap, int *count);
/* Virtual ranks for testing the slab logic on ONE device: nranks handles (same device, capacity, world, slab_axis) form
 * a local group whose collectives are device copies; after sphsm_comm_set_slab on each, sphsm_step_group advances all of
 * them in lockstep through the same phases the NCCL path runs. */
int sphsm_comm_init_local(sphsm_handle **handles, int nranks);
int sphsm_step_group(sphsm_handle **handles, int nranks, int nsteps);

/* ---- recorder of the membrane-potential wave (no reference counterpart) ------------------------------------------------
 * Activation / recovery time maps and probe traces ("virtual electrodes") of Vm, kept on the device by one small kernel at the
 * end of every step, so that watching the wave costs a few bytes per particle per step instead of a download of every particle.
 *
 * Recording is off by default; while it is off nothing is allocated and the step launches nothing extra.  While it is on, every
 * step that advances total_time_steps records that step, on every step path (fused, CUDA-graph replay, strict, staged with stage
 * timing, sphsm_profile_step, the NCCL slab step, sphsm_step_group); a stand-alone sphsm_stage(1..9) records nothing.  The step
 * index is total_time_steps after the step (the first step of a fresh handle is step 1).
 *
 * For each particle the step integrates, pre = the Vm the step started from (after any call made between steps, e.g. turnOffStim
 * zeroing Vm) and post = the Vm the step produced:
 *   upstroke    pre <  vm_up   && post >= vm_up    first_up = step if unset, last_up = step, n_up += 1
 *   downstroke  pre >= vm_down && post <  vm_down  last_down = step
 * A change of Vm made between steps (turnOffStim, uploads, set_masks) is not a crossing.  The rule has no state: in slab mode each
 * crossing is seen by exactly one rank (the one that integrated the particle in that step), and per-rank maps merge exactly:
 * first_up by minimum over set values, last_up / last_down by maximum, n_up by sum (sph_sm_monodomain_b200.slabs.merge_activation).
 *
 * Probes: up to SPHSM_RECORD_MAX_PROBES distinct original particle ids in [0, particle count) (the global count in slab mode),
 * fixed when recording starts.  At every recorded step each rank stores (pos.xyz, Vm) after the step for the probes it integrated,
 * in a ring of trace_rows rows (trace_rows * n_probes <= SPHSM_RECORD_MAX_TRACE_ENTRIES).  Each entry has an owned flag set only by
 * the rank that wrote it, so ranks merge exactly (slabs.merge_traces).  Recording never pauses while it is on: the rows held are
 * the last min(trace_rows, steps recorded) consecutive steps.
 *
 * Lifetime: sphsm_record_start (re)configures and clears; sphsm_record_stop and sphsm_destroy free the buffers; sphsm_record_reset
 * clears the data and keeps the configuration; sphsm_load_state clears the data too (numbering continues at the snapshot's step
 * counter + 1).  In slab mode every rank issues the recorder calls alike, like the state mutators; none of them is collective.
 * Errors: SPHSM_ERR_INVALID for reversed or non-finite thresholds, duplicate or out-of-range probe ids, trace_rows <= 0 with
 * probes, a size over the bounds below, and for reading or resetting while recording is off. */
#define SPHSM_RECORD_MAX_PROBES 65536
#define SPHSM_RECORD_MAX_TRACE_ENTRIES (1 << 24)
int sphsm_record_start(sphsm_handle *h, float vm_up, float vm_down, const int *probe_ids, int n_probes, int trace_rows);
int sphsm_record_stop(sphsm_handle *h);
int sphsm_record_reset(sphsm_handle *h);
/* The maps in original particle order, n entries each (n <= capacity; the particle count, global in slab mode); unset steps
 * are -1.  A null array is skipped.  Synchronises. */
int sphsm_get_activation(sphsm_handle *h, int *first_up, int *last_up, int *last_down, int *n_up, int n);
/* Up to max_rows of the most recent trace rows, oldest first: *rows rows starting at step *first_step; xyzv[rows * n_probes * 4]
 * = (pos.xyz, Vm) in probe order, owned[rows * n_probes] = 1 where this rank wrote the entry (0: entry zeroed).  Synchronises. */
int sphsm_get_probe_trace(sphsm_handle *h, int max_rows, int *rows, int *first_step, float *xyzv, uint8_t *owned);

/* ---- extracellular electrograms at virtual electrodes (no reference counterpart) ----------------------------------------
 * The extracellular potential a fixed electrode sees (a pseudo-ECG, or a surface EMG for the biceps model), summed over every
 * particle on the device each step, so that it costs 20 bytes per particle per step instead of a download of every particle.
 * For step s, each particle i the step integrated and each electrode e:
 *   q_i      = vol_i * L_i        L_i = sum_j vol_j (Vm_j - Vm_i) B2(r_ij): the SPH Laplacian sum step s adds into Inter_Vm
 *                                 (cpp:563), on the configuration and Vm the step started from; vol = mass / dens with the
 *                                 density step s computed
 *   phi_e(s) = gain * sum_i q_i / sqrt(|x_i - e|^2 + softening^2)
 * x_i is the position the step started from.  This is the discrete pseudo-ECG integral (Plonsey; Gima & Rudy), phi =
 * 1/(4 pi sigma_e) * integral of div(sigma_i grad Vm) / r dV, up to the caller's `gain`; no unit conversion is applied.  The
 * softening length (> 0) keeps an electrode inside the tissue finite.  Electrodes stay fixed in space while the tissue moves.
 *
 * Off by default; while off nothing is allocated and the step launches nothing extra.  While on, every step path (as for the
 * recorder above) ends with one extra launch and writes one row of n_electrodes doubles into a ring of `rows` rows; a
 * stand-alone sphsm_stage(1..9) writes no row.  Rows are numbered like the recorder's steps (total_time_steps after the step),
 * and with both on they number every step alike.  The electrograms are independent of the recorder: either can be on alone.
 * On one device the values are bit-reproducible (fixed summation order, no atomics), graph replay or not.
 *
 * Lifetime: sphsm_egm_start (re)configures and clears; sphsm_egm_stop and sphsm_destroy free; sphsm_egm_reset clears the rows;
 * sphsm_load_state clears them too (numbering continues at the snapshot's step counter + 1).  In slab mode each rank holds the
 * partial sum over the particles it integrated (sum the ranks' rows, sph_sm_monodomain_b200.slabs.merge_electrograms); every
 * rank issues the calls alike, and none of them is collective.
 * Errors: SPHSM_ERR_INVALID for n_electrodes outside [1, SPHSM_EGM_MAX_ELECTRODES], non-finite coordinates or gain, a
 * softening that is not positive and finite, rows <= 0 or rows * n_electrodes > SPHSM_RECORD_MAX_TRACE_ENTRIES, and for
 * reading or resetting while off. */
#define SPHSM_EGM_MAX_ELECTRODES 256
/* xyz[3 * n_electrodes]: the electrodes' positions in world coordinates */
int sphsm_egm_start(sphsm_handle *h, const float *xyz, int n_electrodes, float gain, float softening, int rows);
int sphsm_egm_stop(sphsm_handle *h);
int sphsm_egm_reset(sphsm_handle *h);
/* up to max_rows of the most recent rows, oldest first: *rows rows from step *first_step; phi[rows * n_electrodes].  Synchronises. */
int sphsm_get_egm(sphsm_handle *h, int max_rows, int *rows, int *first_step, double *phi);

/* Process-wide switches for tests and tuning (no reference counterpart); the first value is the default:
 *   "warp_path"  = 1 | 0  0: small dense sets take the thread-per-particle neighbour passes too (changes the order of the
 *                         floating-point sums);
 *   "x1_dynamic" = 0 | 1  1: the ncclSend / ncclRecv messages of exchange 1 follow the face populations (sphsm_comm_x1_sizes;
 *                         every rank alike).
 * Both are read once from $SPHSM_WARP_PATH and $SPHSM_X1_DYNAMIC.  Any other name or value returns SPHSM_ERR_INVALID. */
int sphsm_tune(const char *name, int value);

const char *sphsm_last_error(sphsm_handle *h);

#ifdef __cplusplus
}
#endif
#endif /* SPHSM_B200_H */
