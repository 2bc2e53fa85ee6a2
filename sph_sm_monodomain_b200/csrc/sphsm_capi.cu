// sphsm_capi.cu — libsphsm_b200.so: handle, step orchestration and the extern "C" entry points declared in
// include/sphsm_b200.h.  All device work is in the hand-written sm_100a kernels of sphsm_{sort,sm,pass}.cuh;
// there is no CPU fallback anywhere in this file.
#include "../../include/sphsm_b200.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <algorithm>
#include <string>
#include <unordered_set>
#include <vector>

#include "sphsm_comm.cuh"
#include "sphsm_egm.cuh"
#include "sphsm_pass.cuh"
#include "sphsm_pass4.cuh"
#include "sphsm_pass4w.cuh"
#include "sphsm_record.cuh"
#include "sphsm_sm.cuh"
#include "sphsm_sort.cuh"
#include "sphsm_types.cuh"

using namespace sphsm;

// byte offsets inside the reference's Particle (Particle.h:10-29)
enum : int {
    OFF_POS = 0, OFF_VEL = 12, OFF_PVEL = 24, OFF_IVEL = 36, OFF_CVEL = 48, OFF_ACC = 60, OFF_MASS = 72, OFF_ORIG = 76,
    OFF_GOAL = 88, OFF_FIXED = 100, OFF_DENS = 104, OFF_PRES = 108, OFF_VM = 112, OFF_IVM = 116, OFF_IION = 120,
    OFF_STIM = 124, OFF_W = 128
};

static std::string g_create_error;
static int (*g_nccl_destroy)(void *) = nullptr;  // set once libnccl is loaded (sphsm_destroy runs before its definition)

enum KernelGroup { KG_HASH = 0, KG_SORT, KG_GRID, KG_MOMENTS, KG_GOAL, KG_PASS_A, KG_PASS_B, KG_OTHER };
static const char *kGroupNames[SPHSM_NUM_KERNEL_GROUPS] = {"hash", "radix_sort", "cell_bounds+reorder", "sm_moments+solve",
                                                           "goal+corrected_vel", "pass_a(density+xsph)",
                                                           "pass_b(cell+force+laplacian+integrate)", "other"};

struct sphsm_handle {
    sphsm_params prm;
    DevParams dp;
    DevParams *d_dp = nullptr;  // global-memory copy of dp for the fast passes (loop invariants pinned in registers, sphsm_pass4.cuh)
    DevParams dp_uploaded{};
    int n = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t launch_stream = nullptr;  // where LAUNCH enqueues: `stream`, except while the side chain below is built
    cudaStream_t side_stream = nullptr;    // slab step: moment sums + allreduce + solve run here, beside the sort
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_bnd = nullptr, ev_int = nullptr;
    bool moments_forked = false;
    bool allreduce_pending = false;        // slab step: the forked sums still need their allreduce (issued after exchange 1 on a shared communicator)
    double meta_wait_us = 0.0;             // SPHSM_HOST_PROF: host time spent waiting for the plane boundaries
    // NCCL mode: a rank-local step error (halo overflow, a particle crossing two planes) must not leave the peers waiting in
    // a collective.  It is recorded, rides as one extra element on the NEXT step's moment allreduce, and every rank returns the
    // error at the end of that step (so all ranks stop after the same step, at most one step late).
    int local_error = 0;
    std::string local_error_msg;
    bool peer_error = false, failed = false;
    bool reordered = false;                // slab step: the gather was queued before the plane boundaries reached the host
    bool split = false;                    // slab step: exchange 2 in flight on the side stream beside the interior planes
    Arrays cur{}, alt{};
    uint32_t *keys[2] = {nullptr, nullptr}, *vals[2] = {nullptr, nullptr};
    uint32_t *skeys = nullptr;       // counting sort: the cell key of every slot, in slot order (k_cell_scatter)
    uint32_t *key_sorted = nullptr;  // what the neighbour passes read: skeys, or the radix sort's sorted key buffer
    uint32_t *ghist = nullptr, *tile_state = nullptr, *tile_counter = nullptr;
    int sorted_buf = 0;  // which keys[] / vals[] hold the sorted result
    bool order_inline = false;        // the last sort left the slots of a cell in arrival order: the gather applies the canonical order
    const uint32_t *perm = nullptr;   // the permutation the last gather applied (slot -> source slot), for freeze_source
    uint32_t *cell_count = nullptr;               // counting sort: per-cell counts (kept zero between steps)
    unsigned long long *scan_state = nullptr;     // single-pass scan: one published word per tile (k_scan_onepass)
    uint32_t *scan_ctl = nullptr;                 //   ticket, blocks done, epoch (+ pad)
    bool bounds_ready = false;                             // grid_sort already produced the cell_start table
    // CUDA graphs for small single-GPU steps (launch-latency bound): see graph_step
    bool dry_run = false;  // replaying a captured step: the host-side state transitions run, launches and stream calls do not
    struct StepGraph {
        std::string sig;
        cudaGraphExec_t exec;
    };
    std::vector<StepGraph> graphs;
    std::vector<std::string> seen_sigs;
    std::unordered_set<long long> host_cells;  // cells occupied by the positions the host handed in (small sets only): see warp_path
    int *big_cells = nullptr, *big_count = nullptr;  // counting sort: worklist of cells too full for the one-thread in-cell sort
    bool counts_ready = false;  // pass B already filed keys / ranks / per-cell counts of the CURRENT positions (single-GPU fast step)
    int *cell_start = nullptr, *slot_of = nullptr;
    SmState *sm = nullptr;
    double *partial = nullptr, *totals = nullptr;
    float *scratch = nullptr;
    uint8_t *d_aos = nullptr;
    size_t aos_cap_bytes = 0;
    // asynchronous I/O (sphsm_*_async): copy streams beside the compute stream, their own device staging
    cudaStream_t h2d_stream = nullptr, d2h_stream = nullptr;
    cudaEvent_t ev_in_ready = nullptr, ev_in_free = nullptr, ev_out_ready = nullptr, ev_out_done = nullptr;
    float *io_in_f = nullptr, *io_out_f = nullptr;
    uint8_t *io_in_b = nullptr;
    int *io_out_i = nullptr;
    size_t io_in_cap = 0, io_out_cap = 0;
    float *d_tmp = nullptr;  // staging for position lists (stim_mesh / stim_cube / init_fluid)
    size_t tmp_cap = 0;
    int *d_itmp = nullptr;
    size_t itmp_cap = 0;
    bool grid_valid = false, rest_dirty = true, inter_live = true, slot_of_valid = false;
    // the fast path without diagnostics does not keep GOAL / PV (mGoalPos, predicted_vel) current; a particle that becomes fixed
    // between steps must still freeze at the values the last step computed for it (cpp:228, 326): see freeze_source()
    bool goal_pv_stale = false;   // GOAL / PV arrays are older than the last step
    bool prev_vel_valid = false;  // alt.VEL[vals[sorted_buf][s]] is the velocity slot s had BEFORE the last step
    int sort_passes = 1, max_tiles = 1, red_blocks = 1;
    long long launches = 0;
    int total_steps = 0;
    bool stage_timing = false;
    double stage_time[7] = {0, 0, 0, 0, 0, 0, 0};
    cudaEvent_t ev[SPHSM_NUM_KERNEL_GROUPS + 2] = {};
    cudaEvent_t ev_step0 = nullptr, ev_step1 = nullptr, ev_tm[2] = {nullptr, nullptr};
    float last_step_ms = 0.f;
    bool profiling = false;
    float group_ms[SPHSM_NUM_KERNEL_GROUPS] = {};
    int group_launches[SPHSM_NUM_KERNEL_GROUPS] = {};
    std::string err;
    // ---- multi-GPU slab layer (sphsm_comm.cuh) ----
    int comm_mode = 0;        // 0 none, 1 NCCL (one process per GPU), 2 local group (virtual ranks on one device, for tests)
    int nranks = 1, rank = 0;
    void *nccl_comm = nullptr;
    void *nccl_comm_red = nullptr;  // communicator of the moment allreduce: nccl_comm, or a split of it (SPHSM_SPLIT_COMM)
    bool slab_applied = false;
    int send_cap = 0;         // particles per exchange-1 message
    int alloc_n = 0;          // slots allocated per array (capacity + room for two halo messages in slab mode)
    uint8_t *msg_send[2] = {nullptr, nullptr}, *msg_recv[2] = {nullptr, nullptr};  // [0] left neighbour, [1] right neighbour
    // push exchange (NCCL mode, neighbours reachable through CUDA IPC): exchange 1 is written by the packing kernel straight into the
    // neighbour's receive slots over NVLink (x1_send_view), a one-thread kernel publishes count + sequence number, the receiver's
    // unpack kernel polls its own flag word — no ncclSend / ncclRecv, no host-known message size
    uint8_t *p2p_block = nullptr;                   // [flags 256 B][from left, parity 0/1][from right, parity 0/1][allreduce landing area]
    uint8_t *p2p_peer[2] = {nullptr, nullptr};      // the neighbours' blocks, mapped here (entries of p2p_all)
    std::vector<uint8_t *> p2p_all;                 // every rank's block (own = p2p_block): the push allreduce stores into all of them
    uint8_t **d_p2p_all = nullptr;                  //   the same table in device memory
    size_t p2p_slot_bytes = 0;
    bool p2p_on = false, p2p_red_on = false;        // push exchange / push allreduce live (decided collectively in sphsm_comm_init)
    long long red_seq = 0;                          // push allreduces issued so far
    int *d_err = nullptr;
    // slot ranges of the slab (SlabMeta, sphsm_comm.cuh): two device copies written alternately by the sort of each step
    // (meta_cur = the one the latest sort wrote) and a ring of pinned host copies the host reads META_LAG steps late
    SlabMeta *d_meta[2] = {nullptr, nullptr};
    int meta_cur = 0;
    static const int META_RING = 8, META_LAG = 2;
    int *h_ring = nullptr;                 // META_RING x 8 ints, pinned
    cudaEvent_t ev_ring[META_RING] = {};
    long long meta_issued = 0, meta_consumed = 0;  // read-backs queued / applied to the host fields below
    int n_bound = 0;                       // upper bound of the live slot count the grids of the slab step are sized for
    int own_bound = 0;                     // likewise for the owned slots
    int *d_count = nullptr;                // sphsm_download_owned_async: the owned count of the queued gather
    // SPHSM_TRACE=<step>: CUDA events at the phase boundaries of three consecutive slab steps starting at <step>, on both streams, read
    // only after the third one (nothing synchronises inside the traced steps); printed by rank 0 and the last rank (trace_mark / trace_dump)
    struct TraceEv { cudaEvent_t ev; const char *label; int stream; };
    std::vector<TraceEv> trace;
    int trace_from = -1;
    // exchange 1 of the NEXT step issued at the end of a step, behind pass B on the outer planes (it travels while the interior
    // planes are still being integrated).  Anything that changes particle state other than stimulation values between two steps
    // voids it (x1_early_valid = false): the next step then classifies and exchanges again, on every rank alike — state mutators
    // are collective calls in slab mode.
    bool x1_early_pending = false, x1_early_valid = false, check_interior_pending = false, drop_in_unpack = false;
    cudaEvent_t ev_x1 = nullptr, ev_meta_ready = nullptr;
    cudaStream_t meta_stream = nullptr;  // the 32-byte read-backs of SlabMeta travel beside the step, not inside its main stream
    // exchange-1 messages are sized from the populations both sides of a face saw X1_LAG exchanges ago (see x1_plan)
    static constexpr int X1_RING = 8, X1_LAG = 3;
    int x1_send_cap[2] = {0, 0}, x1_recv_cap[2] = {0, 0};  // particles per message of the exchange packed last (<= send_cap)
    long long x1_seq = 0, x1_floor = 0;                    // exchanges packed so far / the first one after the last population change
    int *d_x1rec = nullptr, *h_x1rec = nullptr;            // X1_RING x {sent left, sent right, received left, received right}; pinned copy
    long long x1rec_seq[X1_RING] = {-1, -1, -1, -1, -1, -1, -1, -1};
    cudaEvent_t ev_x1rec[X1_RING] = {}, ev_x1rec_ready = nullptr;
    int b2 = 0, b3 = 0;       // start of the 2nd / of the last owned plane, as of the last applied read-back
    int n_global = 0;         // particles uploaded before sphsm_comm_set_slab filtered them (ids are global)
    int mom_n = 0;            // slab step: extent of the PRE-reorder arrays (old slots + both message regions) the REST-state sums scan
    int mom_begin = 0, mom_end = 0;  // slab step: the slots this rank integrated last step; its share of the per-step moment sums
    struct GroupTimer *gt = nullptr;
    // activation maps / probe traces of Vm (sphsm_record.cuh, sphsm_host_record.cuh): nothing allocated or launched while off
    struct Recorder {
        bool on = false;
        float vm_up = 0.f, vm_down = 0.f;
        int cap = 0, n_probes = 0, rows = 0;
        int *maps = nullptr;      // 4 x cap: first_up, last_up, last_down, n_up (by original id)
        int *probe_of = nullptr;  // cap entries, -1 = not a probe
        float4 *trace = nullptr;  // rows x n_probes ring
        int *stamp = nullptr;     // rows x n_probes: step that wrote the entry
        long long recorded = 0;   // steps recorded since start / reset
    } rec;
    // extracellular electrograms at virtual electrodes (sphsm_egm.cuh, sphsm_host_egm.cuh): nothing allocated or launched while off
    struct Electrograms {
        bool on = false;
        int n_el = 0, rows = 0, grid = 0;  // grid: k_egm's blocks (fixed while on: the summation order depends on it)
        float gain = 0.f, eps2 = 0.f;      // eps2 = softening^2
        float *Q = nullptr;                // alloc_n + 8: pass B's source vol * L by slot (also cur.Q / alt.Q)
        float4 *el = nullptr;              // n_el electrodes
        double *partial = nullptr;         // grid x n_el
        double *ring = nullptr;            // rows x n_el
        long long recorded = 0;            // steps reduced since start / reset
    } egm;
    // the device step counter of the recorder and the electrograms (allocated while either is on; sphsm_host_record.cuh)
    unsigned *step_ctl = nullptr;  // [0] total_time_steps before the step, [1] ticket of the kernel that advances it
    int dev_steps = 0;             // what step_ctl[0] holds once the queued steps have run
};

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            char b_[512];                                                                          \
            snprintf(b_, sizeof b_, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
            if (h) h->err = b_; else g_create_error = b_;                                          \
            return SPHSM_ERR_CUDA;                                                                 \
        }                                                                                          \
    } while (0)

// SPHSM_SYNC_DEBUG=1 in the environment synchronises after every launch and names the kernel that faulted
static const bool g_sync_debug = getenv("SPHSM_SYNC_DEBUG") != nullptr;
// 1: ncclSend / ncclRecv exchange-1 messages sized from the lagged face populations; 0 (default): always the full halo capacity.
// Process-wide: every rank of a group must run with the same setting (the two sides of a face derive the message size from it).
// Off by default: a REGULAR lattice moves a whole lattice plane across a cell boundary in one step, which doubles a face
// population at once (15625 -> 31250 on the 8M benchmark lattice; seen at 8 GPUs) — no margin short of the capacity covers that.
// The push exchange below needs no size at all and is what the NCCL mode uses when the neighbours are reachable through CUDA IPC.
static int g_x1_dynamic = getenv("SPHSM_X1_DYNAMIC") ? atoi(getenv("SPHSM_X1_DYNAMIC")) : 0;
static int g_p2p_red = getenv("SPHSM_P2P_RED") ? atoi(getenv("SPHSM_P2P_RED")) : 1;  // 0: the allreduces stay on ncclAllReduce (collective decision, like SPHSM_P2P)
static int g_p2p = getenv("SPHSM_P2P") ? atoi(getenv("SPHSM_P2P")) : 1;  // 0: exchange 1 stays on ncclSend / ncclRecv (decided collectively at sphsm_comm_init)
static int g_warp_path = getenv("SPHSM_WARP_PATH") ? atoi(getenv("SPHSM_WARP_PATH")) : 1;  // 0: small dense sets take the thread-per-particle kernels too
extern "C" int sphsm_tune(const char *name, int value) {
    if (!name) return SPHSM_ERR_INVALID;
    const std::string n(name);
    if (n == "warp_path" && (value == 0 || value == 1)) g_warp_path = value;
    else if (n == "x1_dynamic" && (value == 0 || value == 1)) g_x1_dynamic = value;
    else return SPHSM_ERR_INVALID;
    return SPHSM_OK;
}
#define LAUNCH(kern, grid, block, ...)                                                                  \
    do {                                                                                                \
        if (!h->dry_run) kern<<<(grid), (block), 0, h->launch_stream>>>(__VA_ARGS__);                   \
        h->launches++;                                                                                  \
        if (g_sync_debug) {                                                                             \
            cudaError_t e_ = cudaStreamSynchronize(h->launch_stream);                                   \
            if (e_ != cudaSuccess) {                                                                    \
                h->err = std::string("kernel ") + #kern + " failed: " + cudaGetErrorString(e_);         \
                fprintf(stderr, "[sphsm] %s\n", h->err.c_str());                                        \
                return SPHSM_ERR_CUDA;                                                                  \
            }                                                                                           \
        }                                                                                               \
    } while (0)

static int slab_refresh(sphsm_handle *h);  // sphsm_host_slab.cuh: apply every queued read-back of the slab's slot ranges to the host fields

static int fail(sphsm_handle *h, int code, const char *msg) {
    if (h) h->err = msg; else g_create_error = msg;
    return code;
}
static inline int cdiv(long long a, int b) { return (int)((a + b - 1) / b); }
static inline void set_n(sphsm_handle *h, int n) {  // single-GPU meaning: every slot is computed
    h->n = n;
    h->dp.n = n;
    h->dp.own_begin = 0;
    h->dp.own_end = n;
}

// ---------------------------------------------------------------------------------------------------
// defaults: the reference ctor, cpp:13-69, with its float/double promotions (SURVEY.md Q16)
extern "C" int sphsm_abi_version(void) { return SPHSM_ABI_VERSION; }

extern "C" int sphsm_default_params(sphsm_params *p) {
    if (!p) return SPHSM_ERR_INVALID;
    memset(p, 0, sizeof(*p));
    p->struct_size = (uint32_t)sizeof(*p);
    p->device = 0;
    p->capacity = 50000;
    p->world[0] = p->world[1] = p->world[2] = 1.5f;
    p->kernel_h = 0.04f;
    p->gravity[0] = 0.0f; p->gravity[1] = -9.8f; p->gravity[2] = 0.0f;
    p->K = 0.5f;
    p->stand_density = 1112.0f;
    const float max_vel2 = 3.0f * 3.0f + 3.0f * 3.0f + 3.0f * 3.0f;                          // max_vel.magnitudeSquared()
    p->time_delta = (float)(0.4 * (double)p->kernel_h / (double)sqrtf(max_vel2));            // cpp:47
    p->wall_hit = -1.0f;
    p->mu = 100.0f;
    p->velocity_mixing = 1.0f;
    const float pi = 3.1415926535897932f;                                                    // m3Pi, m3Real.h:9
    p->poly6_constant = (float)((double)315.0f / ((double)(64.0f * pi) * pow((double)p->kernel_h, 9.0)));  // cpp:54
    p->spiky_constant = (float)((double)45.0f / ((double)pi * pow((double)p->kernel_h, 6.0)));             // cpp:55
    p->bspline_constant = 1.0f / (pi * p->kernel_h * p->kernel_h * p->kernel_h);                           // cpp:57
    p->alpha = 0.3f; p->beta = 0.4f;
    p->quadratic_match = 0; p->volume_conservation = 1; p->allow_flip = 0;
    p->Cm = 1.f; p->Beta = 50;
    {
        float sigma_i = 0.893, sigma_e = 0.67;  // cpp:15 (double literals narrowed to float)
        p->sigma = sigma_i * sigma_e / (sigma_i + sigma_e);
    }
    p->stim_strength = 300.0f;
    p->FH_Vt = -75.0; p->FH_Vp = 15.0; p->FH_Vr = -85.0;
    p->C1 = 0.175; p->C2 = 0.03; p->C3 = 0.011; p->C4 = 0.55;
    p->voltage_constant = 1; p->max_pressure = 15000; p->max_voltage = 200;
    p->particle_mass = 0.2f;
    p->diagnostics = 1;
    p->strict = 0;
    p->slab_axis = -1;
    return SPHSM_OK;
}

// largest float x (searching around `guess`) with pred(x) true, pred monotone (true below, false above)
template <class Pred>
static float max_float_where(Pred pred, float guess) {
    float x = guess;
    while (!pred(x)) x = nextafterf(x, 0.0f);
    while (pred(nextafterf(x, INFINITY))) x = nextafterf(x, INFINITY);
    return x;
}

static void derive_dev_params(sphsm_handle *h) {
    const sphsm_params &q = h->prm;
    DevParams &d = h->dp;
    memset(&d, 0, sizeof d);
    d.n = h->n;
    d.cell_size = q.kernel_h;  // Cell_Size == kernel, cpp:17,31
    d.h = q.kernel_h;
    d.h2 = q.kernel_h * q.kernel_h;
    for (int a = 0; a < 3; a++) {
        d.world[a] = q.world[a];
        d.gravity[a] = q.gravity[a];
        d.g[a] = (int)ceilf(q.world[a] / d.cell_size);  // cpp:32-35
    }
    if (q.slab_axis >= 0 && q.slab_axis <= 2) {
        d.perm[2] = q.slab_axis;
        d.perm[0] = (q.slab_axis + 1) % 3;
        d.perm[1] = (q.slab_axis + 2) % 3;
        if (d.perm[0] > d.perm[1]) std::swap(d.perm[0], d.perm[1]);
    } else {
        d.perm[0] = 0; d.perm[1] = 1; d.perm[2] = 2;
    }
    d.ga = d.g[d.perm[0]] + 2; d.gb = d.g[d.perm[1]] + 2; d.gc = d.g[d.perm[2]];  // ga, gb: one empty border cell per side
    d.c_off = 0; d.gcl = d.gc; d.slab_lo = 0; d.slab_hi = d.gc;
    d.slab_on = 0; d.own_begin = 0; d.own_end = h->n; d.hole_begin = 0; d.hole_len = 0;
    d.num_cells = d.ga * d.gb * d.gcl;
    d.K = q.K; d.rho0 = q.stand_density; d.dt = q.time_delta; d.inv_dt = 1.0f / q.time_delta;  // cpp:661
    d.wall_hit = q.wall_hit; d.mu = q.mu; d.mix = q.velocity_mixing;
    d.c_poly6 = q.poly6_constant; d.c_spiky = q.spiky_constant; d.c_bspline = q.bspline_constant;
    d.alpha = q.alpha; d.beta = q.beta;
    d.quadratic = q.quadratic_match; d.volume = q.volume_conservation; d.allow_flip = q.allow_flip;
    d.Cm = q.Cm; d.Beta = q.Beta; d.sigma = q.sigma;
    d.diff_coef = q.sigma / (q.Beta * q.Cm);  // cpp:571
    d.Vr = q.FH_Vr;
    d.fh_denom = q.FH_Vp - q.FH_Vr;                 // cpp:579
    d.fh_asd = (q.FH_Vt - q.FH_Vr) / d.fh_denom;    // cpp:580
    d.C1 = q.C1; d.C2 = q.C2; d.C3 = q.C3; d.C4 = q.C4;
    d.voltage_constant = q.voltage_constant; d.max_pressure = q.max_pressure; d.max_voltage = q.max_voltage;
    const float hh = d.h;
    d.r2_spiky = max_float_where([hh](float x) { return sqrtf(x) <= hh; }, hh * hh);
    d.r2_q1 = max_float_where([hh](float x) { return (sqrtf(x) / hh) < 1.0f; }, hh * hh);
    d.r2_q2 = max_float_where([hh](float x) { return (sqrtf(x) / hh) < 2.0f; }, 4.0f * hh * hh);
    d.bs_a1 = (float)(4.5 * (double)d.c_bspline / (double)hh);
    d.bs_b1 = (float)(-3.0 * (double)d.c_bspline);
    d.bs_a2 = (float)(-1.5 * (double)d.c_bspline / (double)hh);
    d.bs_b2 = (float)(3.0 * (double)d.c_bspline);
    d.poly6_self = (float)((double)d.c_poly6 * pow((double)(d.h2 - 0.0f), 3.0));  // Poly6(0.0f), cpp:151,483
}

// ---------------------------------------------------------------------------------------------------
static int alloc_arrays(sphsm_handle *h, Arrays &a, int cap, bool with_cold) {
    size_t n4 = ((size_t)cap + 8) * sizeof(float4);  // tail: the pair loops read slot j+1 (masked) up to j+1 == n
    CU(cudaMalloc(&a.P, n4)); CU(cudaMalloc(&a.VEL, n4)); CU(cudaMalloc(&a.O, n4)); CU(cudaMalloc(&a.E, n4));
    CU(cudaMalloc(&a.ID, (size_t)cap * sizeof(int)));
    CU(cudaMalloc(&a.C, n4)); CU(cudaMalloc(&a.V, n4)); CU(cudaMalloc(&a.S, (size_t)cap * sizeof(float2)));
    CU(cudaMalloc(&a.ACC, n4)); CU(cudaMalloc(&a.GOAL, n4)); CU(cudaMalloc(&a.PV, n4)); CU(cudaMalloc(&a.PB, n4));
    CU(cudaMemset(a.PB, 0, n4));
    CU(cudaMalloc(&a.VN, ((size_t)cap + 8) * sizeof(float)));
    CU(cudaMemset(a.VN, 0, ((size_t)cap + 8) * sizeof(float)));
    CU(cudaMemset(a.C, 0, n4)); CU(cudaMemset(a.V, 0, n4)); CU(cudaMemset(a.S, 0, (size_t)cap * sizeof(float2)));
    CU(cudaMemset(a.ACC, 0, n4)); CU(cudaMemset(a.GOAL, 0, n4)); CU(cudaMemset(a.PV, 0, n4));
    if (with_cold) {
        CU(cudaMalloc(&a.COLD_GOAL, n4)); CU(cudaMalloc(&a.COLD_PV, n4));
        CU(cudaMemset(a.COLD_GOAL, 0, n4)); CU(cudaMemset(a.COLD_PV, 0, n4));
    }
    return SPHSM_OK;
}
static void free_arrays(Arrays &a, bool with_cold) {
    cudaFree(a.P); cudaFree(a.VEL); cudaFree(a.O); cudaFree(a.E); cudaFree(a.ID); cudaFree(a.C); cudaFree(a.V);
    cudaFree(a.S); cudaFree(a.ACC); cudaFree(a.GOAL); cudaFree(a.PV); cudaFree(a.PB); cudaFree(a.VN);
    if (with_cold) { cudaFree(a.COLD_GOAL); cudaFree(a.COLD_PV); }
}

static int setup_grid_buffers(sphsm_handle *h) {
    // (re)allocates what depends on the number of cells
    if (h->cell_start) cudaFree(h->cell_start);
    h->cell_start = nullptr;
    CU(cudaMalloc(&h->cell_start, ((size_t)h->dp.num_cells + 2) * sizeof(int)));
    if (h->cell_count) cudaFree(h->cell_count);
    if (h->scan_state) cudaFree(h->scan_state);
    h->cell_count = nullptr;
    h->scan_state = nullptr;
    CU(cudaMalloc(&h->cell_count, ((size_t)h->dp.num_cells + 2 + SCAN_IPT) * sizeof(uint32_t)));
    CU(cudaMemset(h->cell_count, 0, ((size_t)h->dp.num_cells + 2 + SCAN_IPT) * sizeof(uint32_t)));
    h->counts_ready = false;
    {
        const size_t tiles = (size_t)(h->dp.num_cells + 2) / SCAN_TILE + 2;
        CU(cudaMalloc(&h->scan_state, tiles * sizeof(unsigned long long)));
        CU(cudaMemset(h->scan_state, 0, tiles * sizeof(unsigned long long)));
        if (!h->scan_ctl) CU(cudaMalloc(&h->scan_ctl, 4 * sizeof(uint32_t)));
        CU(cudaMemset(h->scan_ctl, 0, 4 * sizeof(uint32_t)));  // epoch 0 again: matches the zeroed state words (status 0 = nothing published)
    }
    int bits = 1;
    while ((1ll << bits) < (long long)h->dp.num_cells + 1) bits++;
    h->sort_passes = (bits + RADIX_BITS - 1) / RADIX_BITS;
    if (h->sort_passes > MAX_SORT_PASSES) return fail(h, SPHSM_ERR_INVALID, "grid too large for the radix sort key");
    // the memsets above run in the legacy default stream, which the handle's non-blocking streams do not wait for: without this the
    // first scan after sphsm_comm_set_slab could meet a not-yet-cleared epoch / state table (seen once as a spurious exchange error)
    CU(cudaDeviceSynchronize());
    return SPHSM_OK;
}

static int create_impl(const sphsm_params *p, sphsm_handle **out, sphsm_handle **partial);
extern "C" int sphsm_create(const sphsm_params *p, sphsm_handle **out) {
    // a failure after the handle exists (a CUDA call, an allocation) must not leak its streams, events and device arrays
    sphsm_handle *partial = nullptr;
    const int rc = create_impl(p, out, &partial);
    if (rc != SPHSM_OK && partial) {
        const std::string why = partial->err.empty() ? g_create_error : partial->err;
        sphsm_destroy(partial);
        g_create_error = why;  // sphsm_last_error(NULL) reports it
    }
    return rc;
}
static int create_impl(const sphsm_params *p, sphsm_handle **out, sphsm_handle **partial) {
    sphsm_handle *h = nullptr;
    if (!p || !out) return fail(nullptr, SPHSM_ERR_INVALID, "null argument");
    if (p->struct_size != sizeof(sphsm_params)) return fail(nullptr, SPHSM_ERR_INVALID, "sphsm_params.struct_size mismatch (ABI)");
    if (p->capacity <= 0 || p->kernel_h <= 0.f || p->world[0] <= 0.f || p->world[1] <= 0.f || p->world[2] <= 0.f)
        return fail(nullptr, SPHSM_ERR_INVALID, "capacity, kernel_h and world must be positive");
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (p->device < 0 || p->device >= ndev) return fail(nullptr, SPHSM_ERR_CUDA, "no such CUDA device (no CPU fallback exists)");
    CU(cudaSetDevice(p->device));
    sphsm_handle *nh = new sphsm_handle();
    nh->prm = *p;
    nh->n = 0;
    derive_dev_params(nh);
    {
        long long cells = (long long)nh->dp.ga * nh->dp.gb * nh->dp.gcl;
        if (cells <= 0 || cells >= (1ll << 30)) {
            delete nh;
            return fail(nullptr, SPHSM_ERR_INVALID, "grid has too many cells");
        }
    }
    h = nh;
    *partial = nh;
    // slab mode appends up to two halo messages behind the local particles before every sort: room for them
    if (p->slab_axis >= 0) {
        int hc = p->reserved[0];  // halo capacity override (particles per message)
        if (hc <= 0) {
            // default: 2.5 times the average population of a cell plane across the slab axis at full capacity (a cell
            // plane of a regular lattice holds one OR two lattice planes), plus slack for migrants
            const double planes = std::max(1.0, ceil((double)p->world[p->slab_axis] / (double)p->kernel_h));
            hc = (int)std::min((double)p->capacity, 2.5 * (double)p->capacity / planes) + 4096;
        }
        h->send_cap = hc;
    }
    h->alloc_n = p->capacity + 2 * h->send_cap;
    const int cap = h->alloc_n;
    int rc;
    CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    {
        int prio_lo = 0, prio_hi = 0;  // the side stream carries the short chains everything else waits for
        CU(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CU(cudaStreamCreateWithPriority(&h->side_stream, cudaStreamNonBlocking, prio_hi));
    }
    CU(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
    CU(cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking));
    for (cudaEvent_t *e : {&h->ev_in_ready, &h->ev_in_free, &h->ev_out_ready, &h->ev_out_done}) CU(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_bnd, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_x1, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_meta_ready, cudaEventDisableTiming));
    CU(cudaStreamCreateWithFlags(&h->meta_stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&h->ev_x1rec_ready, cudaEventDisableTiming));
    for (int k = 0; k < sphsm_handle::X1_RING; k++) CU(cudaEventCreateWithFlags(&h->ev_x1rec[k], cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_int, cudaEventDisableTiming));
    h->launch_stream = h->stream;
    if ((rc = alloc_arrays(h, h->cur, cap, true)) != 0) return rc;
    if ((rc = alloc_arrays(h, h->alt, cap, false)) != 0) return rc;
    h->alt.COLD_GOAL = h->cur.COLD_GOAL;
    h->alt.COLD_PV = h->cur.COLD_PV;
    for (int k = 0; k < 2; k++) {
        CU(cudaMalloc(&h->keys[k], (size_t)cap * sizeof(uint32_t)));
        CU(cudaMalloc(&h->vals[k], (size_t)cap * sizeof(uint32_t)));
    }
    CU(cudaMalloc(&h->skeys, ((size_t)cap + 8) * sizeof(uint32_t)));
    h->max_tiles = cdiv(cap, SORT_TILE);
    CU(cudaMalloc(&h->ghist, MAX_SORT_PASSES * RADIX * sizeof(uint32_t)));
    CU(cudaMalloc(&h->tile_state, (size_t)MAX_SORT_PASSES * h->max_tiles * RADIX * sizeof(uint32_t)));
    CU(cudaMalloc(&h->tile_counter, MAX_SORT_PASSES * sizeof(uint32_t)));
    CU(cudaMalloc(&h->slot_of, (size_t)cap * sizeof(int)));
    CU(cudaMalloc(&h->big_cells, ((size_t)cap / BIG_CELL + 2) * sizeof(int)));
    CU(cudaMalloc(&h->big_count, 2 * sizeof(int)));  // (one per scan epoch parity)
    CU(cudaMemset(h->big_count, 0, 2 * sizeof(int)));
    CU(cudaMalloc(&h->d_dp, sizeof(DevParams)));
    CU(cudaMalloc(&h->sm, sizeof(SmState)));
    CU(cudaMemset(h->sm, 0, sizeof(SmState)));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, p->device));
    h->red_blocks = std::max(1, std::min(8 * prop.multiProcessorCount, cdiv(cap, 256)));  // enough loads in flight to cover HBM latency
    CU(cudaMalloc(&h->partial, (size_t)h->red_blocks * 10 * 9 * sizeof(double)));
    CU(cudaMalloc(&h->totals, 128 * sizeof(double)));
    CU(cudaMalloc(&h->scratch, 162 * sizeof(float)));
    if ((rc = setup_grid_buffers(h)) != 0) return rc;
    for (auto &e : h->ev) CU(cudaEventCreate(&e));
    CU(cudaEventCreate(&h->ev_step0));
    CU(cudaEventCreate(&h->ev_step1));
    CU(cudaEventCreate(&h->ev_tm[0]));
    CU(cudaEventCreate(&h->ev_tm[1]));
    *out = h;
    *partial = nullptr;
    return SPHSM_OK;
}

extern "C" int sphsm_destroy(sphsm_handle *h) {
    if (!h) return SPHSM_OK;
    cudaSetDevice(h->prm.device);
    cudaStreamSynchronize(h->stream);
    free_arrays(h->cur, true);
    free_arrays(h->alt, false);
    for (int k = 0; k < 2; k++) { cudaFree(h->keys[k]); cudaFree(h->vals[k]); }
    cudaFree(h->skeys);
    cudaFree(h->cell_count); cudaFree(h->scan_state); cudaFree(h->scan_ctl); cudaFree(h->big_cells); cudaFree(h->big_count);
    cudaFree(h->ghist); cudaFree(h->tile_state); cudaFree(h->tile_counter); cudaFree(h->cell_start); cudaFree(h->slot_of);
    cudaFree(h->d_dp); cudaFree(h->sm); cudaFree(h->partial); cudaFree(h->totals); cudaFree(h->scratch); cudaFree(h->d_aos); cudaFree(h->d_tmp);
    cudaFree(h->d_itmp);
    cudaFree(h->rec.maps); cudaFree(h->rec.probe_of); cudaFree(h->rec.trace); cudaFree(h->rec.stamp); cudaFree(h->step_ctl);
    cudaFree(h->egm.Q); cudaFree(h->egm.el); cudaFree(h->egm.partial); cudaFree(h->egm.ring);
    for (int k = 0; k < 2; k++) { cudaFree(h->msg_send[k]); cudaFree(h->msg_recv[k]); }
    for (size_t k = 0; k < h->p2p_all.size(); k++)
        if (h->p2p_all[k] && h->p2p_all[k] != h->p2p_block) cudaIpcCloseMemHandle(h->p2p_all[k]);
    if (h->d_p2p_all) cudaFree(h->d_p2p_all);
    // (the exported block itself is NOT freed while the push exchange was live: a neighbour may still have it mapped, and freeing
    //  exported memory under an importer is undefined; destroy is not collective, so there is no safe point — ~13 MB per NCCL-mode
    //  handle stay with the process until it exits)
    if (h->p2p_block && !h->p2p_on) cudaFree(h->p2p_block);
    cudaFree(h->d_err); cudaFree(h->d_meta[0]); cudaFree(h->d_meta[1]); cudaFree(h->d_count);
    if (h->h_ring) cudaFreeHost(h->h_ring);
    for (auto &e : h->ev_ring) if (e) cudaEventDestroy(e);
    if (h->nccl_comm_red && h->nccl_comm_red != h->nccl_comm && g_nccl_destroy) g_nccl_destroy(h->nccl_comm_red);
    if (h->nccl_comm && g_nccl_destroy) g_nccl_destroy(h->nccl_comm);
    for (auto &e : h->ev) if (e) cudaEventDestroy(e);
    if (h->ev_step0) cudaEventDestroy(h->ev_step0);
    if (h->ev_step1) cudaEventDestroy(h->ev_step1);
    for (auto &e : h->ev_tm) if (e) cudaEventDestroy(e);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    for (auto &gx : h->graphs) cudaGraphExecDestroy(gx.exec);
    h->graphs.clear();
    for (cudaEvent_t e : {h->ev_in_ready, h->ev_in_free, h->ev_out_ready, h->ev_out_done})
        if (e) cudaEventDestroy(e);
    if (h->h2d_stream) cudaStreamDestroy(h->h2d_stream);
    if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
    cudaFree(h->io_in_f); cudaFree(h->io_in_b); cudaFree(h->io_out_f); cudaFree(h->io_out_i);
    if (h->ev_bnd) cudaEventDestroy(h->ev_bnd);
    if (h->ev_x1) cudaEventDestroy(h->ev_x1);
    if (h->ev_meta_ready) cudaEventDestroy(h->ev_meta_ready);
    if (h->meta_stream) cudaStreamDestroy(h->meta_stream);
    if (h->ev_x1rec_ready) cudaEventDestroy(h->ev_x1rec_ready);
    for (int k = 0; k < sphsm_handle::X1_RING; k++)
        if (h->ev_x1rec[k]) cudaEventDestroy(h->ev_x1rec[k]);
    if (h->d_x1rec) cudaFree(h->d_x1rec);
    if (h->h_x1rec) cudaFreeHost(h->h_x1rec);
    if (h->ev_int) cudaEventDestroy(h->ev_int);
    if (h->side_stream) cudaStreamDestroy(h->side_stream);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return SPHSM_OK;
}

extern "C" const char *sphsm_last_error(sphsm_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

extern "C" int sphsm_get_params(sphsm_handle *h, sphsm_params *out) {
    if (!h || !out) return SPHSM_ERR_INVALID;
    *out = h->prm;
    return SPHSM_OK;
}

extern "C" int sphsm_set_params(sphsm_handle *h, const sphsm_params *p) {
    if (!h || !p) return SPHSM_ERR_INVALID;
    if (p->struct_size != sizeof(sphsm_params)) return fail(h, SPHSM_ERR_INVALID, "sphsm_params.struct_size mismatch (ABI)");
    if (p->capacity != h->prm.capacity || p->device != h->prm.device || p->kernel_h != h->prm.kernel_h ||
        memcmp(p->world, h->prm.world, sizeof p->world) != 0 || p->slab_axis != h->prm.slab_axis)
        return fail(h, SPHSM_ERR_INVALID, "capacity, device, kernel_h, world and slab_axis are fixed at create");
    const DevParams old = h->dp;
    h->prm = *p;
    derive_dev_params(h);
    h->dp.c_off = old.c_off; h->dp.gcl = old.gcl; h->dp.slab_lo = old.slab_lo; h->dp.slab_hi = old.slab_hi; h->dp.num_cells = old.num_cells;
    h->dp.slab_on = old.slab_on; h->dp.own_begin = old.own_begin; h->dp.own_end = old.own_end;
    return SPHSM_OK;
}

// ---------------------------------------------------------------------------------------------------
// AoS <-> SoA
__device__ __forceinline__ float ldf(const uint8_t *rec, int off) { return *reinterpret_cast<const float *>(rec + off); }
__device__ __forceinline__ void stf(uint8_t *rec, int off, float v) { *reinterpret_cast<float *>(rec + off) = v; }

__global__ void k_aos_to_soa(int first, int count, const uint8_t *__restrict__ aos, int stride, Arrays a) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const int i = first + k;
    const uint8_t *r = aos + (size_t)k * stride;
    const float mass = ldf(r, OFF_MASS), dens = ldf(r, OFF_DENS), Vm = ldf(r, OFF_VM);
    const int fixed = r[OFF_FIXED] != 0;
    a.P[i] = make_float4(ldf(r, OFF_POS), ldf(r, OFF_POS + 4), ldf(r, OFF_POS + 8), mass);
    a.VEL[i] = make_float4(ldf(r, OFF_VEL), ldf(r, OFF_VEL + 4), ldf(r, OFF_VEL + 8), dens);
    a.O[i] = make_float4(ldf(r, OFF_ORIG), ldf(r, OFF_ORIG + 4), ldf(r, OFF_ORIG + 8), __int_as_float(fixed ? i + 1 : 0));
    a.E[i] = make_float4(Vm, ldf(r, OFF_IION), ldf(r, OFF_W), ldf(r, OFF_STIM));
    a.ID[i] = i;
    a.C[i] = make_float4(ldf(r, OFF_CVEL), ldf(r, OFF_CVEL + 4), ldf(r, OFF_CVEL + 8), __fdiv_rn(mass, dens));
    a.V[i] = make_float4(ldf(r, OFF_IVEL), ldf(r, OFF_IVEL + 4), ldf(r, OFF_IVEL + 8), __fdiv_rn(mass, dens));
    a.S[i] = make_float2(ldf(r, OFF_PRES), Vm);
    a.ACC[i] = make_float4(ldf(r, OFF_ACC), ldf(r, OFF_ACC + 4), ldf(r, OFF_ACC + 8), ldf(r, OFF_IVM));
    const float4 goal = make_float4(ldf(r, OFF_GOAL), ldf(r, OFF_GOAL + 4), ldf(r, OFF_GOAL + 8), 0.f);
    const float4 pv = make_float4(ldf(r, OFF_PVEL), ldf(r, OFF_PVEL + 4), ldf(r, OFF_PVEL + 8), 0.f);
    a.GOAL[i] = goal; a.PV[i] = pv;
    a.COLD_GOAL[i] = goal; a.COLD_PV[i] = pv;
}

__global__ void k_soa_to_aos(int first, int count, Arrays a, uint8_t *__restrict__ aos, int stride) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= count) return;
    s += first;
    const int id = a.ID[s];
    uint8_t *r = aos + (size_t)id * stride;
    const float4 p = a.P[s], v = a.VEL[s], o = a.O[s], e = a.E[s], c = a.C[s], iv = a.V[s], acc = a.ACC[s];
    const float2 sp = a.S[s];
    const int flags = __float_as_int(o.w);
    const float4 goal = flags ? a.COLD_GOAL[flags - 1] : a.GOAL[s];
    const float4 pv = flags ? a.COLD_PV[flags - 1] : a.PV[s];
    stf(r, OFF_POS, p.x); stf(r, OFF_POS + 4, p.y); stf(r, OFF_POS + 8, p.z);
    stf(r, OFF_VEL, v.x); stf(r, OFF_VEL + 4, v.y); stf(r, OFF_VEL + 8, v.z);
    stf(r, OFF_PVEL, pv.x); stf(r, OFF_PVEL + 4, pv.y); stf(r, OFF_PVEL + 8, pv.z);
    stf(r, OFF_IVEL, iv.x); stf(r, OFF_IVEL + 4, iv.y); stf(r, OFF_IVEL + 8, iv.z);
    stf(r, OFF_CVEL, c.x); stf(r, OFF_CVEL + 4, c.y); stf(r, OFF_CVEL + 8, c.z);
    stf(r, OFF_ACC, acc.x); stf(r, OFF_ACC + 4, acc.y); stf(r, OFF_ACC + 8, acc.z);
    stf(r, OFF_MASS, p.w);
    stf(r, OFF_ORIG, o.x); stf(r, OFF_ORIG + 4, o.y); stf(r, OFF_ORIG + 8, o.z);
    stf(r, OFF_GOAL, goal.x); stf(r, OFF_GOAL + 4, goal.y); stf(r, OFF_GOAL + 8, goal.z);
    r[OFF_FIXED] = flags ? 1 : 0; r[OFF_FIXED + 1] = 0; r[OFF_FIXED + 2] = 0; r[OFF_FIXED + 3] = 0;
    stf(r, OFF_DENS, v.w); stf(r, OFF_PRES, sp.x); stf(r, OFF_VM, e.x); stf(r, OFF_IVM, acc.w);
    stf(r, OFF_IION, e.y); stf(r, OFF_STIM, e.w); stf(r, OFF_W, e.z);
}

__global__ void k_positions_out(int first, int count, Arrays a, float *__restrict__ xyz) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= count) return;
    s += first;
    const int id = a.ID[s];
    const float4 p = a.P[s];
    xyz[3 * (size_t)id] = p.x; xyz[3 * (size_t)id + 1] = p.y; xyz[3 * (size_t)id + 2] = p.z;
}

// Init_Particle, cpp:101-125
__global__ void k_init_particles(int first, int count, const float *__restrict__ xyz, Arrays a, float mass, float rho0) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const int i = first + k;
    const float x = xyz[3 * (size_t)k], y = xyz[3 * (size_t)k + 1], z = xyz[3 * (size_t)k + 2];
    a.P[i] = make_float4(x, y, z, mass);
    a.VEL[i] = make_float4(0.f, 0.f, 0.f, rho0);
    a.O[i] = make_float4(x, y, z, __int_as_float(0));
    a.E[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    a.ID[i] = i;
    a.C[i] = make_float4(0.f, 0.f, 0.f, __fdiv_rn(mass, rho0));
    a.V[i] = make_float4(0.f, 0.f, 0.f, __fdiv_rn(mass, rho0));
    a.S[i] = make_float2(0.f, 0.f);
    a.ACC[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    a.GOAL[i] = make_float4(x, y, z, 0.f);
    a.PV[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    a.COLD_GOAL[i] = make_float4(x, y, z, 0.f);
    a.COLD_PV[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

__global__ void k_slot_of(int n, const int *__restrict__ id, int *__restrict__ slot_of) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) slot_of[id[s]] = s;
}

// ---- stimulation / fixation ------------------------------------------------------------------------------
// set_stim (cpp:704-717) for a LIST of centres: stim = strength where the squared distance to any centre <= radius
__global__ void __launch_bounds__(256) k_set_stim_list(int n, Arrays a, const float *__restrict__ centres, int m, float radius, float strength) {
    __shared__ float sc[256 * 3];
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    float4 p = make_float4(0, 0, 0, 0);
    if (s < n) p = a.P[s];
    bool hit = false;
    for (int base = 0; base < m; base += 256) {
        const int cnt = min(256, m - base);
        __syncthreads();
        for (int k = threadIdx.x; k < cnt * 3; k += blockDim.x) sc[k] = centres[(size_t)base * 3 + k];
        __syncthreads();
        if (!hit && s < n) {
            for (int k = 0; k < cnt; k++) {
                const float dx = __fsub_rn(p.x, sc[3 * k]), dy = __fsub_rn(p.y, sc[3 * k + 1]), dz = __fsub_rn(p.z, sc[3 * k + 2]);
                if (dist2_exact(dx, dy, dz) <= radius) { hit = true; break; }
            }
        }
        if (__syncthreads_and(hit || s >= n)) break;
    }
    if (hit && s < n) a.E[s].w = strength;
}

// What a particle freezes at when it becomes fixed: the mGoalPos / predicted_vel the LAST step computed for it (the reference
// simply stops updating them, cpp:228, 326).  src 1: the GOAL / PV arrays are current (diagnostics mode, or no fast step since
// the upload).  src 2: recompute them as the last step did — the shape-matching transform of that step is still in SmState, and
// the velocity the particle had before that step is still in the gather's source buffer (prev_vel, indexed through the sorted
// permutation `vals`; nullptr: not available any more, the current velocity stands in).
struct FreezeSrc {
    int src, strict;
    const SmState *sm;
    const float4 *prev_vel;
    const uint32_t *vals;
};
__device__ __forceinline__ void freeze_goal_pv(const DevParams &p, const Arrays &a, const FreezeSrc &f, int s, int id) {
    if (f.src == 1) {
        a.COLD_GOAL[id] = a.GOAL[s];
        a.COLD_PV[id] = a.PV[s];
        return;
    }
    const float4 p4 = a.P[s], o4 = a.O[s];
    float4 v4 = f.prev_vel ? f.prev_vel[f.vals[s]] : a.VEL[s];
    v4.w = 1.0f;
    const float4 o = make_float4(o4.x, o4.y, o4.z, __int_as_float(0));
    float4 goal, pv;
    if (f.strict) goal_cvel_one<true>(p, f.sm, nullptr, nullptr, p4, v4, o, nullptr, goal, pv);
    else goal_cvel_one<false>(p, f.sm, nullptr, nullptr, p4, v4, o, nullptr, goal, pv);
    a.COLD_GOAL[id] = goal;
    a.COLD_PV[id] = pv;
}

// mode 0: turnOnStim_Mesh's fixation rule (cpp:759), 1: turnOnStim_Cube's (cpp:738); comparisons against double
// literals are done in double exactly as the reference's promotions make them.
__global__ void k_fix_rule(const __grid_constant__ DevParams p, int n, Arrays a, int mode, FreezeSrc fz) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const float4 q = a.P[s];
    bool fix;
    if (mode == 0) {
        const double x = q.x, y = q.y;
        fix = (x >= 0.0 && x <= 0.07) || (x >= 0.90 && y >= 0.80);
    } else {
        fix = (q.y == 0.0f && q.x <= 0.48f) || (q.y == 0.0f && (double)q.x >= 1.0);
    }
    if (fix && __float_as_int(a.O[s].w) == 0) {
        const int id = a.ID[s];
        freeze_goal_pv(p, a, fz, s, id);
        a.O[s].w = __int_as_float(id + 1);
    }
}

// n_dev != nullptr (slab mode, where the host's count may lag the device): only the live slots [0, *n_dev) are touched — slots behind
// them hold stale copies of particles that live elsewhere in the array, and freezing one of those would overwrite the frozen
// values of the real one
__global__ void k_set_masks(const __grid_constant__ DevParams p, int n, Arrays a, const uint8_t *__restrict__ fixed, const float *__restrict__ stim,
                            FreezeSrc fz, const int *__restrict__ n_dev) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= (n_dev ? min(*n_dev, n) : n)) return;
    const int id = a.ID[s];
    if (id < 0) return;
    if (fixed) {
        const int was = __float_as_int(a.O[s].w);
        if (fixed[id] && !was) {
            freeze_goal_pv(p, a, fz, s, id);
            a.O[s].w = __int_as_float(id + 1);
        } else if (!fixed[id] && was) {
            a.GOAL[s] = a.COLD_GOAL[was - 1];
            a.PV[s] = a.COLD_PV[was - 1];
            a.O[s].w = __int_as_float(0);
        }
    }
    if (stim) a.E[s].w = stim[id];
}

// stim[k] for the k-th particle of the last owned-particle download (ids[k] as it was delivered; count = how many were).  A
// particle that has left this rank since then is skipped: slot_of is validated against ID, and the slot must still be owned.
__global__ void k_set_stim_owned(Arrays a, const int *__restrict__ ids, const float *__restrict__ stim, int count, const int *__restrict__ slot_of,
                                 const int *__restrict__ rng, int first_h, int end_h) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    const int first = rng ? rng[0] : first_h, end = rng ? rng[1] : end_h;
    const int id = ids[k];
    if (id < 0) return;
    const int s = slot_of[id];
    if (s < first || s >= end || a.ID[s] != id) return;
    a.E[s].w = stim[k];
}
// slot_of over the slots [rng[0], rng[1]) (device range) or [0, n)
__global__ void k_slot_of_range(const int *__restrict__ rng, int n, int bound, const int *__restrict__ id, int *__restrict__ slot_of) {
    const int first = rng ? rng[0] : 0, end = rng ? rng[1] : n;
    const int s = first + blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= end || s - first >= bound) return;
    const int i = id[s];
    if (i >= 0) slot_of[i] = s;
}

// set_stim for every particle inside an axis-aligned box (the O(N) form of turnOnStim_Cube's loop of set_stim calls, cpp:719-743)
__global__ void k_set_stim_box(int n, Arrays a, float x0, float y0, float z0, float x1, float y1, float z1, float strength) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const float4 q = a.P[s];
    if (q.x >= x0 && q.x <= x1 && q.y >= y0 && q.y <= y1 && q.z >= z0 && q.z <= z1) a.E[s].w = strength;
}

// turnOffStim, cpp:764-783
__global__ void k_stim_off(int n, Arrays a) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    a.E[s] = make_float4(0.0f, 0.0f, 0.0f, -10000.0f);  // Vm, Iion, w = 0; stim = -10000
    a.S[s] = make_float2(-10000.0f, 0.0f);              // pres = -10000
    a.ACC[s].w = 0.0f;                                  // Inter_Vm = 0
}

// ---------------------------------------------------------------------------------------------------
static int ensure_tmp(sphsm_handle *h, size_t floats) {
    if (h->tmp_cap >= floats) return SPHSM_OK;
    if (h->d_tmp) cudaFree(h->d_tmp);
    h->d_tmp = nullptr; h->tmp_cap = 0;
    CU(cudaMalloc(&h->d_tmp, floats * sizeof(float)));
    h->tmp_cap = floats;
    return SPHSM_OK;
}
static int ensure_itmp(sphsm_handle *h, size_t ints) {
    if (h->itmp_cap >= ints) return SPHSM_OK;
    if (h->d_itmp) cudaFree(h->d_itmp);
    h->d_itmp = nullptr; h->itmp_cap = 0;
    CU(cudaMalloc(&h->d_itmp, ints * sizeof(int)));
    h->itmp_cap = ints;
    return SPHSM_OK;
}
static int ensure_aos(sphsm_handle *h, size_t bytes) {
    if (h->aos_cap_bytes >= bytes) return SPHSM_OK;
    if (h->d_aos) cudaFree(h->d_aos);
    h->d_aos = nullptr; h->aos_cap_bytes = 0;
    CU(cudaMalloc(&h->d_aos, bytes));
    h->aos_cap_bytes = bytes;
    return SPHSM_OK;
}
// positions (or the grid) are about to change behind pass B's back: its pre-filed counts for the next sort are void
static void drop_counts(sphsm_handle *h) {
    if (!h->counts_ready) return;
    h->counts_ready = false;
    if (h->cell_count) cudaMemsetAsync(h->cell_count, 0, ((size_t)h->dp.num_cells + 2 + SCAN_IPT) * sizeof(uint32_t), h->stream);
}
static void state_changed(sphsm_handle *h, bool rest) {
    drop_counts(h);
    h->grid_valid = false;
    h->slot_of_valid = false;
    h->inter_live = true;
    h->prev_vel_valid = false;
    h->x1_early_valid = false;
    h->x1_floor = h->x1_seq;  // the populations may have changed: full-size messages until X1_LAG fresh exchanges have been seen
    if (rest) {
        h->goal_pv_stale = false;  // uploads / Init_Fluid write GOAL, PV and their frozen copies
        h->rest_dirty = true;
        h->slab_applied = false;  // the particle set was replaced: sphsm_comm_set_slab must be applied again
    }
}

static FreezeSrc freeze_source(const sphsm_handle *h) {
    FreezeSrc f;
    f.src = (h->prm.diagnostics || !h->goal_pv_stale) ? 1 : 2;
    f.strict = h->prm.strict;
    f.sm = h->sm;
    f.prev_vel = h->prev_vel_valid ? h->alt.VEL : nullptr;
    f.vals = h->perm;
    return f;
}

// Host-side estimate of the mean cell occupancy of a small particle set, from the positions as the caller hands them in
// (Init_Fluid / upload): what decides between the thread-per-particle and the warp-per-particle passes is candidates per
// stencil row, i.e. particles per occupied cell, and the host never sees the cell table.  Only tracked up to the warp-path limit.
static void note_host_positions(sphsm_handle *h, const float *x, size_t stride_floats, int count, bool reset) {
    if (reset) h->host_cells.clear();
    if (h->n + count > 4 * WARP_PATH_MAX || (int)h->host_cells.size() > 4 * WARP_PATH_MAX) return;
    const float cs = h->prm.kernel_h;
    for (int k = 0; k < count; k++) {
        const float *q = x + (size_t)k * stride_floats;
        if (!(fabsf(q[0]) < 1e9f && fabsf(q[1]) < 1e9f && fabsf(q[2]) < 1e9f)) continue;  // NaN / absurd: no cell
        const long long cx = (long long)(q[0] / cs), cy = (long long)(q[1] / cs), cz = (long long)(q[2] / cs);
        h->host_cells.insert((cx & 0x1fffff) | ((cy & 0x1fffff) << 21) | ((cz & 0x1fffff) << 42));
    }
}

extern "C" int sphsm_init_fluid(sphsm_handle *h, const float *xyz, int n) {
    if (!h || (!xyz && n > 0) || n < 0) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    const int take = std::min(n, h->prm.capacity - h->n);  // cpp:103: the rest is silently dropped
    if (take <= 0) return SPHSM_OK;
    int rc;
    if ((rc = ensure_tmp(h, (size_t)take * 3)) != 0) return rc;
    CU(cudaMemcpyAsync(h->d_tmp, xyz, (size_t)take * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    LAUNCH(k_init_particles, cdiv(take, 256), 256, h->n, take, h->d_tmp, h->cur, h->prm.particle_mass, h->prm.stand_density);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));  // xyz may be pageable / freed by the caller
    note_host_positions(h, xyz, 3, take, h->n == 0);
    set_n(h, h->n + take);
    state_changed(h, true);
    return SPHSM_OK;
}

extern "C" int sphsm_upload_aos(sphsm_handle *h, const void *particles, int n, int stride) {
    if (!h || !particles || n < 0 || stride < SPHSM_PARTICLE_STRIDE) return SPHSM_ERR_INVALID;
    if (n > h->prm.capacity) return fail(h, SPHSM_ERR_CAPACITY, "more particles than capacity");
    CU(cudaSetDevice(h->prm.device));
    int rc;
    if ((rc = ensure_aos(h, (size_t)std::max(n, 1) * stride)) != 0) return rc;
    CU(cudaMemcpyAsync(h->d_aos, particles, (size_t)n * stride, cudaMemcpyHostToDevice, h->stream));
    if (n > 0) LAUNCH(k_aos_to_soa, cdiv(n, 256), 256, 0, n, h->d_aos, stride, h->cur);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    if (stride % 4 == 0) {
        h->n = 0;
        note_host_positions(h, reinterpret_cast<const float *>(static_cast<const uint8_t *>(particles) + OFF_POS), (size_t)stride / 4, n, true);
    } else h->host_cells.clear();
    set_n(h, n);
    state_changed(h, true);
    return SPHSM_OK;
}

extern "C" int sphsm_download_aos(sphsm_handle *h, void *particles, int n, int stride) {
    if (!h || !particles || n < 0 || stride < SPHSM_PARTICLE_STRIDE) return SPHSM_ERR_INVALID;
    // slab mode: n counts GLOBAL particles (the caller's array is indexed by original id); only the particles this rank
    // owns are written, everything else in the caller's array keeps its bytes
    const bool slab = h->dp.slab_on != 0;
    int rc;
    if ((rc = slab_refresh(h)) != 0) return rc;
    if (n > (slab ? h->prm.capacity : h->n)) return fail(h, SPHSM_ERR_INVALID, "n exceeds the number of particles");
    CU(cudaSetDevice(h->prm.device));
    if ((rc = ensure_aos(h, (size_t)std::max(std::max(h->n, n), 1) * stride)) != 0) return rc;
    if (stride != SPHSM_PARTICLE_STRIDE || slab)  // keep the caller's other bytes: round-trip through the device image
        CU(cudaMemcpyAsync(h->d_aos, particles, (size_t)n * stride, cudaMemcpyHostToDevice, h->stream));
    const int nown = h->dp.own_end - h->dp.own_begin;
    if (nown > 0) LAUNCH(k_soa_to_aos, cdiv(nown, 256), 256, h->dp.own_begin, nown, h->cur, h->d_aos, stride);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(particles, h->d_aos, (size_t)n * stride, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return SPHSM_OK;
}

extern "C" int sphsm_download_positions(sphsm_handle *h, float *xyz, int n) {
    if (!h || !xyz || n < 0) return SPHSM_ERR_INVALID;
    const bool slab = h->dp.slab_on != 0;  // slab mode: n is the GLOBAL count, only owned particles are written
    int rc;
    if ((rc = slab_refresh(h)) != 0) return rc;
    if (n > (slab ? h->prm.capacity : h->n)) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    if ((rc = ensure_tmp(h, (size_t)std::max(std::max(h->n, n), 1) * 3)) != 0) return rc;
    if (slab) CU(cudaMemcpyAsync(h->d_tmp, xyz, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    const int nown = h->dp.own_end - h->dp.own_begin;
    if (nown > 0) LAUNCH(k_positions_out, cdiv(nown, 256), 256, h->dp.own_begin, nown, h->cur, h->d_tmp);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(xyz, h->d_tmp, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return SPHSM_OK;
}

static int stim_list(sphsm_handle *h, const float *centres, int m, float radius, float strength) {
    int rc;
    if ((rc = slab_refresh(h)) != 0) return rc;
    if (m <= 0 || h->n <= 0) return SPHSM_OK;
    if ((rc = ensure_tmp(h, (size_t)m * 3)) != 0) return rc;
    CU(cudaMemcpyAsync(h->d_tmp, centres, (size_t)m * 3 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    LAUNCH(k_set_stim_list, cdiv(h->n, 256), 256, h->n, h->cur, h->d_tmp, m, radius, strength);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    return SPHSM_OK;
}

extern "C" int sphsm_set_stim(sphsm_handle *h, float cx, float cy, float cz, float radius, float strength) {
    if (!h) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    const float c[3] = {cx, cy, cz};
    return stim_list(h, c, 1, radius, strength);
}

extern "C" int sphsm_stim_mesh(sphsm_handle *h, const float *xyz, int n) {
    if (!h || (!xyz && n > 0)) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    h->x1_early_valid = false;
    int rc = stim_list(h, xyz, n, 0.01f, h->prm.stim_strength);  // cpp:753
    if (rc) return rc;
    if (h->n > 0) LAUNCH(k_fix_rule, cdiv(h->n, 256), 256, h->dp, h->n, h->cur, 0, freeze_source(h));
    CU(cudaGetLastError());
    h->rest_dirty = true;
    return SPHSM_OK;
}

extern "C" int sphsm_stim_cube(sphsm_handle *h, const float *xyz, int n) {
    if (!h || (!xyz && n > 0)) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    std::vector<float> sel;
    for (int i = 0; i < n; i++) {  // the position filter of cpp:727 (double-literal comparisons)
        const float px = xyz[3 * i], pz = xyz[3 * i + 2];
        if (((double)px >= 0.45 && (double)px <= 0.48) || ((double)px > 1.0 && pz <= 1.05f)) {
            sel.push_back(px); sel.push_back(xyz[3 * i + 1]); sel.push_back(pz);
        }
    }
    h->x1_early_valid = false;
    int rc = stim_list(h, sel.data(), (int)(sel.size() / 3), 0.001f, h->prm.stim_strength);  // cpp:728
    if (rc) return rc;
    if (h->n > 0) LAUNCH(k_fix_rule, cdiv(h->n, 256), 256, h->dp, h->n, h->cur, 1, freeze_source(h));
    CU(cudaGetLastError());
    h->rest_dirty = true;
    return SPHSM_OK;
}

extern "C" int sphsm_set_stim_box(sphsm_handle *h, const float lo[3], const float hi[3], float strength) {
    if (!h || !lo || !hi) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    const int n_k = h->dp.slab_on ? std::max(h->n_bound, h->n) : h->n;  // (dead slots hold NaN positions: never inside)
    if (n_k > 0) LAUNCH(k_set_stim_box, cdiv(n_k, 256), 256, n_k, h->cur, lo[0], lo[1], lo[2], hi[0], hi[1], hi[2], strength);
    CU(cudaGetLastError());
    return SPHSM_OK;
}

extern "C" int sphsm_stim_off(sphsm_handle *h) {
    if (!h) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    h->x1_early_valid = false;  // (Vm of the halo copies already sent would be stale)
    const int n_k = h->dp.slab_on ? std::max(h->n_bound, h->n) : h->n;  // slab mode: the bound (dead slots are harmless to reset)
    if (n_k > 0) LAUNCH(k_stim_off, cdiv(n_k, 256), 256, n_k, h->cur);
    CU(cudaGetLastError());
    return SPHSM_OK;
}

extern "C" int sphsm_set_masks(sphsm_handle *h, const uint8_t *fixed, const float *stim, int n) {
    // slab mode: the arrays are indexed by ORIGINAL (global) id, so they hold the global particle count
    if (!h || n != (h->dp.slab_on ? h->n_global : h->n)) return fail(h, SPHSM_ERR_INVALID, "set_masks needs exactly num_particles entries");
    if (n == 0 || (!fixed && !stim)) return SPHSM_OK;
    CU(cudaSetDevice(h->prm.device));
    int rc;
    h->x1_early_valid = false;
    if ((rc = slab_refresh(h)) != 0) return rc;
    if ((rc = ensure_tmp(h, (size_t)n)) != 0) return rc;
    if ((rc = ensure_itmp(h, (size_t)(n + 3) / 4)) != 0) return rc;
    if (stim) CU(cudaMemcpyAsync(h->d_tmp, stim, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    if (fixed) CU(cudaMemcpyAsync(h->d_itmp, fixed, (size_t)n, cudaMemcpyHostToDevice, h->stream));
    if (h->n > 0)
        LAUNCH(k_set_masks, cdiv(h->n, 256), 256, h->dp, h->n, h->cur, fixed ? (const uint8_t *)h->d_itmp : nullptr, stim ? h->d_tmp : nullptr,
               freeze_source(h), (const int *)nullptr);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(h->stream));
    if (fixed) h->rest_dirty = true;
    return SPHSM_OK;
}

static void trace_mark(sphsm_handle *h, const char *label, bool side = false);  // SPHSM_TRACE (sphsm_host_slab.cuh)
static void record_clear(sphsm_handle *h);  // sphsm_host_record.cuh
static void egm_clear(sphsm_handle *h);     // sphsm_host_egm.cuh
#include "sphsm_host_io.cuh"      // snapshot / restart, asynchronous per-frame I/O
#include "sphsm_host_record.cuh"  // activation maps / probe traces, the step counter and the per-step hook they share; sphsm_record_*
#include "sphsm_host_egm.cuh"     // electrograms at virtual electrodes: sphsm_egm_* / sphsm_get_egm
#include "sphsm_host_step.cuh"    // timers, neighbour grid, shape-matching sums, staged / fused step, graph replay

extern "C" int sphsm_step(sphsm_handle *h, int nsteps) {
    if (!h || nsteps < 0) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    if (h->comm_mode == 2) return fail(h, SPHSM_ERR_COMM, "a local group steps through sphsm_step_group");
    if (h->failed) return fail(h, SPHSM_ERR_COMM, "the slab group stopped after a step error; re-upload the particle set and apply the slab again");
    int rc0 = observe_sync(h);
    if (rc0) return rc0;
    CU(cudaEventRecord(h->ev_step0, h->stream));
    if (h->comm_mode == 1) {
        for (int s = 0; s < nsteps; s++) {
            int rc = mg_step_nccl(h);
            if (rc) return rc;
        }
        CU(cudaEventRecord(h->ev_step1, h->stream));
        return SPHSM_OK;
    }
    for (int s = 0; s < nsteps; s++) {
        int rc;
        if (h->stage_timing) rc = h->prm.strict ? timed_staged_step<true>(h) : timed_staged_step<false>(h);
        else rc = h->prm.strict ? fused_step<true>(h) : graph_step(h);
        if (rc) return rc;
        h->total_steps++;
    }
    CU(cudaEventRecord(h->ev_step1, h->stream));
    return SPHSM_OK;
}

extern "C" int sphsm_stage(sphsm_handle *h, int stage) {
    if (!h) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    if (stage == SPHSM_STAGE_STEP) return sphsm_step(h, 1);
    h->inter_live = true;
    return h->prm.strict ? run_stage<true>(h, stage) : run_stage<false>(h, stage);
}

extern "C" int sphsm_sync(sphsm_handle *h) {
    if (!h) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    CU(cudaStreamSynchronize(h->h2d_stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaStreamSynchronize(h->d2h_stream));
    CU(cudaGetLastError());
    return SPHSM_OK;
}

extern "C" int sphsm_last_step_ms(sphsm_handle *h, float *ms) {
    if (!h || !ms) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    CU(cudaEventSynchronize(h->ev_step1));
    CU(cudaEventElapsedTime(ms, h->ev_step0, h->ev_step1));
    h->last_step_ms = *ms;
    return SPHSM_OK;
}

// a device-side stopwatch over any sequence of calls on this handle (bench.py: workloads whose timed region is more than one sphsm_step)
extern "C" int sphsm_timer_mark(sphsm_handle *h, int which) {
    if (!h || which < 0 || which > 1) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    CU(cudaEventRecord(h->ev_tm[which], h->stream));
    return SPHSM_OK;
}
extern "C" int sphsm_timer_ms(sphsm_handle *h, float *ms) {
    if (!h || !ms) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    CU(cudaEventSynchronize(h->ev_tm[1]));
    CU(cudaEventElapsedTime(ms, h->ev_tm[0], h->ev_tm[1]));
    return SPHSM_OK;
}

extern "C" int sphsm_profile_step(sphsm_handle *h, int nsteps, float out_ms[SPHSM_NUM_KERNEL_GROUPS]) {
    if (!h || !out_ms || nsteps <= 0) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    for (int g = 0; g < SPHSM_NUM_KERNEL_GROUPS; g++) { h->group_ms[g] = 0.f; h->group_launches[g] = 0; }
    int rc = observe_sync(h);
    if (rc) return rc;
    h->profiling = true;
    for (int s = 0; s < nsteps && rc == SPHSM_OK; s++) {
        if (h->comm_mode == 1) { rc = mg_step_nccl(h); continue; }
        rc = h->prm.strict ? fused_step<true>(h) : fused_step<false>(h);
        if (rc == SPHSM_OK) h->total_steps++;
    }
    h->profiling = false;
    for (int g = 0; g < SPHSM_NUM_KERNEL_GROUPS; g++) out_ms[g] = h->group_ms[g] / (float)nsteps;
    return rc;
}

extern "C" const char *sphsm_kernel_group_name(int g) { return (g >= 0 && g < SPHSM_NUM_KERNEL_GROUPS) ? kGroupNames[g] : ""; }

extern "C" int sphsm_num_particles(sphsm_handle *h) { return h ? h->n : SPHSM_ERR_INVALID; }
extern "C" int sphsm_num_cells(sphsm_handle *h) { return h ? h->dp.g[0] * h->dp.g[1] * h->dp.g[2] : SPHSM_ERR_INVALID; }
extern "C" int sphsm_grid_size(sphsm_handle *h, int out3[3]) {
    if (!h || !out3) return SPHSM_ERR_INVALID;
    for (int a = 0; a < 3; a++) out3[a] = h->dp.g[a];
    return SPHSM_OK;
}
extern "C" int sphsm_total_time_steps(sphsm_handle *h) { return h ? h->total_steps : SPHSM_ERR_INVALID; }

extern "C" int sphsm_enable_stage_timing(sphsm_handle *h, int on) {
    if (!h) return SPHSM_ERR_INVALID;
    h->stage_timing = on != 0;
    return SPHSM_OK;
}
extern "C" int sphsm_get_stage_times(sphsm_handle *h, double out7[7]) {
    if (!h || !out7) return SPHSM_ERR_INVALID;
    for (int k = 0; k < 7; k++) out7[k] = h->stage_time[k];
    return SPHSM_OK;
}
extern "C" int sphsm_get_launch_count(sphsm_handle *h, long long *launches) {
    if (!h || !launches) return SPHSM_ERR_INVALID;
    *launches = h->launches;
    return SPHSM_OK;
}
extern "C" int sphsm_reset_launch_count(sphsm_handle *h) {
    if (!h) return SPHSM_ERR_INVALID;
    h->launches = 0;
    return SPHSM_OK;
}

// ---------------------------------------------------------------------------------------------------
// inspection
extern "C" int sphsm_get_cells_csr(sphsm_handle *h, int *cell_start, int *indices) {
    if (!h || !cell_start || !indices) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    int rc;
    if (!h->grid_valid && (rc = build_grid(h, nullptr)) != 0) return rc;
    const DevParams &d = h->dp;
    const int n = h->n, ncell = d.g[0] * d.g[1] * d.g[2];
    std::vector<int> cs((size_t)d.num_cells + 2);
    std::vector<int> ids(std::max(n, 1));
    CU(cudaMemcpyAsync(cs.data(), h->cell_start, cs.size() * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(ids.data(), h->cur.ID, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    // internal key -> the reference's hash x + Gx*(y + Gy*z) (cpp:142); stable counting sort keeps slot order
    std::vector<int> ref_hash(n, -1);  // slots of the limbo bucket (outside the grid) stay -1
    std::fill(cell_start, cell_start + ncell + 1, 0);
    for (int k = 0; k < d.num_cells; k++) {
        if (cs[k + 1] == cs[k]) continue;
        int c[3];
        c[d.perm[0]] = k % d.ga - 1;  // (the table has a border cell on either side of these two axes)
        c[d.perm[1]] = (k / d.ga) % d.gb - 1;
        c[d.perm[2]] = k / (d.ga * d.gb) + d.c_off;
        const int rh = c[0] + d.g[0] * (c[1] + d.g[1] * c[2]);
        for (int s = cs[k]; s < cs[k + 1]; s++) ref_hash[s] = rh;
        cell_start[rh + 1] += cs[k + 1] - cs[k];
    }
    for (int c = 0; c < ncell; c++) cell_start[c + 1] += cell_start[c];
    std::vector<int> cursor(cell_start, cell_start + ncell);
    for (int s = 0; s < n; s++)
        if (ref_hash[s] >= 0) indices[cursor[ref_hash[s]]++] = ids[s];
    // the reference's bucket order is ascending particle index
    for (int c = 0; c < ncell; c++) std::sort(indices + cell_start[c], indices + cell_start[c + 1]);
    return SPHSM_OK;
}

extern "C" int sphsm_get_neighbor_sets(sphsm_handle *h, int kind, const int *query, int n_query, int cap, int *counts, int *indices) {
    if (!h || !query || !counts || !indices || n_query < 0 || cap <= 0 || kind < 0 || kind > 3) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    for (int i = 0; i < n_query; i++)
        if (query[i] < 0 || query[i] >= h->n) return fail(h, SPHSM_ERR_INVALID, "query index out of range");
    if (n_query == 0) return SPHSM_OK;
    int rc;
    if (!h->grid_valid && (rc = build_grid(h, nullptr)) != 0) return rc;
    if ((rc = ensure_slot_of(h)) != 0) return rc;
    if ((rc = ensure_itmp(h, (size_t)n_query * (2 + (size_t)cap))) != 0) return rc;
    int *d_query = h->d_itmp, *d_counts = h->d_itmp + n_query, *d_idx = h->d_itmp + 2 * (size_t)n_query;
    CU(cudaMemcpyAsync(d_query, query, (size_t)n_query * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    LAUNCH(k_neighbor_sets, cdiv(n_query, 64), 64, h->dp, h->cur, h->cell_start, h->slot_of, d_query, n_query, kind, cap, d_counts, d_idx);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(counts, d_counts, (size_t)n_query * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(indices, d_idx, (size_t)n_query * cap * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < n_query; i++) std::sort(indices + (size_t)i * cap, indices + (size_t)i * cap + std::min(counts[i], cap));
    return SPHSM_OK;
}

extern "C" int sphsm_get_sm_transform(sphsm_handle *h, float cm[3], float ocm[3], float xform[27]) {
    if (!h || !cm || !ocm || !xform) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    SmState s;
    CU(cudaMemcpyAsync(&s, h->sm, sizeof s, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    memcpy(cm, s.cm, sizeof s.cm);
    memcpy(ocm, s.ocm, sizeof s.ocm);
    memcpy(xform, s.xform, sizeof s.xform);
    return SPHSM_OK;
}

#include "sphsm_host_slab.cuh"  // multi-GPU slab layer (NCCL and virtual ranks)
