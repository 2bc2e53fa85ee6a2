// sphsm_host_slab.cuh — the multi-GPU slab layer: NCCL loader, communicator setup, slab bookkeeping, exchanges, the phase program of the slab step (NCCL and virtual ranks)
// Host code of libsphsm_b200.so, textually included by sphsm_capi.cu (one translation unit: the handle, the LAUNCH / CU macros and
// the static helpers defined there are in scope).
#pragma once

// ---------------------------------------------------------------------------------------------------
// multi-GPU slab layer, host side.  NCCL is resolved at run time (dlopen), so single-GPU hosts need no NCCL.
typedef struct { char internal[128]; } nccl_unique_id;
struct NcclApi {
    void *lib = nullptr;
    int (*GetUniqueId)(nccl_unique_id *) = nullptr;
    int (*CommInitRank)(void **, int, nccl_unique_id, int) = nullptr;
    int (*CommSplit)(void *, int, int, void **, void *) = nullptr;  // optional (NCCL >= 2.18)
    int (*CommDestroy)(void *) = nullptr;
    int (*Send)(const void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*Recv)(void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, void *, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
enum { NCCL_CHAR = 0, NCCL_FLOAT = 7, NCCL_DOUBLE = 8, NCCL_SUM = 0 };  // ncclDataType_t / ncclRedOp_t values (nccl.h)

static int load_nccl(sphsm_handle *h) {
    if (g_nccl.lib) return SPHSM_OK;
    const char *names[] = {getenv("SPHSM_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    void *lib = nullptr;
    for (const char *nm : names)
        if (nm && (lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL)) != nullptr) break;
    if (!lib) return fail(h, SPHSM_ERR_COMM, "libnccl.so.2 not found (set SPHSM_NCCL_LIB)");
    bool ok = true;
    auto sym = [&](const char *nm) { void *f = dlsym(lib, nm); if (!f) ok = false; return f; };
    g_nccl.GetUniqueId = (int (*)(nccl_unique_id *))sym("ncclGetUniqueId");
    g_nccl.CommInitRank = (int (*)(void **, int, nccl_unique_id, int))sym("ncclCommInitRank");
    g_nccl.CommSplit = (int (*)(void *, int, int, void **, void *))dlsym(lib, "ncclCommSplit");
    g_nccl.CommDestroy = (int (*)(void *))sym("ncclCommDestroy");
    g_nccl.Send = (int (*)(const void *, size_t, int, int, void *, cudaStream_t))sym("ncclSend");
    g_nccl.Recv = (int (*)(void *, size_t, int, int, void *, cudaStream_t))sym("ncclRecv");
    g_nccl.AllReduce = (int (*)(const void *, void *, size_t, int, int, void *, cudaStream_t))sym("ncclAllReduce");
    g_nccl.GroupStart = (int (*)())sym("ncclGroupStart");
    g_nccl.GroupEnd = (int (*)())sym("ncclGroupEnd");
    g_nccl.GetErrorString = (const char *(*)(int))sym("ncclGetErrorString");
    if (!ok) return fail(h, SPHSM_ERR_COMM, "libnccl is missing a required entry point");
    g_nccl.lib = lib;
    g_nccl_destroy = g_nccl.CommDestroy;
    return SPHSM_OK;
}
#define NC(call)                                                                                        \
    do {                                                                                                \
        int r_ = (call);                                                                                \
        if (r_ != 0) {                                                                                  \
            std::string m_ = std::string(#call) + " failed: " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r_) : "?"); \
            if (h) h->err = m_; else g_create_error = m_;                                               \
            return SPHSM_ERR_COMM;                                                                      \
        }                                                                                               \
    } while (0)

static int comm_alloc(sphsm_handle *h) {
    if (h->msg_send[0]) return SPHSM_OK;
    const int cap = h->send_cap;  // fixed at create (array room was allocated for it)
    for (int k = 0; k < 2; k++) {
        CU(cudaMalloc(&h->msg_send[k], msg_bytes(cap)));
        CU(cudaMalloc(&h->msg_recv[k], msg_bytes(cap)));
        CU(cudaMemset(h->msg_send[k], 0, 16));
        CU(cudaMemset(h->msg_recv[k], 0, 16));
    }
    CU(cudaMalloc(&h->d_err, 4 * sizeof(int)));
    CU(cudaMemset(h->d_err, 0, 4 * sizeof(int)));
    for (int k = 0; k < 2; k++) {
        CU(cudaMalloc(&h->d_meta[k], sizeof(SlabMeta)));
        CU(cudaMemset(h->d_meta[k], 0, sizeof(SlabMeta)));
    }
    CU(cudaMalloc(&h->d_count, sizeof(int)));
    CU(cudaMalloc(&h->d_x1rec, sphsm_handle::X1_RING * 4 * sizeof(int)));
    CU(cudaMemset(h->d_x1rec, 0, sphsm_handle::X1_RING * 4 * sizeof(int)));
    CU(cudaMallocHost(&h->h_x1rec, sphsm_handle::X1_RING * 4 * sizeof(int)));
    h->x1_send_cap[0] = h->x1_send_cap[1] = h->x1_recv_cap[0] = h->x1_recv_cap[1] = cap;
    CU(cudaMallocHost(&h->h_ring, sphsm_handle::META_RING * 8 * sizeof(int)));
    for (auto &e : h->ev_ring) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    CU(cudaDeviceSynchronize());  // (legacy-stream memsets above: the handle's non-blocking streams do not wait for them)
    return SPHSM_OK;
}

// ---- push exchange / push allreduce set-up: every rank maps every other rank's block (CUDA IPC over NVLink); all ranks or none ---
// (collective: called by every rank from sphsm_comm_init, whatever its own outcome so far)
static int p2p_setup(sphsm_handle *h) {
    h->p2p_on = h->p2p_red_on = false;
    const int nr = h->nranks;
    if (nr < 2) return SPHSM_OK;
    const int cap = h->send_cap;
    int ok = (g_p2p && nr <= P2P_MAX_RANKS) ? 1 : 0;
    const size_t hb = sizeof(cudaIpcMemHandle_t);
    std::vector<cudaIpcMemHandle_t> hs(nr);
    memset(hs.data(), 0, hb * nr);
    if (ok && cudaMalloc(&h->p2p_block, p2p_block_bytes(cap, nr)) != cudaSuccess) { ok = 0; h->p2p_block = nullptr; }
    if (ok) {
        ok = cudaMemset(h->p2p_block, 0, p2p_block_bytes(cap, nr)) == cudaSuccess && cudaMemset(h->p2p_block, 0xff, P2P_FLAGS_BYTES) == cudaSuccess &&  // flags = -1
             cudaIpcGetMemHandle(&hs[h->rank], h->p2p_block) == cudaSuccess;
    }
    cudaDeviceSynchronize();  // (the memsets ran in the legacy stream; peers may store into this block as soon as they have mapped it)
    cudaGetLastError();
    uint8_t *d_hs = nullptr;
    double *d_ok = nullptr;
    CU(cudaMalloc(&d_hs, hb * nr));
    CU(cudaMalloc(&d_ok, 2 * sizeof(double)));
    CU(cudaMemcpy(d_hs, hs.data(), hb * nr, cudaMemcpyHostToDevice));
    NC(g_nccl.GroupStart());
    for (int p = 0; p < nr; p++) {
        if (p == h->rank) continue;
        NC(g_nccl.Send(d_hs + hb * h->rank, hb, NCCL_CHAR, p, h->nccl_comm, h->stream));
        NC(g_nccl.Recv(d_hs + hb * p, hb, NCCL_CHAR, p, h->nccl_comm, h->stream));
    }
    NC(g_nccl.GroupEnd());
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(hs.data(), d_hs, hb * nr, cudaMemcpyDeviceToHost));
    h->p2p_all.assign(nr, nullptr);
    for (int p = 0; p < nr && ok; p++) {
        if (p == h->rank) { h->p2p_all[p] = h->p2p_block; continue; }
        void *ptr = nullptr;
        if (cudaIpcOpenMemHandle(&ptr, hs[p], cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) { ok = 0; cudaGetLastError(); }
        else h->p2p_all[p] = static_cast<uint8_t *>(ptr);
    }
    const double mine[2] = {ok ? 1.0 : 0.0, (ok && g_p2p_red) ? 1.0 : 0.0};
    double sum[2] = {0.0, 0.0};
    CU(cudaMemcpy(d_ok, mine, sizeof mine, cudaMemcpyHostToDevice));
    NC(g_nccl.AllReduce(d_ok, d_ok, 2, NCCL_DOUBLE, NCCL_SUM, h->nccl_comm, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpy(sum, d_ok, sizeof sum, cudaMemcpyDeviceToHost));
    cudaFree(d_hs);
    cudaFree(d_ok);
    if ((int)(sum[0] + 0.5) == nr) {
        h->p2p_on = true;
        h->p2p_red_on = (int)(sum[1] + 0.5) == nr;
        h->p2p_slot_bytes = p2p_slot_bytes(cap);
        if (h->rank > 0) h->p2p_peer[0] = h->p2p_all[h->rank - 1];
        if (h->rank < nr - 1) h->p2p_peer[1] = h->p2p_all[h->rank + 1];
        CU(cudaMalloc(&h->d_p2p_all, nr * sizeof(uint8_t *)));
        CU(cudaMemcpy(h->d_p2p_all, h->p2p_all.data(), nr * sizeof(uint8_t *), cudaMemcpyHostToDevice));
    } else {  // some rank could not map a peer (or runs with SPHSM_P2P=0): everybody stays on NCCL
        for (int p = 0; p < nr; p++)
            if (h->p2p_all[p] && h->p2p_all[p] != h->p2p_block) cudaIpcCloseMemHandle(h->p2p_all[p]);
        h->p2p_all.clear();
        if (h->p2p_block) { cudaFree(h->p2p_block); h->p2p_block = nullptr; }
    }
    return SPHSM_OK;
}
extern "C" int sphsm_comm_p2p(sphsm_handle *h) { return !h ? 0 : (h->p2p_on ? 1 : 0) | (h->p2p_red_on ? 2 : 0); }

extern "C" int sphsm_comm_unique_id(void *id128) {
    sphsm_handle *h = nullptr;
    if (!id128) return SPHSM_ERR_INVALID;
    int rc = load_nccl(nullptr);
    if (rc) return rc;
    nccl_unique_id id;
    NC(g_nccl.GetUniqueId(&id));
    memcpy(id128, &id, sizeof id);
    return SPHSM_OK;
}

extern "C" int sphsm_comm_init(sphsm_handle *h, int nranks, int rank, const void *id128) {
    if (!h || !id128 || nranks < 1 || rank < 0 || rank >= nranks) return SPHSM_ERR_INVALID;
    if (h->prm.slab_axis < 0) return fail(h, SPHSM_ERR_INVALID, "create the handle with params.slab_axis = 0, 1 or 2 for multi-GPU");
    if (h->prm.strict) return fail(h, SPHSM_ERR_INVALID, "strict mode is single-GPU only");
    CU(cudaSetDevice(h->prm.device));
    int rc = load_nccl(h);
    if (rc) return rc;
    nccl_unique_id id;
    memcpy(&id, id128, sizeof id);
    NC(g_nccl.CommInitRank(&h->nccl_comm, nranks, id, rank));
    h->nccl_comm_red = h->nccl_comm;
    // SPHSM_SPLIT_COMM=1: allreduce on a second communicator.  Off by default: measured at 8 GPUs / 8M it gained nothing (the
    // allreduce queued behind exchange 1 still ends before the sort does) and the two NCCL kernels then share the SMs.
    if (g_nccl.CommSplit && getenv("SPHSM_SPLIT_COMM")) NC(g_nccl.CommSplit(h->nccl_comm, 0, rank, &h->nccl_comm_red, nullptr));
    h->comm_mode = 1; h->nranks = nranks; h->rank = rank;
    if ((rc = comm_alloc(h)) != 0) return rc;
    return p2p_setup(h);
}

extern "C" int sphsm_comm_init_local(sphsm_handle **hs, int nranks) {
    if (!hs || nranks < 1) return SPHSM_ERR_INVALID;
    for (int r = 0; r < nranks; r++) {
        sphsm_handle *h = hs[r];
        if (!h) return SPHSM_ERR_INVALID;
        if (h->prm.slab_axis < 0) return fail(h, SPHSM_ERR_INVALID, "create the handle with params.slab_axis = 0, 1 or 2 for multi-GPU");
        if (h->prm.strict) return fail(h, SPHSM_ERR_INVALID, "strict mode is single-GPU only");
        if (h->prm.device != hs[0]->prm.device || h->prm.capacity != hs[0]->prm.capacity)
            return fail(h, SPHSM_ERR_INVALID, "a local group shares one device and one capacity");
        CU(cudaSetDevice(h->prm.device));
        h->comm_mode = 2; h->nranks = nranks; h->rank = r;
        int rc = comm_alloc(h);
        if (rc) return rc;
    }
    return SPHSM_OK;
}

// ---- the slot ranges of the slab: written on the device by every sort, read back by the host with a fixed lag --------------
// The kernels of the slab step take their ranges from SlabMeta in device memory and their grids from the bounds below, so the
// host only needs the numbers for (a) those bounds, (b) the accessors, (c) the error state.  Each sort queues a 32-byte copy of
// the fresh SlabMeta into a ring of pinned slots; the NCCL step applies the copy of step t - META_LAG at the start of step t
// (an event wait that has normally completed long before), which keeps the host up to META_LAG steps ahead of the device while
// every rank still sees a given step's error flag at the SAME step (the lag is fixed, not "whatever has arrived").
static bool g_host_prof_early() { static const bool v = getenv("SPHSM_HOST_PROF") != nullptr; return v; }
static double now_us_early() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}
// queue k_mg_meta for the freshly sorted array (it becomes d_meta[meta_cur]) and its read-back
static int slab_meta_launch(sphsm_handle *h, const double *flag_src) {
    const DevParams &d = h->dp;
    if (h->meta_issued - h->meta_consumed >= sphsm_handle::META_RING) return fail(h, SPHSM_ERR_COMM, "internal: slab read-back ring overrun");
    h->meta_cur ^= 1;
    // (this buffer was last read back two sorts ago: its copy has long left, the wait is for form)
    if (h->meta_issued >= 2) CU(cudaStreamWaitEvent(h->launch_stream, h->ev_ring[(h->meta_issued - 2) % sphsm_handle::META_RING], 0));
    LAUNCH(k_mg_meta, 1, 32, h->cell_start, d.num_cells, d.ga * d.gb, d.gcl, h->d_err, flag_src, h->n_bound, h->d_meta[h->meta_cur]);
    // the read-back runs on its own stream: a copy inside the main stream held the gather back by 6-8 us (SPHSM_TRACE at 8 GPUs)
    const int slot = (int)(h->meta_issued % sphsm_handle::META_RING);
    CU(cudaEventRecord(h->ev_meta_ready, h->launch_stream));
    CU(cudaStreamWaitEvent(h->meta_stream, h->ev_meta_ready, 0));
    CU(cudaMemcpyAsync(h->h_ring + 8 * slot, h->d_meta[h->meta_cur], 8 * sizeof(int), cudaMemcpyDeviceToHost, h->meta_stream));
    CU(cudaEventRecord(h->ev_ring[slot], h->meta_stream));
    h->meta_issued++;
    return SPHSM_OK;
}
static void slab_set_bounds(sphsm_handle *h, int n_live, int n_owned) {
    // a step changes the populations by at most the contents of two halo messages; the grids are sized for a few steps of that
    const int slack = 2 * h->send_cap + 4096;
    h->n_bound = std::min(h->alloc_n - 2 * h->send_cap, n_live + slack);
    h->own_bound = std::min(h->alloc_n - 2 * h->send_cap, n_owned + slack);
}
// apply the read-backs up to and including number `upto` (0-based count of sorts) to the host-side fields; blocks until they are there
static int slab_meta_consume(sphsm_handle *h, long long upto) {
    upto = std::min(upto, h->meta_issued - 1);
    while (h->meta_consumed <= upto) {
        const int slot = (int)(h->meta_consumed % sphsm_handle::META_RING);
        const double tw = g_host_prof_early() ? now_us_early() : 0.0;
        CU(cudaEventSynchronize(h->ev_ring[slot]));
        if (tw != 0.0) h->meta_wait_us += now_us_early() - tw;
        const int *m = h->h_ring + 8 * slot;
        h->meta_consumed++;
        h->n = m[0];
        h->dp.n = m[0];
        h->dp.own_begin = m[1];
        h->b2 = m[2];
        h->b3 = m[3];
        h->dp.own_end = m[4];
        slab_set_bounds(h, m[0], m[4] - m[1]);
        const char *what = m[5] ? "a particle crossed more than one cell plane in one step (or left the slab window)"
                           : m[6] ? "halo message overflow or a slab face whose two sides disagree: raise params.reserved[0] (halo capacity)" : nullptr;
        if (what && !h->local_error) {
            h->local_error = 1;
            h->local_error_msg = what;
        }
        if (m[7] != 0) h->peer_error = true;  // the allreduced flag: some rank (maybe this one) has failed
    }
    return SPHSM_OK;
}
// everything queued so far, now (accessors, mutators, virtual ranks): the host fields are exact afterwards
static int slab_refresh(sphsm_handle *h) {
    if (!h->dp.slab_on || h->meta_consumed >= h->meta_issued) return SPHSM_OK;
    return slab_meta_consume(h, h->meta_issued - 1);
}
static int slab_check_local_error(sphsm_handle *h) {
    if (h->local_error) return fail(h, SPHSM_ERR_COMM, h->local_error_msg.c_str());
    return SPHSM_OK;
}

extern "C" int sphsm_comm_set_slab(sphsm_handle *h, int cell_lo, int cell_hi) {
    if (!h) return SPHSM_ERR_INVALID;
    if (!h->comm_mode) return fail(h, SPHSM_ERR_COMM, "sphsm_comm_init first");
    if (cell_lo < 0 || cell_hi > h->dp.gc || cell_hi - cell_lo < 1) return fail(h, SPHSM_ERR_INVALID, "slab must hold at least one cell plane of the grid");
    CU(cudaSetDevice(h->prm.device));
    DevParams &d = h->dp;
    if (!d.slab_on) h->n_global = h->n;
    d.slab_lo = cell_lo; d.slab_hi = cell_hi;
    d.c_off = cell_lo - 1; d.gcl = cell_hi - cell_lo + 2;
    d.num_cells = d.ga * d.gb * d.gcl;
    d.slab_on = 1;
    int rc;
    if ((rc = setup_grid_buffers(h)) != 0) return rc;
    // keep only the owned planes: dead entries sort into the limbo bucket and fall off the end
    h->local_error = 0; h->peer_error = false; h->failed = false;
    h->x1_early_pending = false; h->x1_early_valid = false;
    h->x1_floor = h->x1_seq;
    h->meta_consumed = h->meta_issued;  // (read-backs of an earlier slab are void)
    if (h->d_err) CU(cudaMemsetAsync(h->d_err, 0, 4 * sizeof(int), h->stream));
    h->n_bound = h->alloc_n;
    if (h->n > 0) {
        d.own_begin = 0; d.own_end = h->n;
        LAUNCH(k_mg_filter, cdiv(h->n, 256), 256, h->dp, h->cur);
        h->inter_live = true;
        if ((rc = build_grid(h, nullptr)) != 0) return rc;
        if ((rc = slab_meta_launch(h, nullptr)) != 0 || (rc = slab_refresh(h)) != 0 || (rc = slab_check_local_error(h)) != 0) return rc;
    } else {
        CU(cudaMemsetAsync(h->d_meta[h->meta_cur], 0, sizeof(SlabMeta), h->stream));
        slab_set_bounds(h, 0, 0);
    }
    h->grid_valid = false;
    h->slab_applied = true;
    return SPHSM_OK;
}

extern "C" int sphsm_comm_x1_sizes(sphsm_handle *h, int out[4]) {
    if (!h || !out) return SPHSM_ERR_INVALID;
    out[0] = h->x1_send_cap[0]; out[1] = h->x1_send_cap[1]; out[2] = h->x1_recv_cap[0]; out[3] = h->x1_recv_cap[1];
    return SPHSM_OK;
}

extern "C" int sphsm_comm_info(sphsm_handle *h, int out[8]) {
    if (!h || !out) return SPHSM_ERR_INVALID;
    int rc0 = slab_refresh(h);
    if (rc0) return rc0;
    out[0] = h->comm_mode; out[1] = h->nranks; out[2] = h->rank; out[3] = h->n;
    out[4] = h->dp.own_begin; out[5] = h->dp.own_end; out[6] = h->send_cap; out[7] = h->dp.slab_on;
    return SPHSM_OK;
}

extern "C" int sphsm_download_owned(sphsm_handle *h, int *ids, float *xyz, int cap, int *count) {
    if (!h || !ids || !xyz || !count || cap < 0) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    int rc;
    if ((rc = slab_refresh(h)) != 0) return rc;
    const int first = h->dp.own_begin, nown = h->dp.own_end - h->dp.own_begin;
    *count = nown;
    if (nown > cap) return fail(h, SPHSM_ERR_CAPACITY, "output arrays smaller than the number of owned particles");
    if (nown == 0) return SPHSM_OK;
    if ((rc = ensure_tmp(h, (size_t)nown * 3)) != 0 || (rc = ensure_itmp(h, (size_t)nown)) != 0) return rc;
    LAUNCH(k_mg_owned_out, cdiv(nown, 256), 256, (const int *)nullptr, first, nown, nown, h->cur, h->d_itmp, h->d_tmp, (int *)nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpyAsync(ids, h->d_itmp, (size_t)nown * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(xyz, h->d_tmp, (size_t)nown * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return SPHSM_OK;
}

// ---- collectives: NCCL (one process per GPU) --------------------------------------------------------------------
static unsigned long long p2p_timeout_ns() {
    static const unsigned long long v =
        (unsigned long long)(getenv("SPHSM_P2P_TIMEOUT_S") ? std::max(1, atoi(getenv("SPHSM_P2P_TIMEOUT_S"))) : 120) * 1000000000ull;
    return v;
}
static int comm_allreduce(sphsm_handle *h, int count) {
    if (h->comm_mode != 1 || h->nranks == 1) return SPHSM_OK;  // single GPU; the local group sums between phases
    if (h->p2p_red_on && count <= P2P_RED_MAX) {  // push allreduce: one launch, one NVLink round trip (k_p2p_allreduce)
        LAUNCH(k_p2p_allreduce, 1, 128, h->totals, count, h->rank, h->nranks, (int)(h->red_seq++), h->d_p2p_all, p2p_red_offset(h->send_cap), h->d_err,
               p2p_timeout_ns());
        return SPHSM_OK;
    }
    NC(g_nccl.AllReduce(h->totals, h->totals, (size_t)count, NCCL_DOUBLE, NCCL_SUM, h->nccl_comm_red, h->launch_stream));
    return SPHSM_OK;
}
// Exchange-1 message sizes.  A message carries one cell plane's worth of particles (plus migrants), but how many that is only the
// device knows; sending the full halo capacity every step cost 68 us per step at 8 GPUs / 8M particles (SPHSM_TRACE), 2-4 times
// what the live entries need.  So every unpack files {sent left, sent right, received left, received right} of ITS exchange into a
// small ring that is read back beside the step, and the exchange packed X1_LAG exchanges later is sized from it: my "sent right" of
// exchange q is by construction my right neighbour's "received left" of exchange q (it is the header of the same message, and both
// sides count exchanges alike because every exchange is a matched send / receive), so the two sides of a face always derive the
// same size without talking to each other.  The margin (a quarter + 2048 particles over X1_LAG steps) is far above what a step
// that moves no particle further than one cell plane can add; a message that overflows anyway is flagged like any halo overflow.
// Population changes from outside (uploads, a new slab: collective by contract, like every mutator) reset the history.
static int x1_plan(sphsm_handle *h) {
    const int cap = h->send_cap;
    const long long q = h->x1_seq++, src = q - sphsm_handle::X1_LAG;
    for (int k = 0; k < 2; k++) h->x1_send_cap[k] = h->x1_recv_cap[k] = cap;
    if (!g_x1_dynamic || h->p2p_on) return SPHSM_OK;  // (the push exchange moves the live entries only: nothing to size)
    // the newest exchange at least X1_LAG back that was unpacked (one voided by a mutator before its unpack left no record: on
    // every rank alike) and is still in the ring
    int slot = -1;
    for (long long c = src; c >= 0 && c >= h->x1_floor && c > q - sphsm_handle::X1_RING; c--)
        if (h->x1rec_seq[c % sphsm_handle::X1_RING] == c) { slot = (int)(c % sphsm_handle::X1_RING); break; }
    if (slot < 0) return SPHSM_OK;
    CU(cudaEventSynchronize(h->ev_x1rec[slot]));  // X1_LAG is one more than the SlabMeta lag: the host has already waited for a later copy
    const int *r = h->h_x1rec + 4 * slot;
    auto sized = [cap](int c) {
        const long long m = ((long long)c + c / 4 + 2048 + 255) / 256 * 256;
        return (int)std::min<long long>(cap, m);
    };
    h->x1_send_cap[0] = sized(r[0]); h->x1_send_cap[1] = sized(r[1]);
    h->x1_recv_cap[0] = sized(r[2]); h->x1_recv_cap[1] = sized(r[3]);
    return SPHSM_OK;
}
// the record of the exchange that was just unpacked (k_mg_unpack wrote it) starts its way to the host
static int x1_record_launch(sphsm_handle *h) {
    const long long q = h->x1_seq - 1;
    const int slot = (int)(q % sphsm_handle::X1_RING);
    CU(cudaEventRecord(h->ev_x1rec_ready, h->launch_stream));
    CU(cudaStreamWaitEvent(h->meta_stream, h->ev_x1rec_ready, 0));
    CU(cudaMemcpyAsync(h->h_x1rec + 4 * slot, h->d_x1rec + 4 * slot, 4 * sizeof(int), cudaMemcpyDeviceToHost, h->meta_stream));
    CU(cudaEventRecord(h->ev_x1rec[slot], h->meta_stream));
    h->x1rec_seq[slot] = q;
    return SPHSM_OK;
}
static int nccl_exchange1(sphsm_handle *h, cudaStream_t st) {
    NC(g_nccl.GroupStart());
    if (h->rank > 0) {
        NC(g_nccl.Send(h->msg_send[0], msg_bytes(h->x1_send_cap[0]), NCCL_CHAR, h->rank - 1, h->nccl_comm, st));
        NC(g_nccl.Recv(h->msg_recv[0], msg_bytes(h->x1_recv_cap[0]), NCCL_CHAR, h->rank - 1, h->nccl_comm, st));
    }
    if (h->rank < h->nranks - 1) {
        NC(g_nccl.Send(h->msg_send[1], msg_bytes(h->x1_send_cap[1]), NCCL_CHAR, h->rank + 1, h->nccl_comm, st));
        NC(g_nccl.Recv(h->msg_recv[1], msg_bytes(h->x1_recv_cap[1]), NCCL_CHAR, h->rank + 1, h->nccl_comm, st));
    }
    NC(g_nccl.GroupEnd());
    return SPHSM_OK;
}
// ---- push exchange (p2p_on): where the packing kernels store, the publish, the wait ---------------------------------------------
// message k (0: to the left neighbour, 1: to the right) of the exchange packed last: the arrays are the neighbour's receive slot
// (my left neighbour receives it "from its right": side 1 of its block), the counter stays here (atomics)
static MsgView x1_send_view(sphsm_handle *h, int k) {
    if (!h->p2p_on || !h->p2p_peer[k]) return msg_view(h->msg_send[k], h->x1_send_cap[k]);
    MsgView v = msg_view(p2p_slot(h->p2p_peer[k], h->send_cap, 1 - k, (int)((h->x1_seq - 1) & 1)), h->send_cap);
    v.count = reinterpret_cast<int *>(h->msg_send[k]);
    return v;
}
static MsgView x1_recv_view(sphsm_handle *h, int k) {
    if (!h->p2p_on) return msg_view(h->msg_recv[k], h->x1_recv_cap[k]);
    return msg_view(p2p_slot(h->p2p_block, h->send_cap, k, (int)((h->x1_seq - 1) & 1)), h->send_cap);
}
static int p2p_signal(sphsm_handle *h) {  // (on h->launch_stream, behind the packing kernel)
    const int q = (int)(h->x1_seq - 1), par = q & 1, cap = h->send_cap;
    const bool has_left = h->rank > 0, has_right = h->rank < h->nranks - 1;
    LAUNCH(k_p2p_signal, 1, 32, reinterpret_cast<const int *>(h->msg_send[0]), reinterpret_cast<const int *>(h->msg_send[1]),
           has_left ? reinterpret_cast<int *>(p2p_slot(h->p2p_peer[0], cap, 1, par)) : nullptr,
           has_right ? reinterpret_cast<int *>(p2p_slot(h->p2p_peer[1], cap, 0, par)) : nullptr,
           has_left ? p2p_flag(h->p2p_peer[0], 1) : nullptr, has_right ? p2p_flag(h->p2p_peer[1], 0) : nullptr, q);
    return SPHSM_OK;
}

// exchange 2: pass A's records of the two boundary planes, packed by k_mg_pack2 into the (free by now) message buffers.  The
// messages have a fixed size like those of exchange 1 — the plane populations are only known on the device — and carry the
// population in their header; the receiver (k_mg_unpack2) checks it against its own halo plane.
static int nccl_exchange2(sphsm_handle *h, cudaStream_t st) {
    const size_t bytes = msg2_bytes(h->send_cap);
    NC(g_nccl.GroupStart());
    if (h->rank > 0) {
        NC(g_nccl.Send(h->msg_send[0], bytes, NCCL_CHAR, h->rank - 1, h->nccl_comm, st));
        NC(g_nccl.Recv(h->msg_recv[0], bytes, NCCL_CHAR, h->rank - 1, h->nccl_comm, st));
    }
    if (h->rank < h->nranks - 1) {
        NC(g_nccl.Send(h->msg_send[1], bytes, NCCL_CHAR, h->rank + 1, h->nccl_comm, st));
        NC(g_nccl.Recv(h->msg_recv[1], bytes, NCCL_CHAR, h->rank + 1, h->nccl_comm, st));
    }
    NC(g_nccl.GroupEnd());
    return SPHSM_OK;
}
static int pack2(sphsm_handle *h) {
    const int cap = h->send_cap;
    LAUNCH(k_mg_pack2, cdiv(2 * cap, 256), 256, h->d_meta[h->meta_cur], h->cur, h->rank > 0 ? 1 : 0, h->rank < h->nranks - 1 ? 1 : 0,
           msg2_view(h->msg_send[0], cap), msg2_view(h->msg_send[1], cap), cap);
    return SPHSM_OK;
}
static int unpack2(sphsm_handle *h) {
    const int cap = h->send_cap;
    LAUNCH(k_mg_unpack2, cdiv(2 * cap, 256), 256, h->d_meta[h->meta_cur], h->cur, h->rank > 0 ? 1 : 0, h->rank < h->nranks - 1 ? 1 : 0,
           msg2_view(h->msg_recv[0], cap), msg2_view(h->msg_recv[1], cap), cap, h->d_err, reinterpret_cast<int *>(h->msg_send[0]),
           reinterpret_cast<int *>(h->msg_send[1]));
    return SPHSM_OK;
}

// ---- SPHSM_TRACE: event timeline of the slab step ------------------------------------------------------------------------
static bool trace_on(sphsm_handle *h) {
    if (h->trace_from == -1) h->trace_from = getenv("SPHSM_TRACE") ? atoi(getenv("SPHSM_TRACE")) : -2;
    return h->trace_from >= 0 && h->total_steps >= h->trace_from && h->total_steps < h->trace_from + 3;
}
static void trace_mark(sphsm_handle *h, const char *label, bool side) {
    if (!trace_on(h)) return;
    cudaEvent_t e;
    if (cudaEventCreate(&e) != cudaSuccess) return;
    cudaEventRecord(e, side ? h->side_stream : h->stream);
    h->trace.push_back({e, label, side ? 1 : 0});
}
static void trace_dump(sphsm_handle *h) {
    if (h->trace.empty() || h->total_steps != h->trace_from + 3) return;
    cudaStreamSynchronize(h->stream);
    cudaStreamSynchronize(h->side_stream);
    if (h->rank == 0 || h->rank == h->nranks - 1 || h->rank == h->nranks / 2) {
        std::string out = "[sphsm trace rank " + std::to_string(h->rank) + "] us since the first mark (M = main stream, S = side stream)\n";
        for (auto &t : h->trace) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, h->trace[0].ev, t.ev);
            char b[160];
            snprintf(b, sizeof b, "  %9.1f %s %s\n", ms * 1e3, t.stream ? "S" : "M", t.label);
            out += b;
        }
        fputs(out.c_str(), stderr);
    }
    for (auto &t : h->trace) cudaEventDestroy(t.ev);
    h->trace.clear();
}

// ---- the slab step as phases; every phase ends in the collective named by *coll ----------------------------------------
enum { COLL_NONE = 0, COLL_EXCH1, COLL_ALLREDUCE, COLL_EXCH2, COLL_DONE, COLL_ALLREDUCE_MOMENTS, COLL_EXCH1_TAKEN, COLL_EXCH1_EARLY };
static const int MG_PHASES = 7;

static int mg_forked_allreduce(sphsm_handle *h);
// `sync_meta`: the host waits for the plane boundaries in every step (virtual ranks, profiling, the first step after the
// rest state changed: its sums need host-side extents); otherwise it runs ahead (slab_meta_consume with the fixed lag)
static bool mg_sync_meta(const sphsm_handle *h) { return h->comm_mode != 1 || h->nranks == 1 || h->profiling || h->rest_dirty; }

static int mg_phase(sphsm_handle *h, int phase, int *coll, int *count) {
    const bool diag = h->prm.diagnostics != 0;
    const bool has_left = h->rank > 0, has_right = h->rank < h->nranks - 1;
    const int cap = h->send_cap;
    int rc;
    *coll = COLL_NONE; *count = 0;
    switch (phase) {
        case 0: {  // classify + pack
            if (h->profiling) h->gt = new GroupTimer(h);
            if (mg_sync_meta(h)) {
                if ((rc = slab_refresh(h)) != 0) return rc;
            } else if ((rc = slab_meta_consume(h, h->meta_issued - 1 - sphsm_handle::META_LAG)) != 0) return rc;
            if (h->comm_mode != 1 || h->nranks == 1) {
                if ((rc = slab_check_local_error(h)) != 0) return rc;  // (NCCL ranks stop together, through the allreduced flag)
            }
            h->moments_forked = false;
            trace_mark(h, "step begin");
            if (h->comm_mode == 1 && !h->rest_dirty && !h->profiling) {
                // the moment sums, their allreduce and the solve only need last step's owned slots: they run on the side
                // stream beside the exchange, the hash and the sort, and rejoin before the gather applies the transform
                CU(cudaEventRecord(h->ev_fork, h->stream));
                CU(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
                h->launch_stream = h->side_stream;
                // (the NCCL form of the allreduce is issued after exchange 1, in mg_forked_allreduce: NCCL runs one communicator's
                // operations in issue order whatever their streams, and the exchange must not queue behind the sums; the push
                // allreduce has no such order, it simply takes the same place)
                rc = moments_part(h);
                h->launch_stream = h->stream;
                if (rc) return rc;
                trace_mark(h, "moment sums done", true);
                h->moments_forked = true;
                h->allreduce_pending = true;
                if (h->nccl_comm_red != h->nccl_comm) {  // own communicator: nothing to queue behind
                    if ((rc = mg_forked_allreduce(h)) != 0) return rc;
                    h->allreduce_pending = false;
                }
            }
            if (h->x1_early_pending && h->x1_early_valid) {
                // exchange 1 of this step left at the end of the previous one (phase 5): only the stale halo copies have to go,
                // and nothing in the interior may sit where it should have been sent from (checked beside the sums)
                h->x1_early_pending = false;
                h->drop_in_unpack = true;  // (k_mg_unpack retires them on its way)
                h->check_interior_pending = true;  // (queued behind the allreduce + solve: see mg_check_interior)
                CU(cudaStreamWaitEvent(h->stream, h->ev_x1, 0));
                trace_mark(h, "early exchange 1 awaited");
                if (h->gt) h->gt->end_group(KG_OTHER);
                *coll = COLL_EXCH1_TAKEN;
                return SPHSM_OK;
            }
            h->x1_early_pending = false;  // (voided by a mutator: the messages are packed and exchanged again, on every rank alike)
            CU(cudaMemsetAsync(h->msg_send[0], 0, 16, h->stream));
            CU(cudaMemsetAsync(h->msg_send[1], 0, 16, h->stream));
            if ((rc = x1_plan(h)) != 0) return rc;
            LAUNCH(k_mg_classify, cdiv(std::max(h->n_bound, 1), 256), 256, h->dp, h->cur, has_left ? 1 : 0, has_right ? 1 : 0,
                   x1_send_view(h, 0), x1_send_view(h, 1), h->x1_send_cap[0], h->x1_send_cap[1], h->d_err, h->d_meta[h->meta_cur]);
            if (h->gt) h->gt->end_group(KG_OTHER);
            *coll = COLL_EXCH1;
            return SPHSM_OK;
        }
        case 1: {  // unpack arrivals, hash + sort everything, cell table, plane boundaries
            if (h->n_bound + 2 * cap > h->alloc_n) return fail(h, SPHSM_ERR_CAPACITY, "capacity too small for the halo arrivals");
            const SlabMeta *prev = h->d_meta[h->meta_cur];
            {
                const int slot = (int)((h->x1_seq - 1) % sphsm_handle::X1_RING);  // (its last read-back left X1_RING exchanges ago: a wait for form)
                const bool record = g_x1_dynamic && !h->p2p_on;  // (only the sized ncclSend / ncclRecv messages need the populations on the host)
                if (record && h->x1rec_seq[slot] >= 0) CU(cudaStreamWaitEvent(h->stream, h->ev_x1rec[slot], 0));
                // push exchange: the blocks poll the flag words the neighbours publish this exchange in
                const int *fl = h->p2p_on && has_left ? p2p_flag(h->p2p_block, 0) : nullptr, *fr = h->p2p_on && has_right ? p2p_flag(h->p2p_block, 1) : nullptr;
                LAUNCH(k_mg_unpack, cdiv(2 * cap, 256), 256, prev, h->cur, has_left ? 1 : 0, has_right ? 1 : 0, x1_recv_view(h, 0), x1_recv_view(h, 1), cap,
                       h->x1_recv_cap[0], h->x1_recv_cap[1], h->d_err,
                       (const int *)h->msg_send[0], (const int *)h->msg_send[1], h->d_x1rec + 4 * slot, fl, fr, (int)(h->x1_seq - 1), p2p_timeout_ns(),
                       h->drop_in_unpack ? 1 : 0);
                h->drop_in_unpack = false;
                if (record && (rc = x1_record_launch(h)) != 0) return rc;
            }
            // the entries to sort are the previous live slots + both message regions; the kernels read that count from `prev`,
            // the grids are sized for its upper bound.  (h->n itself is the host's last applied read-back: exact whenever the
            // host waits for the boundaries, i.e. in every step whose rest-state sums need the extent below.)
            h->mom_n = h->n + 2 * cap;
            if (h->gt) h->gt->end_group(KG_OTHER);
            trace_mark(h, "unpacked");
            if ((rc = grid_sort(h, h->gt, &prev->n_live, 2 * cap, h->n_bound + 2 * cap)) != 0) return rc;
            trace_mark(h, "sorted");
            h->reordered = false;
            const int nacc = h->dp.quadratic ? 33 : 15;
            if (h->moments_forked) {
                // the forked chain has delivered the transform and the summed error flag: plane boundaries + flag -> SlabMeta,
                // then the gather, which takes the live count from there
                CU(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
                trace_mark(h, "transform joined");
                h->moments_forked = false;
                if ((rc = slab_meta_launch(h, h->totals + nacc)) != 0) return rc;
                if ((rc = grid_finish(h, h->gt, diag ? 2 : 1, true, &h->d_meta[h->meta_cur]->n_live, h->n_bound + 2 * cap)) != 0) return rc;
                trace_mark(h, "gathered");
                h->reordered = true;
            } else {
                if ((rc = slab_meta_launch(h, nullptr)) != 0) return rc;
                if ((rc = slab_refresh(h)) != 0) return rc;  // n = live slots from here on (host-side extents for the sums below)
            }
            if (h->gt) h->gt->end_group(KG_GRID);
            if (h->rest_dirty) {  // (the sums scan the PRE-gather arrays: old slots + both message regions, mom_n entries)
                if ((rc = rest_part1(h)) != 0) return rc;
                *coll = COLL_ALLREDUCE; *count = 5;
            }
            return SPHSM_OK;
        }
        case 2:
            if (h->rest_dirty) {
                if ((rc = rest_part2(h)) != 0) return rc;
                *coll = COLL_ALLREDUCE; *count = 90;
            }
            return SPHSM_OK;
        case 3:
            if (h->reordered) return SPHSM_OK;
            if (h->rest_dirty && (rc = rest_part3(h)) != 0) return rc;
            // (not forked: the per-step sums run here, over the PREVIOUS layout's owned range, which the arrays still have)
            h->meta_cur ^= 1;
            rc = moments_part(h);
            h->meta_cur ^= 1;
            if (rc) return rc;
            *coll = COLL_ALLREDUCE_MOMENTS; *count = h->dp.quadratic ? 33 : 15;
            return SPHSM_OK;
        case 4: {  // solve, gather + stage 2, pass A
            if (memcmp(&h->dp, &h->dp_uploaded, sizeof(DevParams)) != 0) {
                h->dp_uploaded = h->dp;
                CU(cudaMemcpyAsync(h->d_dp, &h->dp_uploaded, sizeof(DevParams), cudaMemcpyHostToDevice, h->stream));
            }
            const SlabMeta *m = h->d_meta[h->meta_cur];
            if (!h->reordered) {
                LAUNCH(k_sm_solve, 1, 1, h->dp, h->totals, h->sm);
                h->mom_n = 0;
                if (h->gt) h->gt->end_group(KG_MOMENTS);
                if ((rc = grid_finish(h, h->gt, diag ? 2 : 1, true, &m->n_live, h->n_bound + 2 * cap)) != 0) return rc;
            } else {
                h->mom_n = 0;
                if (h->gt) h->gt->end_group(KG_MOMENTS);
            }
            // NCCL mode with at least three owned planes: pass A on the two boundary planes first, their V / S records travel
            // on the side stream while the interior planes are computed here (and pass B's interior after them)
            h->split = h->comm_mode == 1 && h->nranks > 1 && !h->profiling && h->dp.slab_hi - h->dp.slab_lo >= 3;
            if (h->split) {
                // side stream (high priority): pass A on the two boundary planes -> exchange 2 -> pass B on them;
                // main stream: pass A, then pass B on the interior planes.  Cross dependencies: pass B's interior reads the
                // boundary planes' pass-A records (ev_bnd), pass B's boundary reads the interior's (ev_int).
                CU(cudaEventRecord(h->ev_fork, h->stream));
                CU(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
                h->launch_stream = h->side_stream;
                rc = launch_pass_a(h, 0, 2 * cap, 0, 0, m->rng_bnd);
                if (!rc) rc = pack2(h);
                h->launch_stream = h->stream;
                if (rc) return rc;
                trace_mark(h, "pass A boundary + pack2 done", true);
                CU(cudaEventRecord(h->ev_bnd, h->side_stream));
                if ((rc = launch_pass_a(h, 0, h->own_bound, 0, 0, m->rng_int)) != 0) return rc;  // (queued before the NCCL calls: they take host time)
                CU(cudaEventRecord(h->ev_int, h->stream));
                trace_mark(h, "pass A interior done");
                // pass B is cut two planes deep: the planes at least two away from a face read no boundary-plane record at all, so
                // they follow pass A's interior directly; the two outer planes of either side wait for exchange 2 on the side stream
                // (they do not need the boundary planes' records, but everything queued on the side stream before them — the interior
                // check reads the buffer pass B is about to overwrite with the new positions — must have finished: ev_bnd is long past)
                CU(cudaStreamWaitEvent(h->stream, h->ev_bnd, 0));
                if ((rc = launch_pass_b(h, 0, h->own_bound, diag, 0, 0, false, m->rng_int2)) != 0) return rc;
                trace_mark(h, "pass B inner planes done");
                rc = nccl_exchange2(h, h->side_stream);
                trace_mark(h, "exchange 2 done", true);
                return rc;
            }
            if ((rc = launch_pass_a(h, 0, h->own_bound, 0, 0, m->rng_all)) != 0) return rc;
            if ((rc = pack2(h)) != 0) return rc;
            if (h->gt) h->gt->end_group(KG_PASS_A);
            *coll = COLL_EXCH2;
            return SPHSM_OK;
        }
        case 5: {  // pass B on the owned slots
            if (h->gt) h->gt->end_group(KG_OTHER);  // exchange 2
            const SlabMeta *m = h->d_meta[h->meta_cur];
            if (h->split) {  // the outer planes wait for exchange 2 (stream order) and for pass A's interior (ev_int)
                CU(cudaStreamWaitEvent(h->side_stream, h->ev_int, 0));
                h->launch_stream = h->side_stream;
                rc = unpack2(h);
                if (!rc) rc = launch_pass_b(h, 0, 4 * cap, diag, 0, 0, false, m->rng_bnd2);
                // their new positions decide what the neighbours get next step: pack it now and let exchange 1 travel while the
                // main stream is still busy with the inner planes
                if (!rc) rc = x1_plan(h);
                if (!rc) rc = [&]() -> int {
                    LAUNCH(k_mg_classify_rng, cdiv(4 * cap, 256), 256, h->dp, h->cur, (const float4 *)h->alt.P, m->rng_bnd2, has_left ? 1 : 0, has_right ? 1 : 0,
                           x1_send_view(h, 0), x1_send_view(h, 1), h->x1_send_cap[0], h->x1_send_cap[1], h->d_err);
                    return SPHSM_OK;
                }();
                h->launch_stream = h->stream;
                if (rc) return rc;
                trace_mark(h, "pass B outer planes + classify done", true);
                *coll = COLL_EXCH1_EARLY;
                return SPHSM_OK;
            }
            if ((rc = unpack2(h)) != 0) return rc;
            if ((rc = launch_pass_b(h, 0, h->own_bound, diag, 0, 0, false, m->rng_all)) != 0) return rc;
            return SPHSM_OK;
        }
        case 6: {  // the two streams meet; bookkeeping
            if (h->split) {
                trace_mark(h, "early exchange 1 done", true);
                CU(cudaEventRecord(h->ev_join, h->side_stream));
                CU(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
                trace_mark(h, "step end (streams joined)");
            }
            std::swap(h->cur.P, h->alt.P);
            if (h->gt) h->gt->end_group(KG_PASS_B);
            if (observe_on(h)) {  // over the owned slots this step integrated (both streams have joined)
                if ((rc = observe_launch(h, h->d_meta[h->meta_cur]->rng_all, h->own_bound)) != 0) return rc;
                if (h->gt) h->gt->end_group(KG_OTHER);
            }
            if (h->gt) {
                h->gt->finish();
                delete h->gt;
                h->gt = nullptr;
            }
            CU(cudaGetLastError());
            h->grid_valid = false;
            h->inter_live = false;
            h->goal_pv_stale = !diag;
            h->prev_vel_valid = true;
            h->total_steps++;
            trace_dump(h);
            *coll = COLL_DONE;
            return SPHSM_OK;
        }
    }
    return fail(h, SPHSM_ERR_INVALID, "bad phase");
}

// beside the sort, on the side stream BEHIND the moment chain (in front of it, it delayed the allreduce by its own 8 us)
static int mg_check_interior(sphsm_handle *h) {
    if (!h->check_interior_pending) return SPHSM_OK;
    h->check_interior_pending = false;
    const bool has_left = h->rank > 0, has_right = h->rank < h->nranks - 1;
    if (!h->moments_forked) {  // (the side stream is not forked in this step: order it behind the main stream first)
        CU(cudaEventRecord(h->ev_fork, h->stream));
        CU(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
    }
    h->launch_stream = h->side_stream;
    // (h->meta_cur still names the previous layout here: the sort of this step has not been queued yet)
    int rc = [&]() -> int {
        LAUNCH(k_mg_check_interior, cdiv(std::max(h->own_bound, 1), 256), 256, h->dp, h->cur.P, h->d_meta[h->meta_cur], has_left ? 1 : 0, has_right ? 1 : 0,
               h->d_err);
        return SPHSM_OK;
    }();
    h->launch_stream = h->stream;
    return rc;
}

static int mg_check(sphsm_handle *h) {
    if (!h->slab_applied) return fail(h, SPHSM_ERR_COMM, "sphsm_comm_set_slab must be applied after the particle set is uploaded");
    if (h->stage_timing) return fail(h, SPHSM_ERR_INVALID, "stage timing is single-GPU only");
    return SPHSM_OK;
}

// second half of the forked moment chain: allreduce + solve on the side stream, then the join event
static int mg_forked_allreduce(sphsm_handle *h) {
    h->launch_stream = h->side_stream;
    int rc = moment_allreduce(h);
    trace_mark(h, "allreduce done", true);
    if (!rc) rc = [&]() -> int { LAUNCH(k_sm_solve, 1, 1, h->dp, h->totals, h->sm); return SPHSM_OK; }();
    h->launch_stream = h->stream;
    if (rc) return rc;
    trace_mark(h, "solve done", true);
    CU(cudaEventRecord(h->ev_join, h->side_stream));
    return SPHSM_OK;
}

// SPHSM_HOST_PROF=1: host-side time of the slab step per phase (kernel launches / NCCL calls / the read-back wait), printed
// by rank 0 every 64 steps — tells a launch-bound step from a device-bound one (the device side has its own tool: SPHSM_TRACE)
static const bool g_host_prof = getenv("SPHSM_HOST_PROF") != nullptr;
static double now_us() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}
static int mg_step_nccl(sphsm_handle *h) {
    int rc, coll, count;
    if ((rc = mg_check(h)) != 0) return rc;
    static double acc[MG_PHASES + 1][2];
    static int steps_seen = 0;
    for (int ph = 0; ph < MG_PHASES; ph++) {
        const double t0 = g_host_prof ? now_us() : 0.0;
        if ((rc = mg_phase(h, ph, &coll, &count)) != 0) return rc;
        const double t1 = g_host_prof ? now_us() : 0.0;
        if (coll == COLL_EXCH1) {
            rc = h->p2p_on ? p2p_signal(h) : nccl_exchange1(h, h->stream);
            if (!rc && h->moments_forked && h->allreduce_pending) rc = mg_forked_allreduce(h);
            h->allreduce_pending = false;
        }
        else if (coll == COLL_EXCH1_TAKEN) {  // the exchange happened at the end of the previous step: only the allreduce is left
            if (h->moments_forked && h->allreduce_pending) rc = mg_forked_allreduce(h);
            h->allreduce_pending = false;
            if (!rc) rc = mg_check_interior(h);
        } else if (coll == COLL_EXCH1_EARLY) {  // next step's exchange 1, on the side stream behind the outer planes' pass B
            if (h->p2p_on) {
                h->launch_stream = h->side_stream;
                rc = p2p_signal(h);
                h->launch_stream = h->stream;
            } else rc = nccl_exchange1(h, h->side_stream);
            if (!rc) CU(cudaEventRecord(h->ev_x1, h->side_stream));
            h->x1_early_pending = true;
            h->x1_early_valid = true;
        }
        else if (coll == COLL_ALLREDUCE) rc = comm_allreduce(h, count);
        else if (coll == COLL_ALLREDUCE_MOMENTS) rc = moment_allreduce(h);
        else if (coll == COLL_EXCH2) rc = nccl_exchange2(h, h->stream);
        if (rc) return rc;
        if (g_host_prof) {
            acc[ph][0] += t1 - t0;
            acc[ph][1] += now_us() - t1;
        }
    }
    if (h->peer_error) {  // some rank (maybe this one) failed in the previous step: every rank stops here
        h->failed = true;
        return fail(h, SPHSM_ERR_COMM, h->local_error ? h->local_error_msg.c_str()
                                                      : "another rank of the slab group reported a step error (its sphsm_last_error has the cause)");
    }
    if (g_host_prof) steps_seen++;
    if (g_host_prof && steps_seen % 64 == 0 && h->rank == 0) {
        fprintf(stderr, "[sphsm host prof, us/step over %d steps] ", steps_seen);
        double tot = 0;
        for (int ph = 0; ph < MG_PHASES; ph++) {
            fprintf(stderr, "ph%d %.1f+%.1f  ", ph, acc[ph][0] / steps_seen, acc[ph][1] / steps_seen);
            tot += acc[ph][0] + acc[ph][1];
        }
        fprintf(stderr, "total %.1f (read-back wait %.1f)\n", tot / steps_seen, h->meta_wait_us / steps_seen);
    }
    return SPHSM_OK;
}

// virtual ranks: the same phases in lockstep over handles that share one device; collectives are device copies
extern "C" int sphsm_step_group(sphsm_handle **hs, int nranks, int nsteps) {
    if (!hs || nranks < 1 || nsteps < 0) return SPHSM_ERR_INVALID;
    for (int r = 0; r < nranks; r++) {
        sphsm_handle *h = hs[r];
        if (!h || h->comm_mode != 2 || h->nranks != nranks || h->rank != r) return fail(h, SPHSM_ERR_COMM, "not the local group made by sphsm_comm_init_local");
        int rc = mg_check(h);
        if (!rc) rc = observe_sync(h);
        if (rc) return rc;
    }
    sphsm_handle *h = hs[0];
    CU(cudaSetDevice(h->prm.device));
    std::vector<int> coll(nranks), count(nranks);
    std::vector<double> sum(128), part(128);
    for (int s = 0; s < nsteps; s++) {
        for (int ph = 0; ph < MG_PHASES; ph++) {
            for (int r = 0; r < nranks; r++) {
                int rc = mg_phase(hs[r], ph, &coll[r], &count[r]);
                if (rc) return rc;
                if (coll[r] != coll[0] || count[r] != count[0]) return fail(hs[r], SPHSM_ERR_COMM, "ranks disagree on the phase program");
            }
            for (int r = 0; r < nranks; r++) CU(cudaStreamSynchronize(hs[r]->stream));
            if (coll[0] == COLL_EXCH1) {  // (message sizes as the NCCL step derives them: the two sides of a face must agree)
                for (int r = 0; r < nranks; r++) {
                    if (r > 0) {
                        if (hs[r]->x1_recv_cap[0] != hs[r - 1]->x1_send_cap[1]) return fail(hs[r], SPHSM_ERR_COMM, "internal: the two sides of a slab face sized exchange 1 differently");
                        CU(cudaMemcpy(hs[r]->msg_recv[0], hs[r - 1]->msg_send[1], msg_bytes(hs[r]->x1_recv_cap[0]), cudaMemcpyDeviceToDevice));
                    }
                    if (r < nranks - 1) {
                        if (hs[r]->x1_recv_cap[1] != hs[r + 1]->x1_send_cap[0]) return fail(hs[r], SPHSM_ERR_COMM, "internal: the two sides of a slab face sized exchange 1 differently");
                        CU(cudaMemcpy(hs[r]->msg_recv[1], hs[r + 1]->msg_send[0], msg_bytes(hs[r]->x1_recv_cap[1]), cudaMemcpyDeviceToDevice));
                    }
                }
            } else if (coll[0] == COLL_ALLREDUCE || coll[0] == COLL_ALLREDUCE_MOMENTS) {
                const int c = count[0];
                std::fill(sum.begin(), sum.end(), 0.0);
                for (int r = 0; r < nranks; r++) {
                    CU(cudaMemcpy(part.data(), hs[r]->totals, c * sizeof(double), cudaMemcpyDeviceToHost));
                    for (int k = 0; k < c; k++) sum[k] += part[k];
                }
                for (int r = 0; r < nranks; r++) CU(cudaMemcpy(hs[r]->totals, sum.data(), c * sizeof(double), cudaMemcpyHostToDevice));
            } else if (coll[0] == COLL_EXCH2) {
                const size_t bytes = msg2_bytes(h->send_cap);
                for (int r = 0; r < nranks; r++) {
                    if (r > 0) CU(cudaMemcpy(hs[r]->msg_recv[0], hs[r - 1]->msg_send[1], bytes, cudaMemcpyDeviceToDevice));
                    if (r < nranks - 1) CU(cudaMemcpy(hs[r]->msg_recv[1], hs[r + 1]->msg_send[0], bytes, cudaMemcpyDeviceToDevice));
                }
            }
        }
    }
    for (int r = 0; r < nranks; r++) {  // the last step's boundaries and error counters, now
        int rc = slab_refresh(hs[r]);
        if (!rc) rc = slab_check_local_error(hs[r]);
        if (rc) return rc;
    }
    return SPHSM_OK;
}
