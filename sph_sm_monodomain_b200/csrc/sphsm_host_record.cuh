// sphsm_host_record.cuh — host side of the Vm recorder (sphsm_record.cuh): the sphsm_record_* / sphsm_get_* entry points, and
// the per-step hook and device step counter it shares with the electrograms (sphsm_host_egm.cuh).  Host code of libsphsm_b200.so,
// textually included by sphsm_capi.cu (one translation unit: the handle, the LAUNCH / CU macros and the static helpers defined
// there are in scope).
//
// While recording is off nothing is allocated and the step launches nothing extra.  While it is on, every step path (fused,
// graph replay, strict, staged with stage timing, sphsm_profile_step, the NCCL slab step, sphsm_step_group) ends with one k_record
// launch; sphsm_stage(1..9) records nothing.  The recorder's pointers and thresholds are part of the CUDA-graph signature
// (step_signature), so starting or stopping recording picks or captures a different graph.
#pragma once

// ---- the step counter and the per-step hook shared by the recorder and the electrograms -------------------------------------
static bool observe_on(const sphsm_handle *h) { return h->rec.on || h->egm.on; }

// the device step counter follows total_time_steps: set it again when the host counter moved outside an observed step
// (sphsm_load_state, a step with no particles).  Called at the entry of every stepping call, never inside a graph capture.
static int observe_sync(sphsm_handle *h) {
    if (!observe_on(h) || h->dev_steps == h->total_steps) return SPHSM_OK;
    const unsigned v[2] = {(unsigned)h->total_steps, 0u};
    CU(cudaMemcpyAsync(h->step_ctl, v, sizeof v, cudaMemcpyHostToDevice, h->stream));
    h->dev_steps = h->total_steps;
    return SPHSM_OK;
}

// a start: the counter exists while either observer is on (called once the starting one is on)
static int step_ctl_attach(sphsm_handle *h) {
    if (!h->step_ctl) CU(cudaMalloc(&h->step_ctl, 2 * sizeof(unsigned)));
    h->dev_steps = h->total_steps - 1;  // (forces the counter upload)
    return observe_sync(h);
}

// a stop: the last observer to go frees the counter (called once the stopping one is off)
static void step_ctl_detach(sphsm_handle *h) {
    if (observe_on(h) || !h->step_ctl) return;
    cudaStreamSynchronize(h->stream);  // (a queued step may still write it)
    cudaFree(h->step_ctl);
    h->step_ctl = nullptr;
    h->dev_steps = 0;
}

static int record_launch(sphsm_handle *h, const int *rng, int count, bool advance);
static int egm_launch(sphsm_handle *h, const int *rng, int count);  // sphsm_host_egm.cuh

// the per-step hook: right after the kernel that integrated the step, over the slots it integrated
// (rng == nullptr: h->dp's own range, count = its length; slab step: the device range rng_all, count = own_bound).
// One launch per observer that is on; the last one advances the step counter, so both number the step alike.
static int observe_launch(sphsm_handle *h, const int *rng, int count) {
    if (!observe_on(h)) return SPHSM_OK;
    int rc;
    count = std::max(count, 0);
    if (h->rec.on && (rc = record_launch(h, rng, count, !h->egm.on)) != 0) return rc;
    if (h->egm.on && (rc = egm_launch(h, rng, count)) != 0) return rc;
    h->dev_steps++;
    return SPHSM_OK;
}

// ---- the recorder ---------------------------------------------------------------------------------------------------------
static void record_free(sphsm_handle *h) {
    auto &r = h->rec;
    if (r.maps) cudaStreamSynchronize(h->stream);  // (a queued step may still write them)
    cudaFree(r.maps); cudaFree(r.probe_of); cudaFree(r.trace); cudaFree(r.stamp);
    r = sphsm_handle::Recorder{};
    step_ctl_detach(h);
}

// data cleared, configuration kept: steps unset (-1), n_up 0, no trace row owned
static void record_clear(sphsm_handle *h) {
    auto &r = h->rec;
    if (!r.on) return;
    cudaMemsetAsync(r.maps, 0xff, (size_t)3 * r.cap * sizeof(int), h->stream);
    cudaMemsetAsync(r.maps + (size_t)3 * r.cap, 0, (size_t)r.cap * sizeof(int), h->stream);
    if (r.stamp) cudaMemsetAsync(r.stamp, 0, (size_t)r.rows * r.n_probes * sizeof(int), h->stream);
    r.recorded = 0;
}

// advance: this launch is the hook's last and advances the step counter
static int record_launch(sphsm_handle *h, const int *rng, int count, bool advance) {
    auto &r = h->rec;
    RecArgs a;
    a.first_up = r.maps;
    a.last_up = r.maps + (size_t)r.cap;
    a.last_down = r.maps + (size_t)2 * r.cap;
    a.n_up = r.maps + (size_t)3 * r.cap;
    a.probe_of = r.probe_of;
    a.trace = r.trace;
    a.stamp = r.stamp;
    a.n_probes = r.n_probes;
    a.rows = std::max(r.rows, 1);
    a.vm_up = r.vm_up;
    a.vm_down = r.vm_down;
    a.ctl = h->step_ctl;
    a.advance = advance ? 1 : 0;
    LAUNCH(k_record, std::max(1, cdiv(count, REC_THREADS)), REC_THREADS, h->dp, rng, count, (const int *)h->cur.ID, (const float4 *)h->cur.PB,
           (const float4 *)h->cur.E, (const float4 *)h->cur.P, a);
    r.recorded++;
    return SPHSM_OK;
}

static int record_count(const sphsm_handle *h) { return h->dp.slab_on ? h->n_global : h->n; }

extern "C" int sphsm_record_start(sphsm_handle *h, float vm_up, float vm_down, const int *probe_ids, int n_probes, int trace_rows) {
    if (!h) return SPHSM_ERR_INVALID;
    if (!isfinite(vm_up) || !isfinite(vm_down) || vm_down > vm_up)
        return fail(h, SPHSM_ERR_INVALID, "record thresholds must be finite with vm_down <= vm_up");
    if (n_probes < 0 || n_probes > SPHSM_RECORD_MAX_PROBES || (n_probes > 0 && !probe_ids))
        return fail(h, SPHSM_ERR_INVALID, "n_probes must be in [0, SPHSM_RECORD_MAX_PROBES] with a probe id array");
    if (n_probes > 0 && (trace_rows <= 0 || (long long)trace_rows * n_probes > SPHSM_RECORD_MAX_TRACE_ENTRIES))
        return fail(h, SPHSM_ERR_INVALID, "trace_rows must be positive with trace_rows * n_probes <= SPHSM_RECORD_MAX_TRACE_ENTRIES");
    const int count = record_count(h);
    {
        std::unordered_set<int> seen;
        for (int k = 0; k < n_probes; k++) {
            if (probe_ids[k] < 0 || probe_ids[k] >= count) return fail(h, SPHSM_ERR_INVALID, "probe id outside the particle count");
            if (!seen.insert(probe_ids[k]).second) return fail(h, SPHSM_ERR_INVALID, "duplicate probe id");
        }
    }
    CU(cudaSetDevice(h->prm.device));
    record_free(h);  // (a running recording is replaced)
    auto &r = h->rec;
    r.cap = h->prm.capacity;
    r.vm_up = vm_up;
    r.vm_down = vm_down;
    r.n_probes = n_probes;
    r.rows = n_probes > 0 ? trace_rows : 0;
    int rc = [&]() -> int {
        CU(cudaMalloc(&r.maps, (size_t)4 * r.cap * sizeof(int)));
        if (n_probes > 0) {
            CU(cudaMalloc(&r.probe_of, (size_t)r.cap * sizeof(int)));
            CU(cudaMalloc(&r.trace, (size_t)r.rows * n_probes * sizeof(float4)));
            CU(cudaMalloc(&r.stamp, (size_t)r.rows * n_probes * sizeof(int)));
            CU(cudaMemsetAsync(r.probe_of, 0xff, (size_t)r.cap * sizeof(int), h->stream));
            CU(cudaMemsetAsync(r.trace, 0, (size_t)r.rows * n_probes * sizeof(float4), h->stream));
            int rc2;
            if ((rc2 = ensure_itmp(h, (size_t)n_probes)) != 0) return rc2;
            CU(cudaMemcpyAsync(h->d_itmp, probe_ids, (size_t)n_probes * sizeof(int), cudaMemcpyHostToDevice, h->stream));
            LAUNCH(k_record_probes, cdiv(n_probes, 256), 256, (const int *)h->d_itmp, n_probes, r.probe_of);
        }
        r.on = true;
        record_clear(h);
        int rc3 = step_ctl_attach(h);
        if (rc3) return rc3;
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(h->stream));
        return SPHSM_OK;
    }();
    if (rc) {
        const std::string why = h->err;
        record_free(h);
        h->err = why;
    }
    return rc;
}

extern "C" int sphsm_record_stop(sphsm_handle *h) {
    if (!h) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    record_free(h);
    return SPHSM_OK;
}

extern "C" int sphsm_record_reset(sphsm_handle *h) {
    if (!h) return SPHSM_ERR_INVALID;
    if (!h->rec.on) return fail(h, SPHSM_ERR_INVALID, "recording is off");
    CU(cudaSetDevice(h->prm.device));
    record_clear(h);
    CU(cudaGetLastError());
    return SPHSM_OK;
}

extern "C" int sphsm_get_activation(sphsm_handle *h, int *first_up, int *last_up, int *last_down, int *n_up, int n) {
    if (!h) return SPHSM_ERR_INVALID;
    const auto &r = h->rec;
    if (!r.on) return fail(h, SPHSM_ERR_INVALID, "recording is off");
    if (n < 0 || n > r.cap) return fail(h, SPHSM_ERR_INVALID, "n must be in [0, capacity]");
    CU(cudaSetDevice(h->prm.device));
    int *outs[4] = {first_up, last_up, last_down, n_up};  // (a null pointer skips that map)
    for (int m = 0; m < 4; m++)
        if (outs[m] && n > 0) CU(cudaMemcpyAsync(outs[m], r.maps + (size_t)m * r.cap, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return SPHSM_OK;
}

extern "C" int sphsm_get_probe_trace(sphsm_handle *h, int max_rows, int *rows, int *first_step, float *xyzv, uint8_t *owned) {
    if (!h || !rows || !first_step || max_rows < 0) return SPHSM_ERR_INVALID;
    const auto &r = h->rec;
    if (!r.on) return fail(h, SPHSM_ERR_INVALID, "recording is off");
    const int K = r.n_probes;
    const int held = K > 0 ? (int)std::min<long long>(std::min<long long>(r.rows, r.recorded), max_rows) : 0;
    if (held > 0 && (!xyzv || !owned)) return fail(h, SPHSM_ERR_INVALID, "null output array");
    const int last = h->dev_steps, first = last - held + 1;  // the last `held` steps, oldest first
    *rows = held;
    *first_step = held > 0 ? first : last + 1;
    if (held == 0) return SPHSM_OK;
    CU(cudaSetDevice(h->prm.device));
    std::vector<float4> tr((size_t)r.rows * K);
    std::vector<int> st((size_t)r.rows * K);
    CU(cudaMemcpyAsync(tr.data(), r.trace, tr.size() * sizeof(float4), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(st.data(), r.stamp, st.size() * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int j = 0; j < held; j++) {
        const int s = first + j;
        const size_t src = (size_t)(s % r.rows) * K, dst = (size_t)j * K;
        for (int k = 0; k < K; k++) {
            const bool mine = st[src + k] == s;
            const float4 v = mine ? tr[src + k] : make_float4(0.f, 0.f, 0.f, 0.f);
            xyzv[4 * (dst + k)] = v.x; xyzv[4 * (dst + k) + 1] = v.y; xyzv[4 * (dst + k) + 2] = v.z; xyzv[4 * (dst + k) + 3] = v.w;
            owned[dst + k] = mine ? 1 : 0;
        }
    }
    return SPHSM_OK;
}
