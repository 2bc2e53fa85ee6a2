// sphsm_host_egm.cuh — host side of the electrograms at virtual electrodes (sphsm_egm.cuh): the k_egm launch of the per-step hook
// (observe_launch, sphsm_host_record.cuh) and the sphsm_egm_* / sphsm_get_egm entry points.  Host code of libsphsm_b200.so,
// textually included by sphsm_capi.cu after sphsm_host_record.cuh.
//
// While electrograms are off nothing is allocated and the step launches nothing extra.  While they are on, pass B takes its EGM
// variant (it also stores Q = vol * L) and every step path ends with one k_egm launch, after k_record when the recorder is on too;
// sphsm_stage(1..9) produces no row.  The pointers and the configuration are part of the CUDA-graph signature (step_signature).
// Lifetime follows the recorder: start (re)configures and clears, stop frees, reset and sphsm_load_state clear the rows.
#pragma once

static_assert(SPHSM_EGM_MAX_ELECTRODES == EGM_MAX_ELECTRODES, "k_egm stages every electrode in shared memory");

static void egm_free(sphsm_handle *h) {
    auto &g = h->egm;
    if (g.Q) cudaStreamSynchronize(h->stream);  // (a queued step may still write them)
    cudaFree(g.Q); cudaFree(g.el); cudaFree(g.partial); cudaFree(g.ring);
    g = sphsm_handle::Electrograms{};
    h->cur.Q = h->alt.Q = nullptr;
    step_ctl_detach(h);
}

// the rows are cleared; the configuration is kept (every recorded step writes a whole row: nothing on the device to clear)
static void egm_clear(sphsm_handle *h) { h->egm.recorded = 0; }

static int egm_launch(sphsm_handle *h, const int *rng, int count) {
    const auto &g = h->egm;
    EgmArgs a;
    a.el = g.el;
    a.n_el = g.n_el;
    a.rows = g.rows;
    a.gain = g.gain;
    a.eps2 = g.eps2;
    a.partial = g.partial;
    a.ring = g.ring;
    a.ctl = h->step_ctl;
    LAUNCH(k_egm, g.grid, EGM_THREADS, h->dp, rng, count, (const float4 *)h->cur.PB, (const float *)g.Q, a);
    h->egm.recorded++;
    return SPHSM_OK;
}

extern "C" int sphsm_egm_start(sphsm_handle *h, const float *xyz, int n_electrodes, float gain, float softening, int rows) {
    if (!h) return SPHSM_ERR_INVALID;
    if (n_electrodes < 1 || n_electrodes > SPHSM_EGM_MAX_ELECTRODES || !xyz)
        return fail(h, SPHSM_ERR_INVALID, "n_electrodes must be in [1, SPHSM_EGM_MAX_ELECTRODES] with a coordinate array");
    for (int k = 0; k < 3 * n_electrodes; k++)
        if (!isfinite(xyz[k])) return fail(h, SPHSM_ERR_INVALID, "electrode coordinates must be finite");
    if (!isfinite(gain)) return fail(h, SPHSM_ERR_INVALID, "gain must be finite");
    if (!isfinite(softening) || softening <= 0.f) return fail(h, SPHSM_ERR_INVALID, "softening must be positive and finite");
    if (rows <= 0 || (long long)rows * n_electrodes > SPHSM_RECORD_MAX_TRACE_ENTRIES)
        return fail(h, SPHSM_ERR_INVALID, "rows must be positive with rows * n_electrodes <= SPHSM_RECORD_MAX_TRACE_ENTRIES");
    CU(cudaSetDevice(h->prm.device));
    egm_free(h);  // (running electrograms are replaced)
    auto &g = h->egm;
    int sms = 0;
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->prm.device));
    g.n_el = n_electrodes;
    g.rows = rows;
    g.gain = gain;
    g.eps2 = softening * softening;
    // persistent grid: enough blocks for every SM while the slots last (the particle capacity bounds every launch's count)
    g.grid = std::max(1, std::min(EGM_BLOCKS_PER_SM * sms, cdiv(h->alloc_n, EGM_THREADS * EGM_SLOTS)));
    int rc = [&]() -> int {
        std::vector<float4> el(n_electrodes);
        for (int k = 0; k < n_electrodes; k++) el[k] = make_float4(xyz[3 * k], xyz[3 * k + 1], xyz[3 * k + 2], 0.f);
        CU(cudaMalloc(&g.Q, ((size_t)h->alloc_n + 8) * sizeof(float)));
        CU(cudaMalloc(&g.el, (size_t)n_electrodes * sizeof(float4)));
        CU(cudaMalloc(&g.partial, (size_t)g.grid * n_electrodes * sizeof(double)));
        CU(cudaMalloc(&g.ring, (size_t)rows * n_electrodes * sizeof(double)));
        CU(cudaMemsetAsync(g.Q, 0, ((size_t)h->alloc_n + 8) * sizeof(float), h->stream));
        CU(cudaMemsetAsync(g.ring, 0, (size_t)rows * n_electrodes * sizeof(double), h->stream));
        CU(cudaMemcpyAsync(g.el, el.data(), el.size() * sizeof(float4), cudaMemcpyHostToDevice, h->stream));
        h->cur.Q = h->alt.Q = g.Q;
        g.on = true;
        egm_clear(h);
        int rc2 = step_ctl_attach(h);
        if (rc2) return rc2;
        CU(cudaGetLastError());
        CU(cudaStreamSynchronize(h->stream));
        return SPHSM_OK;
    }();
    if (rc) {
        const std::string why = h->err;
        egm_free(h);
        h->err = why;
    }
    return rc;
}

extern "C" int sphsm_egm_stop(sphsm_handle *h) {
    if (!h) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    egm_free(h);
    return SPHSM_OK;
}

extern "C" int sphsm_egm_reset(sphsm_handle *h) {
    if (!h) return SPHSM_ERR_INVALID;
    if (!h->egm.on) return fail(h, SPHSM_ERR_INVALID, "electrograms are off");
    egm_clear(h);
    return SPHSM_OK;
}

extern "C" int sphsm_get_egm(sphsm_handle *h, int max_rows, int *rows, int *first_step, double *phi) {
    if (!h || !rows || !first_step || max_rows < 0) return SPHSM_ERR_INVALID;
    const auto &g = h->egm;
    if (!g.on) return fail(h, SPHSM_ERR_INVALID, "electrograms are off");
    const int E = g.n_el;
    const int held = (int)std::min<long long>(std::min<long long>(g.rows, g.recorded), max_rows);
    if (held > 0 && !phi) return fail(h, SPHSM_ERR_INVALID, "null output array");
    const int last = h->dev_steps, first = last - held + 1;  // the last `held` steps, oldest first
    *rows = held;
    *first_step = held > 0 ? first : last + 1;
    if (held == 0) return SPHSM_OK;
    CU(cudaSetDevice(h->prm.device));
    std::vector<double> ring((size_t)g.rows * E);
    CU(cudaMemcpyAsync(ring.data(), g.ring, ring.size() * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    for (int j = 0; j < held; j++) {
        const int s = first + j;
        memcpy(phi + (size_t)j * E, ring.data() + (size_t)(s % g.rows) * E, (size_t)E * sizeof(double));
    }
    return SPHSM_OK;
}
