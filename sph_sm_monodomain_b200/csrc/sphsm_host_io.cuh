// sphsm_host_io.cuh — state snapshot / restart and the asynchronous per-frame I/O entry points
// Host code of libsphsm_b200.so, textually included by sphsm_capi.cu (one translation unit: the handle, the LAUNCH / CU macros and
// the static helpers defined there are in scope).
#pragma once

// ---------------------------------------------------------------------------------------------------
// State snapshot / restart (SURVEY.md §8 f.4; the reference has none).  File = header + sphsm_params + the particles in
// the reference's own Particle layout (132 B, all 33 fields, original order), i.e. exactly what Get_Paticles() shows.
struct SnapshotHeader {
    char magic[8];  // "SPHSMB2\0"
    uint32_t version, header_bytes, params_bytes, stride;
    int32_t n, total_steps;
};
extern "C" int sphsm_save_state(sphsm_handle *h, const char *path) {
    if (!h || !path) return SPHSM_ERR_INVALID;
    if (h->dp.slab_on) return fail(h, SPHSM_ERR_INVALID, "snapshots are written from a single-GPU handle");
    std::vector<uint8_t> buf((size_t)std::max(h->n, 1) * SPHSM_PARTICLE_STRIDE);
    int rc = h->n > 0 ? sphsm_download_aos(h, buf.data(), h->n, SPHSM_PARTICLE_STRIDE) : SPHSM_OK;
    if (rc) return rc;
    SnapshotHeader hd;
    memset(&hd, 0, sizeof(hd));
    memcpy(hd.magic, "SPHSMB2", 8);
    hd.version = 1; hd.header_bytes = sizeof(hd); hd.params_bytes = sizeof(sphsm_params); hd.stride = SPHSM_PARTICLE_STRIDE;
    hd.n = h->n; hd.total_steps = h->total_steps;
    FILE *f = fopen(path, "wb");
    if (!f) return fail(h, SPHSM_ERR_INVALID, "cannot open the snapshot file for writing");
    bool ok = fwrite(&hd, sizeof(hd), 1, f) == 1 && fwrite(&h->prm, sizeof(sphsm_params), 1, f) == 1 &&
              (h->n == 0 || fwrite(buf.data(), (size_t)h->n * SPHSM_PARTICLE_STRIDE, 1, f) == 1);
    ok = (fclose(f) == 0) && ok;
    return ok ? SPHSM_OK : fail(h, SPHSM_ERR_INVALID, "short write on the snapshot file");
}
// Restores particles, tunable parameters and the step counter into an existing handle (its capacity, device and world
// stay its own: the snapshot must fit, and its world must match).
extern "C" int sphsm_load_state(sphsm_handle *h, const char *path) {
    if (!h || !path) return SPHSM_ERR_INVALID;
    if (h->dp.slab_on) return fail(h, SPHSM_ERR_INVALID, "load the snapshot before sphsm_comm_set_slab");
    FILE *f = fopen(path, "rb");
    if (!f) return fail(h, SPHSM_ERR_INVALID, "cannot open the snapshot file");
    SnapshotHeader hd;
    sphsm_params sp;
    int rc = SPHSM_OK;
    std::vector<uint8_t> buf;
    if (fread(&hd, sizeof(hd), 1, f) != 1 || memcmp(hd.magic, "SPHSMB2", 8) != 0 || hd.version != 1 || hd.header_bytes != sizeof(hd) ||
        hd.params_bytes != sizeof(sphsm_params) || hd.stride != SPHSM_PARTICLE_STRIDE || hd.n < 0)
        rc = fail(h, SPHSM_ERR_INVALID, "not a snapshot of this library version");
    else if (fread(&sp, sizeof(sp), 1, f) != 1)
        rc = fail(h, SPHSM_ERR_INVALID, "truncated snapshot");
    else if (hd.n > h->prm.capacity)
        rc = fail(h, SPHSM_ERR_CAPACITY, "snapshot holds more particles than this handle's capacity");
    else if (sp.world[0] != h->prm.world[0] || sp.world[1] != h->prm.world[1] || sp.world[2] != h->prm.world[2] || sp.kernel_h != h->prm.kernel_h)
        rc = fail(h, SPHSM_ERR_INVALID, "snapshot was taken in a different world / kernel size");
    else {
        buf.resize((size_t)std::max(hd.n, 1) * SPHSM_PARTICLE_STRIDE);
        if (hd.n > 0 && fread(buf.data(), (size_t)hd.n * SPHSM_PARTICLE_STRIDE, 1, f) != 1) rc = fail(h, SPHSM_ERR_INVALID, "truncated snapshot");
    }
    fclose(f);
    if (rc) return rc;
    sp.device = h->prm.device; sp.capacity = h->prm.capacity; sp.slab_axis = h->prm.slab_axis; sp.strict = h->prm.strict;
    sp.diagnostics = h->prm.diagnostics;
    memcpy(sp.reserved, h->prm.reserved, sizeof sp.reserved);  // the handle's own switches (sort algorithm, graphs ...) are not state
    const sphsm_params before = h->prm;
    if ((rc = sphsm_set_params(h, &sp)) != 0) return rc;
    if ((rc = sphsm_upload_aos(h, buf.data(), hd.n, SPHSM_PARTICLE_STRIDE)) != 0) {
        const std::string why = h->err;
        sphsm_set_params(h, &before);  // a failed load leaves the handle as it was
        h->err = why;
        return rc;
    }
    h->total_steps = hd.total_steps;
    record_clear(h);  // recorded data belongs to the replaced particle set; numbering continues at the snapshot's step + 1
    egm_clear(h);
    return SPHSM_OK;
}

// ---------------------------------------------------------------------------------------------------
// Asynchronous I/O.  The host arrays must be page-locked for the copies to overlap and must stay untouched until
// sphsm_io_wait (or sphsm_sync) returns.  Input copies run on their own stream into their own staging and the kernel that
// applies them waits for the copy; output is gathered on the compute stream and copied out on a second copy stream, so a
// caller that loops { set_masks_async; step; download_*_async } has step k+1 computing while the results of step k cross
// PCIe one way and the inputs of step k+2 cross it the other way.
static int ensure_io_in(sphsm_handle *h, size_t n) {
    if (h->io_in_cap >= n) return SPHSM_OK;
    CU(cudaStreamSynchronize(h->h2d_stream));
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(h->io_in_f); cudaFree(h->io_in_b);
    h->io_in_f = nullptr; h->io_in_b = nullptr; h->io_in_cap = 0;
    CU(cudaMalloc(&h->io_in_f, n * sizeof(float)));
    CU(cudaMalloc(&h->io_in_b, n));
    h->io_in_cap = n;
    return SPHSM_OK;
}
static int ensure_io_out(sphsm_handle *h, size_t n) {
    if (h->io_out_cap >= n) return SPHSM_OK;
    CU(cudaStreamSynchronize(h->d2h_stream));
    CU(cudaStreamSynchronize(h->stream));
    cudaFree(h->io_out_f); cudaFree(h->io_out_i);
    h->io_out_f = nullptr; h->io_out_i = nullptr; h->io_out_cap = 0;
    CU(cudaMalloc(&h->io_out_f, n * 3 * sizeof(float)));
    CU(cudaMalloc(&h->io_out_i, n * sizeof(int)));
    h->io_out_cap = n;
    return SPHSM_OK;
}

extern "C" int sphsm_set_masks_async(sphsm_handle *h, const uint8_t *fixed, const float *stim, int n) {
    if (!h || n != (h->dp.slab_on ? h->n_global : h->n)) return fail(h, SPHSM_ERR_INVALID, "set_masks needs exactly num_particles entries");
    if (n == 0 || (!fixed && !stim)) return SPHSM_OK;
    CU(cudaSetDevice(h->prm.device));
    int rc;
    h->x1_early_valid = false;
    if ((rc = ensure_io_in(h, (size_t)n)) != 0) return rc;
    CU(cudaStreamWaitEvent(h->h2d_stream, h->ev_in_free, 0));  // the previous call's kernel has consumed the staging
    if (stim) CU(cudaMemcpyAsync(h->io_in_f, stim, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, h->h2d_stream));
    if (fixed) CU(cudaMemcpyAsync(h->io_in_b, fixed, (size_t)n, cudaMemcpyHostToDevice, h->h2d_stream));
    CU(cudaEventRecord(h->ev_in_ready, h->h2d_stream));
    CU(cudaStreamWaitEvent(h->stream, h->ev_in_ready, 0));
    // slab mode: h->n may lag the device by a step or two; the grid covers the bound and every live slot has a valid id (dead ones: -1)
    const int n_k = h->dp.slab_on ? std::max(h->n_bound, h->n) : h->n;
    if (n_k > 0)
        LAUNCH(k_set_masks, cdiv(n_k, 256), 256, h->dp, n_k, h->cur, fixed ? (const uint8_t *)h->io_in_b : nullptr, stim ? h->io_in_f : nullptr,
               freeze_source(h), h->dp.slab_on ? (const int *)&h->d_meta[h->meta_cur]->n_live : (const int *)nullptr);
    CU(cudaGetLastError());
    CU(cudaEventRecord(h->ev_in_free, h->stream));
    if (fixed) h->rest_dirty = true;
    return SPHSM_OK;
}

static int io_copy_out(sphsm_handle *h, int *ids, float *xyz, size_t count) {
    CU(cudaEventRecord(h->ev_out_ready, h->stream));
    CU(cudaStreamWaitEvent(h->d2h_stream, h->ev_out_ready, 0));
    if (ids) CU(cudaMemcpyAsync(ids, h->io_out_i, count * sizeof(int), cudaMemcpyDeviceToHost, h->d2h_stream));
    CU(cudaMemcpyAsync(xyz, h->io_out_f, count * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->d2h_stream));
    CU(cudaEventRecord(h->ev_out_done, h->d2h_stream));
    return SPHSM_OK;
}

extern "C" int sphsm_download_positions_async(sphsm_handle *h, float *xyz, int n) {
    if (!h || !xyz || n < 0) return SPHSM_ERR_INVALID;
    if (h->dp.slab_on) return fail(h, SPHSM_ERR_INVALID, "slab mode: use sphsm_download_owned_async");
    if (n > h->n) return SPHSM_ERR_INVALID;
    if (n == 0) return SPHSM_OK;
    CU(cudaSetDevice(h->prm.device));
    int rc;
    if ((rc = ensure_io_out(h, (size_t)h->n)) != 0) return rc;
    CU(cudaStreamWaitEvent(h->stream, h->ev_out_done, 0));  // the previous copy has left the staging
    LAUNCH(k_positions_out, cdiv(h->n, 256), 256, 0, h->n, h->cur, h->io_out_f);
    CU(cudaGetLastError());
    return io_copy_out(h, nullptr, xyz, (size_t)n);
}

extern "C" int sphsm_download_owned_async(sphsm_handle *h, int *ids, float *xyz, int cap, int *count) {
    if (!h || !ids || !xyz || !count || cap < 0) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    int rc;
    if (!h->dp.slab_on) {  // one GPU: every particle is owned, the count is known
        const int nown = h->n;
        *count = nown;
        if (nown > cap) return fail(h, SPHSM_ERR_CAPACITY, "output arrays smaller than the number of owned particles");
        if (nown == 0) return SPHSM_OK;
        if ((rc = ensure_io_out(h, (size_t)nown)) != 0) return rc;
        CU(cudaStreamWaitEvent(h->stream, h->ev_out_done, 0));
        LAUNCH(k_mg_owned_out, cdiv(nown, 256), 256, (const int *)nullptr, 0, nown, nown, h->cur, h->io_out_i, h->io_out_f, (int *)nullptr);
        CU(cudaGetLastError());
        return io_copy_out(h, ids, xyz, (size_t)nown);
    }
    // Slab mode: the owned range lives in device memory (the host does not wait for a step to learn it), so the gather covers
    // the owned-count bound, min(cap, bound) records cross PCIe and the count follows them into *count — valid, like the
    // arrays, once sphsm_io_wait / sphsm_sync has returned.  More owned particles than `cap`: the surplus is not delivered
    // and *count says so.
    const int take = std::min(cap, h->own_bound);
    if (take <= 0) { *count = 0; return SPHSM_OK; }
    if ((rc = ensure_io_out(h, (size_t)std::max(take, h->prm.capacity / std::max(h->nranks, 1) + 65536))) != 0) return rc;
    if ((size_t)take > h->io_out_cap && (rc = ensure_io_out(h, (size_t)take)) != 0) return rc;
    CU(cudaStreamWaitEvent(h->stream, h->ev_out_done, 0));
    LAUNCH(k_mg_owned_out, cdiv(take, 256), 256, h->d_meta[h->meta_cur]->rng_all, 0, 0, take, h->cur, h->io_out_i, h->io_out_f, h->d_count);
    CU(cudaGetLastError());
    CU(cudaEventRecord(h->ev_out_ready, h->stream));
    CU(cudaStreamWaitEvent(h->d2h_stream, h->ev_out_ready, 0));
    CU(cudaMemcpyAsync(count, h->d_count, sizeof(int), cudaMemcpyDeviceToHost, h->d2h_stream));
    CU(cudaMemcpyAsync(ids, h->io_out_i, (size_t)take * sizeof(int), cudaMemcpyDeviceToHost, h->d2h_stream));
    CU(cudaMemcpyAsync(xyz, h->io_out_f, (size_t)take * 3 * sizeof(float), cudaMemcpyDeviceToHost, h->d2h_stream));
    CU(cudaEventRecord(h->ev_out_done, h->d2h_stream));
    return SPHSM_OK;
}

// Per-step stimulation input for the particles a rank owns: stim[k] belongs to the k-th particle of the most recent
// sphsm_download_owned_async on this handle (the device still holds that id list).  4 bytes per OWNED particle cross PCIe,
// so the input traffic of a multi-GPU run does not grow with the number of ranks (sphsm_set_masks_async needs the global array
// on every rank).  A particle that has migrated to a neighbour since that download keeps its previous value for one step.
extern "C" int sphsm_set_stim_owned_async(sphsm_handle *h, const float *stim, int count) {
    if (!h || !stim || count < 0) return SPHSM_ERR_INVALID;
    if (count == 0) return SPHSM_OK;
    if (!h->io_out_i || (size_t)count > h->io_out_cap) return fail(h, SPHSM_ERR_INVALID, "sphsm_set_stim_owned_async follows a sphsm_download_owned_async of at least `count` particles");
    CU(cudaSetDevice(h->prm.device));
    int rc;
    if ((rc = ensure_io_in(h, (size_t)count)) != 0) return rc;
    CU(cudaStreamWaitEvent(h->h2d_stream, h->ev_in_free, 0));  // the previous call's kernel has consumed the staging
    CU(cudaMemcpyAsync(h->io_in_f, stim, (size_t)count * sizeof(float), cudaMemcpyHostToDevice, h->h2d_stream));
    CU(cudaEventRecord(h->ev_in_ready, h->h2d_stream));
    CU(cudaStreamWaitEvent(h->stream, h->ev_in_ready, 0));
    const bool slab = h->dp.slab_on != 0;
    const int *rng = slab ? h->d_meta[h->meta_cur]->rng_all : nullptr;
    const int bound = slab ? h->own_bound : h->n;
    if (bound > 0) {
        LAUNCH(k_slot_of_range, cdiv(bound, 256), 256, rng, h->n, bound, h->cur.ID, h->slot_of);
        LAUNCH(k_set_stim_owned, cdiv(count, 256), 256, h->cur, (const int *)h->io_out_i, (const float *)h->io_in_f, count, (const int *)h->slot_of, rng, 0, h->n);
        h->slot_of_valid = false;
    }
    CU(cudaGetLastError());
    CU(cudaEventRecord(h->ev_in_free, h->stream));
    return SPHSM_OK;
}

extern "C" int sphsm_io_wait(sphsm_handle *h) {
    if (!h) return SPHSM_ERR_INVALID;
    CU(cudaSetDevice(h->prm.device));
    CU(cudaStreamSynchronize(h->h2d_stream));
    CU(cudaStreamSynchronize(h->d2h_stream));
    return SPHSM_OK;
}

