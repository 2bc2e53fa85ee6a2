// sphsm_host_step.cuh — the step on one GPU: per-group timers, neighbour grid (counting / radix sort, gather), shape-matching sums, staged and fused step, CUDA-graph replay
// Host code of libsphsm_b200.so, textually included by sphsm_capi.cu (one translation unit: the handle, the LAUNCH / CU macros and
// the static helpers defined there are in scope).
#pragma once

// ---------------------------------------------------------------------------------------------------
// the step
struct GroupTimer {  // records an event at each kernel-group boundary while profiling
    sphsm_handle *h;
    int idx = 0;
    int groups[SPHSM_NUM_KERNEL_GROUPS + 2];
    long long l0;
    explicit GroupTimer(sphsm_handle *hh) : h(hh) {
        l0 = h->launches;
        if (h->profiling) cudaEventRecord(h->ev[0], h->stream);
    }
    void end_group(int g) {
        if (!h->profiling) return;
        groups[idx] = g;
        h->group_launches[g] += (int)(h->launches - l0);
        l0 = h->launches;
        idx++;
        cudaEventRecord(h->ev[idx], h->stream);
    }
    void finish() {
        if (!h->profiling) return;
        cudaEventSynchronize(h->ev[idx]);
        for (int k = 0; k < idx; k++) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, h->ev[k], h->ev[k + 1]);
            h->group_ms[groups[k]] += ms;
        }
    }
};

static void swap_sets(sphsm_handle *h, bool all) {
    std::swap(h->cur.P, h->alt.P); std::swap(h->cur.VEL, h->alt.VEL); std::swap(h->cur.O, h->alt.O);
    std::swap(h->cur.E, h->alt.E); std::swap(h->cur.ID, h->alt.ID); std::swap(h->cur.PB, h->alt.PB);
    if (all) {
        std::swap(h->cur.C, h->alt.C); std::swap(h->cur.V, h->alt.V); std::swap(h->cur.S, h->alt.S);
        std::swap(h->cur.ACC, h->alt.ACC); std::swap(h->cur.GOAL, h->alt.GOAL); std::swap(h->cur.PV, h->alt.PV);
    }
}

// Find_neighbors: hash -> radix sort -> cell table -> reorder.  grid_sort() is the first half (keys + sorted
// permutation), grid_finish() the second (cell table + gather into the new slot order).  The fast path runs the
// shape-matching sums and solve BETWEEN the two halves (they do not depend on slot order) so that the gather can apply
// stage 2's per-particle map while the values are in registers (k_reorder_goal).
static bool use_counting_sort(const sphsm_handle *h) {
    const int mode = h->prm.reserved[2];  // 0 auto, 1 LSD radix sort, 2 counting sort
    if (mode == 1) return false;
    if (mode == 2) return true;
    return (long long)h->dp.num_cells <= 8ll * std::max(h->n, 1) + (1ll << 20);
}

// one pass over the full key: count per cell -> scan (= the cell table) -> scatter -> canonical in-cell order
// n_dev != nullptr (slab step): the entry count is *n_dev + n_add in device memory and h->n is an upper bound for the grids
static int grid_sort_counting(sphsm_handle *h, GroupTimer *gt, const int *n_dev = nullptr, int n_add = 0, int n_grid = -1) {
    const int n = n_grid >= 0 ? n_grid : h->n, m = h->dp.num_cells + 1;  // cells + the limbo bucket
    const int tiles = cdiv(m + 1, SCAN_TILE);
    if (h->counts_ready) h->counts_ready = false;  // pass B filed keys, ranks and counts of these positions while it held them
    else LAUNCH(k_cell_count, cdiv(n, 256), 256, h->dp, h->cur.P, h->keys[0], h->keys[1], h->cell_count, n_dev, n_add);
    if (gt) gt->end_group(KG_HASH);
    if (n_dev) trace_mark(h, "  cells counted");
    LAUNCH(k_scan_onepass, tiles, SCAN_THREADS, h->cell_count, m, h->cell_start, h->scan_state, h->scan_ctl, h->big_cells, h->big_count);
    if (n_dev) trace_mark(h, "  cell table scanned");
    LAUNCH(k_cell_scatter, cdiv(n, 256), 256, n, h->keys[0], h->keys[1], h->cell_start, h->vals[0], h->skeys, n_dev, n_add);
    if (n_dev) trace_mark(h, "  slots scattered");
    h->key_sorted = h->skeys;
    // cells of up to BIG_CELL entries get their canonical order inside the gather (grid_finish); the listed fuller ones here
    LAUNCH(k_cell_sort_big, 64, 256, h->cell_start, h->vals[0], h->vals[1], h->cur.ID, h->big_cells, h->big_count, h->scan_ctl);
    h->sorted_buf = 0;
    h->order_inline = true;
    h->bounds_ready = true;
    if (gt) gt->end_group(KG_SORT);
    return SPHSM_OK;
}

static int grid_sort(sphsm_handle *h, GroupTimer *gt, const int *n_dev = nullptr, int n_add = 0, int n_grid = -1) {
    const int n = h->n;
    if (use_counting_sort(h) || n_dev) return grid_sort_counting(h, gt, n_dev, n_add, n_grid);  // (the slab step always sorts by counting)
    drop_counts(h);
    h->bounds_ready = false;
    h->order_inline = false;
    const int passes = h->sort_passes;
    const int tiles = cdiv(n, SORT_TILE);
    if (!h->dry_run) {  // (a replayed graph carries its own copies of these nodes)
        CU(cudaMemsetAsync(h->ghist, 0, MAX_SORT_PASSES * RADIX * sizeof(uint32_t), h->stream));
        CU(cudaMemsetAsync(h->tile_state, 0, (size_t)passes * tiles * RADIX * sizeof(uint32_t), h->stream));
        CU(cudaMemsetAsync(h->tile_counter, 0, MAX_SORT_PASSES * sizeof(uint32_t), h->stream));
    }
    LAUNCH(k_hash, std::min(cdiv(n, 256), 8 * 148), 256, h->dp, h->cur.P, h->keys[0], h->ghist, passes);
    if (gt) gt->end_group(KG_HASH);
    int src = 0;
    for (int k = 0; k < passes; k++) {
        LAUNCH(k_radix_pass, tiles, SORT_THREADS, h->keys[src], k == 0 ? nullptr : h->vals[src], h->keys[src ^ 1], h->vals[src ^ 1], n,
               k * RADIX_BITS, h->ghist + k * RADIX, h->tile_state + (size_t)k * tiles * RADIX, h->tile_counter + k);
        src ^= 1;
    }
    h->sorted_buf = src;
    h->key_sorted = h->keys[src];
    // in-cell order = ascending original index: the reference's bucket order (strict mode), and the canonical order that
    // makes both sides of a slab face hold the shared plane identically (slab mode; reserved[1] forces it on one GPU)
    // (the slab step orders only the planes on either side of its faces, once the plane boundaries are known)
    if (h->prm.strict || h->prm.reserved[1])
        LAUNCH(k_cell_order_fix, cdiv(n, 128), 128, h->keys[src], h->vals[src], h->cur.ID, n, (uint32_t)h->dp.num_cells, 0, n);
    if (gt) gt->end_group(KG_SORT);
    return SPHSM_OK;
}

// fuse_goal: 0 = plain gather; 1 / 2 = gather + goal / predicted / corrected velocity (2 also stores GOAL and PV)
// n_dev != nullptr: the live count is read from device memory (grid sized for h->n, an upper bound)
static int grid_finish(sphsm_handle *h, GroupTimer *gt, int fuse_goal, bool bounds_done = false, const int *n_dev = nullptr, int n_grid = -1) {
    const int n = n_grid >= 0 ? n_grid : h->n, src = h->sorted_buf;
    if (!bounds_done && !h->bounds_ready) LAUNCH(k_cell_bounds, cdiv(n + 1, 256), 256, h->keys[src], h->cell_start, n, h->dp.num_cells);
    // counting sort: the gather applies the in-cell order itself and leaves the final permutation in the other index buffer
    const int order_cells = h->order_inline ? h->dp.num_cells : 0;
    h->perm = h->order_inline ? h->vals[src ^ 1] : h->vals[src];
    if (fuse_goal) {
        if (fuse_goal == 2) LAUNCH(k_reorder_goal<true>, cdiv(n, 256), 256, h->dp, h->vals[src], h->cur, h->alt, h->sm, n_dev, h->skeys, h->cell_start, order_cells, h->vals[src ^ 1]);
        else LAUNCH(k_reorder_goal<false>, cdiv(n, 256), 256, h->dp, h->vals[src], h->cur, h->alt, h->sm, n_dev, h->skeys, h->cell_start, order_cells, h->vals[src ^ 1]);
        swap_sets(h, false);
        std::swap(h->cur.C, h->alt.C);
        std::swap(h->cur.GOAL, h->alt.GOAL);
        std::swap(h->cur.PV, h->alt.PV);
    } else {
        const bool all = h->prm.diagnostics || h->inter_live;
        LAUNCH(k_reorder, cdiv(n, 256), 256, n, h->vals[src], h->cur, h->alt, all ? 1 : 0, h->skeys, h->cell_start, order_cells, h->vals[src ^ 1]);
        swap_sets(h, all);
    }
    if (gt) gt->end_group(KG_GRID);
    CU(cudaGetLastError());
    h->grid_valid = true;
    h->slot_of_valid = false;
    return SPHSM_OK;
}

static int build_grid(sphsm_handle *h, GroupTimer *gt) {
    if (h->n == 0) { h->grid_valid = true; return SPHSM_OK; }
    h->prev_vel_valid = false;  // a stand-alone re-sort moves every slot: the last step's gather source no longer lines up (freeze_source)
    int rc;
    if ((rc = grid_sort(h, gt)) != 0) return rc;
    return grid_finish(h, gt, 0);
}

static int ensure_slot_of(sphsm_handle *h) {
    if (h->slot_of_valid || h->n == 0) return SPHSM_OK;
    LAUNCH(k_slot_of, cdiv(h->n, 256), 256, h->n, h->cur.ID, h->slot_of);
    CU(cudaGetLastError());
    h->slot_of_valid = true;
    return SPHSM_OK;
}

// sums over particles end in h->totals; in slab mode the host combines them across ranks (ncclAllReduce) between parts
static int comm_allreduce(sphsm_handle *h, int count);

// the sums run BEFORE the gather, over the unsorted arrays: in slab mode that extent includes the message regions
static DevParams moment_params(sphsm_handle *h) {
    DevParams d = h->dp;
    if (h->mom_n) d.n = h->mom_n;
    return d;
}
static int rest_part1(sphsm_handle *h) {
    const int B = h->red_blocks;
    LAUNCH(k_rest_pass1, B, 256, moment_params(h), h->cur.P, h->cur.O, h->partial);
    LAUNCH(k_sum_partials_par, 5, 256, h->partial, B, 5, h->totals);
    return SPHSM_OK;
}
static int rest_part2(sphsm_handle *h) {
    const int B = h->red_blocks;
    LAUNCH(k_rest_finalize1, 1, 1, h->totals, h->sm);
    LAUNCH(k_rest_pass2, dim3(B, 10), 256, moment_params(h), h->cur.P, h->cur.O, h->sm, h->partial);
    for (int r = 0; r < 10; r++) LAUNCH(k_sum_partials_par, 9, 256, h->partial + (size_t)r * B * 9, B, 9, h->totals + r * 9);
    return SPHSM_OK;
}
static int rest_part3(sphsm_handle *h) {
    LAUNCH(k_rest_finalize2, 1, 1, h->totals, h->sm, h->scratch);
    CU(cudaGetLastError());
    h->rest_dirty = false;
    return SPHSM_OK;
}
static int moments_part(sphsm_handle *h) {
    // one partial per block and a 33-double block reduction each: keep >= 2048 particles per block (at a slab's 1M
    // particles the full 8 x SMs grid spent most of its 32 us in the reductions)
    // Slab mode: every particle is summed by the rank that integrated it last step, i.e. over that rank's owned slot range
    // as it stood BEFORE this step's exchange (migrants on their way out included, arrivals not): each particle exactly
    // once across ranks, and the sums need neither the exchange nor the sort, so they start with the step.  The range is
    // read from device memory (the SlabMeta the previous step's sort wrote).
    DevParams d = h->dp;
    const int *rng = nullptr;
    int count = d.n;
    if (d.slab_on) {
        rng = h->d_meta[h->meta_cur]->rng_all;
        count = h->own_bound;
        d.slab_on = 0;
    }
    const int B = std::max(1, std::min(h->red_blocks, cdiv(std::max(count, 1), 2048)));
    if (h->dp.quadratic) LAUNCH(k_moments<9>, B, 256, d, h->cur.P, h->cur.O, h->sm, h->partial, rng);
    else LAUNCH(k_moments<3>, B, 256, d, h->cur.P, h->cur.O, h->sm, h->partial, rng);
    const int nacc = h->dp.quadratic ? 33 : 15;
    if (h->comm_mode == 1) LAUNCH(k_sum_partials_par, nacc + 1, 256, h->partial, B, nacc, h->totals, (const int *)h->d_err);  // + the rank's error state: it rides on the allreduce
    else LAUNCH(k_sum_partials_par, nacc, 256, h->partial, B, nacc, h->totals, (const int *)nullptr);
    return SPHSM_OK;
}
// the per-step moment allreduce (NCCL mode: + the summed error flag, which the sort's k_mg_meta passes on to the host read-back)
static int moment_allreduce(sphsm_handle *h) {
    const int nacc = h->dp.quadratic ? 33 : 15;
    if (h->comm_mode != 1 || h->nranks == 1) return comm_allreduce(h, nacc);
    return comm_allreduce(h, nacc + 1);
}

static int rest_moments(sphsm_handle *h) {
    int rc;
    if ((rc = rest_part1(h)) != 0 || (rc = comm_allreduce(h, 5)) != 0) return rc;
    if ((rc = rest_part2(h)) != 0 || (rc = comm_allreduce(h, 90)) != 0) return rc;
    return rest_part3(h);
}

// calculate_corrected_velocity
// the fast path's shape-matching transform of this step: moment sums (any slot order) + the single-thread solve
static int sm_transform_fast(sphsm_handle *h) {
    int rc;
    if (h->rest_dirty && (rc = rest_moments(h)) != 0) return rc;
    if ((rc = moments_part(h)) != 0 || (rc = moment_allreduce(h)) != 0) return rc;
    LAUNCH(k_sm_solve, 1, 1, h->dp, h->totals, h->sm);
    return SPHSM_OK;
}

template <bool STRICT>
static int corrected_velocity(sphsm_handle *h, bool diag, GroupTimer *gt, int store = 7) {
    const int n = h->n;
    if (n == 0) return SPHSM_OK;
    int rc;
    if (n > 1 && (store & 3)) {  // projectPositions returns early for <= 1 particle, cpp:236
        if (STRICT) {
            if ((rc = ensure_slot_of(h)) != 0) return rc;
            LAUNCH(k_sm_strict, 1, 1, h->dp, h->cur.P, h->cur.O, h->slot_of, h->sm, h->scratch);
        } else if ((rc = sm_transform_fast(h)) != 0) return rc;
    }
    if (gt) gt->end_group(KG_MOMENTS);
    const int keep_goal = n <= 1;  // projectPositions returned early: mGoalPos keeps its previous value
    if ((diag || keep_goal) && store == 7) h->goal_pv_stale = false;
    else if (!(diag || keep_goal)) h->goal_pv_stale = true;
    // the fast path comes here only with diag (sphsm_stage) or keep_goal (the single-particle step): one form of the kernel
    if (STRICT && !(diag || keep_goal)) LAUNCH((k_goal_cvel<true, false>), cdiv(n, 256), 256, h->dp, h->cur, h->sm, 0, store);
    else LAUNCH((k_goal_cvel<STRICT, true>), cdiv(n, 256), 256, h->dp, h->cur, h->sm, keep_goal, store);
    if (gt) gt->end_group(KG_GOAL);
    CU(cudaGetLastError());
    return SPHSM_OK;
}

template <bool STRICT>
static int run_stage(sphsm_handle *h, int stage) {
    const int n = h->n;
    int rc;
    if (stage < SPHSM_STAGE_FIND_NEIGHBORS || stage > SPHSM_STAGE_PROJECT_POSITIONS) return fail(h, SPHSM_ERR_INVALID, "unknown stage id");
    if (n == 0) return SPHSM_OK;
    if ((stage == 3 || stage == 4 || stage == 6) && !h->grid_valid && (rc = build_grid(h, nullptr)) != 0) return rc;
    switch (stage) {
        case SPHSM_STAGE_FIND_NEIGHBORS:
            return build_grid(h, nullptr);
        case SPHSM_STAGE_CORRECTED_VELOCITY:
            return corrected_velocity<STRICT>(h, true, nullptr);
        case SPHSM_STAGE_EXTERNAL_FORCES:  // predicted_vel only
            return corrected_velocity<STRICT>(h, true, nullptr, 4);
        case SPHSM_STAGE_PROJECT_POSITIONS:  // mGoalPos only
            return corrected_velocity<STRICT>(h, true, nullptr, 2);
        case SPHSM_STAGE_INTERMEDIATE_VELOCITY:
            LAUNCH(k_refresh_derived, cdiv(n, 256), 256, n, h->cur, 1, 0);
            LAUNCH((k_pass_a<STRICT, false, true>), cdiv(n, 128), 128, h->dp, h->cur, h->cell_start);
            break;
        case SPHSM_STAGE_DENSITY_PRESSURE:
            LAUNCH((k_pass_a<STRICT, true, false>), cdiv(n, 128), 128, h->dp, h->cur, h->cell_start);
            break;
        case SPHSM_STAGE_CELL_MODEL:
            LAUNCH(k_cell_model<STRICT>, cdiv(n, 256), 256, h->dp, h->cur);
            break;
        case SPHSM_STAGE_FORCE:
            LAUNCH(k_refresh_derived, cdiv(n, 256), 256, n, h->cur, 0, 1);
            if (h->egm.on) LAUNCH((k_pass_b<STRICT, PB_FORCE_ONLY | PB_EGM>), cdiv(n, 128), 128, h->dp, h->cur, (float4 *)nullptr, h->cell_start);
            else LAUNCH((k_pass_b<STRICT, PB_FORCE_ONLY>), cdiv(n, 128), 128, h->dp, h->cur, (float4 *)nullptr, h->cell_start);
            break;
        case SPHSM_STAGE_UPDATE:
            drop_counts(h);
            LAUNCH(k_update<STRICT>, cdiv(n, 256), 256, h->dp, h->cur);
            h->grid_valid = false;
            break;
        default:
            return fail(h, SPHSM_ERR_INVALID, "unknown stage id");
    }
    CU(cudaGetLastError());
    return SPHSM_OK;
}

// the fast-path neighbour passes over the owned slot range (count = own_end - own_begin)
// Small particle sets (the reference's own ~5k-particle inputs) take one warp per particle (sphsm_pass4w.cuh).  The choice
// follows the GLOBAL particle count, so that a slab rank and the single-GPU run of the same set use the same kernels (the
// bit-level slab parity depends on identical summation order).  SPHSM_WARP_PATH=0 disables it.
// The limit is a particle count because that is all the host knows; what actually decides is candidates per stencil row:
// measured with the limit lifted, a 64k LATTICE (3-6 candidates per row, most lanes idle) runs pass A / B in 56 / 108 us on
// this path against 16 / 21 us on the thread path, while the reference's meshes (45 per row) gain 10x.  Hence the second
// condition: at least 3 particles per occupied cell, estimated on the host from the positions as they were handed in
// (note_host_positions; the reference's sets have 4.9-5.1, lattices of spacing 0.9 h have 1.4).
static bool warp_path(const sphsm_handle *h) {
    if (!g_warp_path) return false;
    const int n = h->dp.slab_on ? h->n_global : h->n;
    if (n > WARP_PATH_MAX || h->host_cells.empty()) return false;
    return (double)n >= 3.0 * (double)h->host_cells.size();  // >= 3 particles per occupied cell: rows long enough for a warp
}

// slots [begin, end) minus the hole [hole_b, hole_e).  rng != nullptr (slab step): the range is read from device memory
// ({begin, end, hole_begin, hole_len}) and [begin, end) / the hole only size the grid: `end - begin - hole` is an upper bound of the
// target count.
static int launch_pass_a(sphsm_handle *h, int begin, int end, int hole_b = 0, int hole_e = 0, const int *rng = nullptr) {
    const int count = end - begin - (hole_e - hole_b);
    if (count <= 0) return SPHSM_OK;
    DevParams d = h->dp;
    d.own_begin = begin; d.own_end = end; d.hole_begin = hole_b; d.hole_len = hole_e - hole_b;

    if (warp_path(h)) LAUNCH(k_pass_a4w, cdiv((long long)count * 32, PTW), PTW, d, h->cur, h->cell_start, count, rng);
    else if (rng) LAUNCH(k_pass_a4<true>, cdiv(count, PT4), PT4, d, h->d_dp, h->cur, h->cell_start, h->key_sorted, rng);
    else LAUNCH(k_pass_a4<false>, cdiv(count, PT4), PT4, d, h->d_dp, h->cur, h->cell_start, h->key_sorted, rng);
    return SPHSM_OK;
}
// DIAG: ACC for the diagnostics download; EGM: the electrogram source Q (while electrograms are on)
template <bool DIAG, bool EGM>
static int launch_pass_b_as(sphsm_handle *h, const DevParams &d, int count, uint32_t *nk, uint32_t *nr, uint32_t *ncnt, const int *rng) {
    if (warp_path(h)) LAUNCH((k_pass_b4w<DIAG, EGM>), cdiv((long long)count * 32, PTW), PTW, d, h->cur, h->alt.P, h->cell_start, nk, nr, ncnt, count, rng);
    else if (rng) LAUNCH((k_pass_b4<DIAG, true, EGM>), cdiv(count, PT4), PT4, d, h->d_dp, h->cur, h->alt.P, h->cell_start, h->key_sorted, nk, nr, ncnt, rng);
    else LAUNCH((k_pass_b4<DIAG, false, EGM>), cdiv(count, PT4), PT4, d, h->d_dp, h->cur, h->alt.P, h->cell_start, h->key_sorted, nk, nr, ncnt, rng);
    return SPHSM_OK;
}
static int launch_pass_b(sphsm_handle *h, int begin, int end, bool diag, int hole_b = 0, int hole_e = 0, bool file_counts = false,
                         const int *rng = nullptr) {
    uint32_t *nk = file_counts ? h->keys[0] : nullptr, *nr = file_counts ? h->keys[1] : nullptr, *ncnt = file_counts ? h->cell_count : nullptr;
    const int count = end - begin - (hole_e - hole_b);
    if (count <= 0) return SPHSM_OK;
    DevParams d = h->dp;
    d.own_begin = begin; d.own_end = end; d.hole_begin = hole_b; d.hole_len = hole_e - hole_b;
    if (h->egm.on)
        return diag ? launch_pass_b_as<true, true>(h, d, count, nk, nr, ncnt, rng) : launch_pass_b_as<false, true>(h, d, count, nk, nr, ncnt, rng);
    return diag ? launch_pass_b_as<true, false>(h, d, count, nk, nr, ncnt, rng) : launch_pass_b_as<false, false>(h, d, count, nk, nr, ncnt, rng);
}

// one fused step: grid, shape matching, pass A, pass B
template <bool STRICT>
static int fused_step(sphsm_handle *h) {
    const int n = h->n;
    int rc;
    if (n == 0) return SPHSM_OK;
    const bool diag = h->prm.diagnostics != 0;
    if (memcmp(&h->dp, &h->dp_uploaded, sizeof(DevParams)) != 0) {  // n or a tunable changed since the last upload
        h->dp_uploaded = h->dp;
        CU(cudaMemcpyAsync(h->d_dp, &h->dp_uploaded, sizeof(DevParams), cudaMemcpyHostToDevice, h->stream));
    }
    GroupTimer gt(h);
    if constexpr (STRICT) {
        if ((rc = build_grid(h, &gt)) != 0) return rc;
        if ((rc = corrected_velocity<true>(h, diag, &gt)) != 0) return rc;
        LAUNCH((k_pass_a<true, true, true>), cdiv(n, 128), 128, h->dp, h->cur, h->cell_start);
        gt.end_group(KG_PASS_A);
        if (diag && h->egm.on) LAUNCH((k_pass_b<true, PB_FUSED_DIAG | PB_EGM>), cdiv(n, 128), 128, h->dp, h->cur, h->alt.P, h->cell_start);
        else if (diag) LAUNCH((k_pass_b<true, PB_FUSED_DIAG>), cdiv(n, 128), 128, h->dp, h->cur, h->alt.P, h->cell_start);
        else if (h->egm.on) LAUNCH((k_pass_b<true, PB_FUSED | PB_EGM>), cdiv(n, 128), 128, h->dp, h->cur, h->alt.P, h->cell_start);
        else LAUNCH((k_pass_b<true, PB_FUSED>), cdiv(n, 128), 128, h->dp, h->cur, h->alt.P, h->cell_start);
    } else {
        if (n > 1) {
            // sort -> shape-matching transform (slot-order independent) -> cell table + gather fused with stage 2's map
            // the moment sums and the solve only read the not-yet-sorted arrays: they run on the side stream beside the sort
            // and rejoin before the gather applies the transform (kept in line while the per-group timers are on)
            const bool fork = !h->rest_dirty && !h->profiling;
            if (fork) {
                if (!h->dry_run) {
                    CU(cudaEventRecord(h->ev_fork, h->stream));
                    CU(cudaStreamWaitEvent(h->side_stream, h->ev_fork, 0));
                }
                h->launch_stream = h->side_stream;
                rc = sm_transform_fast(h);
                h->launch_stream = h->stream;
                if (rc) return rc;
                if (!h->dry_run) CU(cudaEventRecord(h->ev_join, h->side_stream));
            }
            if ((rc = grid_sort(h, &gt)) != 0) return rc;
            if (fork) {
                if (!h->dry_run) CU(cudaStreamWaitEvent(h->stream, h->ev_join, 0));
            } else if ((rc = sm_transform_fast(h)) != 0) return rc;
            gt.end_group(KG_MOMENTS);
            if ((rc = grid_finish(h, &gt, diag ? 2 : 1)) != 0) return rc;
        } else {
            if ((rc = build_grid(h, &gt)) != 0) return rc;
            if ((rc = corrected_velocity<false>(h, diag, &gt)) != 0) return rc;
        }
        if ((rc = launch_pass_a(h, 0, n)) != 0) return rc;  // single GPU: own range = [0, n)
        gt.end_group(KG_PASS_A);
        // the counting sort of the NEXT step starts inside pass B: each thread files the key / rank / count of the position it
        // has just integrated (valid until anything else moves particles: drop_counts)
        const bool file_counts = h->comm_mode == 0 && use_counting_sort(h);
        if ((rc = launch_pass_b(h, 0, n, diag, 0, 0, file_counts)) != 0) return rc;
        h->counts_ready = file_counts;
    }
    std::swap(h->cur.P, h->alt.P);
    gt.end_group(KG_PASS_B);
    if (observe_on(h)) {  // pre-step Vm in PB.w, post-step Vm in E.x, new positions in cur.P, the source in Q
        if ((rc = observe_launch(h, nullptr, n)) != 0) return rc;
        gt.end_group(KG_OTHER);
    }
    CU(cudaGetLastError());
    gt.finish();
    h->grid_valid = false;
    h->inter_live = false;
    if (n > 1) {
        if (!STRICT) h->goal_pv_stale = !diag;  // (the strict path went through corrected_velocity, which set it)
        h->prev_vel_valid = true;
    }
    return SPHSM_OK;
}

// the staged step with an event pair around every stage (what the class's d_* timers report)
template <bool STRICT>
static int timed_staged_step(sphsm_handle *h) {
    for (int st = 1; st <= 7; st++) {
        CU(cudaEventRecord(h->ev[0], h->stream));
        int rc = run_stage<STRICT>(h, st);
        if (rc) return rc;
        CU(cudaEventRecord(h->ev[1], h->stream));
        CU(cudaEventSynchronize(h->ev[1]));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
        h->stage_time[st - 1] += ms * 1e-3;
    }
    h->inter_live = false;
    return observe_launch(h, nullptr, h->n);  // (outside the stage timers; PB.w is stage 6's pre-step Vm, E.x stage 7's result, Q stage 6's)
}

static int mg_step_nccl(sphsm_handle *h);  // the slab step (below)

// Small single-GPU steps are launch-latency bound (13 dependent launches of 3-5 us for a few microseconds of work each at the
// reference's own ~5k particles; still 2-4 % of the step at 1-2M), so the fast step is captured into a CUDA graph and replayed.  A step's launch sequence and
// arguments are a function of the handle's state only (no data-dependent host decisions on one GPU): that state — buffer
// pointers of both ping-pong sets, the device parameter block, the sort / counting flags — is the graph's signature.  A
// signature seen for the second time is captured (the ping-pong gives two signatures in steady state); on a hit the host
// runs the step's bookkeeping with launches suppressed (dry_run) and launches the graph.  Any mutator that changes what a
// step would launch changes the signature, so a stale graph cannot be picked.  params.reserved[4] = 1 turns graphs off.
static const int GRAPH_MAX_N = getenv("SPHSM_GRAPH_MAX_N") ? atoi(getenv("SPHSM_GRAPH_MAX_N")) : (1 << 22);  // measured: -22 % at 5k, -3.6 % at 1M, -2.2 % at 2M particles
static bool graph_eligible(const sphsm_handle *h) {
    static const bool env_off = getenv("SPHSM_NO_GRAPH") != nullptr;
    return !env_off && h->comm_mode == 0 && !h->prm.strict && !h->profiling && !h->stage_timing && !g_sync_debug && h->prm.reserved[4] != 1 && h->n > 1 &&
           h->n <= GRAPH_MAX_N && !h->rest_dirty && memcmp(&h->dp, &h->dp_uploaded, sizeof(DevParams)) == 0;
}
static std::string step_signature(const sphsm_handle *h) {
    std::string sig;
    auto put = [&](const void *ptr, size_t bytes) { sig.append(reinterpret_cast<const char *>(ptr), bytes); };
    put(&h->cur, sizeof(Arrays));
    put(&h->alt, sizeof(Arrays));
    put(&h->dp, sizeof(DevParams));
    put(&h->prm, sizeof(sphsm_params));
    const void *ptrs[] = {h->cell_start, h->cell_count, h->scan_state, h->scan_ctl, h->keys[0], h->keys[1], h->vals[0], h->vals[1], h->big_cells, h->big_count,
                          h->sm, h->partial, h->totals, h->d_dp, h->ghist, h->tile_state, h->tile_counter, h->scratch, h->skeys};
    put(ptrs, sizeof(ptrs));
    const void *rec_ptrs[] = {h->rec.maps, h->rec.probe_of, h->rec.trace, h->rec.stamp, h->step_ctl};  // (all null while recording is off)
    put(rec_ptrs, sizeof(rec_ptrs));
    const float rec_vm[] = {h->rec.vm_up, h->rec.vm_down};
    put(rec_vm, sizeof(rec_vm));
    const int rec_cfg[] = {(int)h->rec.on, h->rec.cap, h->rec.n_probes, h->rec.rows};
    put(rec_cfg, sizeof(rec_cfg));
    const void *egm_ptrs[] = {h->egm.Q, h->egm.el, h->egm.partial, h->egm.ring};  // (all null while electrograms are off; Q is in Arrays too)
    put(egm_ptrs, sizeof(egm_ptrs));
    const float egm_f[] = {h->egm.gain, h->egm.eps2};
    put(egm_f, sizeof(egm_f));
    const int egm_cfg[] = {(int)h->egm.on, h->egm.n_el, h->egm.rows, h->egm.grid};
    put(egm_cfg, sizeof(egm_cfg));
    const int flags[] = {h->counts_ready, h->bounds_ready, h->sorted_buf, h->red_blocks, h->sort_passes, (int)h->grid_valid, (int)warp_path(h)};
    put(flags, sizeof(flags));
    return sig;
}
static int graph_step(sphsm_handle *h) {
    if (!graph_eligible(h)) return fused_step<false>(h);
    const std::string sig = step_signature(h);
    for (auto &gx : h->graphs) {
        if (gx.sig == sig) {
            h->dry_run = true;
            const int rc = fused_step<false>(h);
            h->dry_run = false;
            if (rc) return rc;
            CU(cudaGraphLaunch(gx.exec, h->stream));
            return SPHSM_OK;
        }
    }
    bool seen = false;
    for (auto &x : h->seen_sigs) seen = seen || x == sig;
    if (!seen) {
        if (h->seen_sigs.size() >= 16) h->seen_sigs.clear();
        h->seen_sigs.push_back(sig);
        return fused_step<false>(h);
    }
    // second sighting: capture this step (it executes when the graph is launched below)
    cudaGraph_t graph = nullptr;
    CU(cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeRelaxed));
    const int rc = fused_step<false>(h);
    cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
    if (rc || ce != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        return rc ? rc : fail(h, SPHSM_ERR_CUDA, "CUDA graph capture of the step failed");
    }
    cudaGraphExec_t exec = nullptr;
    ce = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce != cudaSuccess) return fail(h, SPHSM_ERR_CUDA, "cudaGraphInstantiate failed");
    if (h->graphs.size() >= 8) {
        for (auto &gx : h->graphs) cudaGraphExecDestroy(gx.exec);
        h->graphs.clear();
    }
    h->graphs.push_back({sig, exec});
    CU(cudaGraphLaunch(exec, h->stream));
    return SPHSM_OK;
}

