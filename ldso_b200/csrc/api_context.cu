// ldso_b200 C ABI implementation (include/ldso_b200.h): default settings, context lifetime, stream, image slots and pyramids,
// the one-shot scratch, kernel timing and debug getters. The other entry points live in api_ba.cu, api_frontend.cu,
// api_tracker.cu and api_posegraph.cu. No CPU fallback anywhere: every compute entry point launches sm_100a kernels or fails.
#include "context.h"
#include "img_kernels.cuh"

// ---------------------------------------------------------------------------------------------- kernel timing
static const char *const KT_NAMES[] = {"k1", "k2a", "k2b", "k3", "k2r", "actsel"};
#define KT_N 6
// average duration in microseconds per name of KT_NAMES (0 where none ran) of the timed launches so far; consumes their events
static void kt_collect(ldso_b200_ctx *c, double avg_us[KT_N], int cnt[KT_N]) {
    double tot[KT_N] = {};
    for (int i = 0; i < KT_N; i++) cnt[i] = 0;
    for (auto &k : c->kt) {
        float ms = 0;
        cudaEventElapsedTime(&ms, k.a, k.b);
        for (int i = 0; i < KT_N; i++) if (!strcmp(KT_NAMES[i], k.name)) { tot[i] += ms; cnt[i]++; }
        cudaEventDestroy(k.a); cudaEventDestroy(k.b);
    }
    c->kt.clear();
    for (int i = 0; i < KT_N; i++) avg_us[i] = cnt[i] ? 1e3 * tot[i] / cnt[i] : 0.0;
}
// LDSO_B200_KTIME times the loop kernels one by one, so the GN iteration then runs without its CUDA graph
static void read_timing_env(ldso_b200_ctx *c) {
    c->ktime = getenv("LDSO_B200_KTIME") != nullptr;
    c->use_graph = !c->ktime && getenv("LDSO_B200_NO_GRAPH") == nullptr;
}

extern "C" void ldso_b200_default_settings(ldso_b200_settings *s) {
    s->huberTH = 9;
    s->outlierTHSumComponent = 50 * 50;
    s->affineOptModeA = 1e12f;
    s->affineOptModeB = 1e8f;
    s->idepthFixPrior = 50 * 50;
    s->initialTransPrior = 1e10f;
    s->initialRotPrior = 1e11f;
    s->initialAffAPrior = 1e14f;
    s->initialAffBPrior = 1e14f;
    s->initialCalibHessian = 5e9f;
    s->frameEnergyTHN = 0.7f;
    s->frameEnergyTHFacMedian = 1.5f;
    s->frameEnergyTHConstWeight = 0.5f;
    s->overallEnergyTHWeight = 1;
    s->coarseCutoffTH = 20;
    s->thOptIterations = 1.2f;
    s->solverModeDelta = 0.00001;
    s->margWeightFac = 0.5f * 0.5f;
    s->maxPixSearch = 0.027f;
    s->outlierTH = 12 * 12;
    s->trace_stepsize = 1.0f;
    s->trace_GNThreshold = 0.1f;
    s->trace_extraSlackOnTH = 1.2f;
    s->trace_slackInterval = 1.5f;
    s->trace_minImprovementFactor = 2;
    s->minTraceTestRadius = 2;
    s->trace_GNIterations = 3;
}

extern "C" ldso_b200_ctx *ldso_b200_create(int device, int w, int h, int pyr_levels, const ldso_b200_settings *settings) {
    if (w <= 0 || h <= 0 || pyr_levels < 1 || pyr_levels > MAXLVL) return nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0 || device >= ndev) {
        fprintf(stderr, "ldso_b200: no CUDA device available (there is no CPU fallback)\n");
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    ldso_b200_ctx *c = new ldso_b200_ctx();
    c->device = device; c->w = w; c->h = h; c->levels = pyr_levels;
    if (settings) c->S = *settings; else ldso_b200_default_settings(&c->S);
    for (int l = 0; l < MAXLVL; l++) { c->lw[l] = w >> l; c->lh[l] = h >> l; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) c->sm_count = prop.multiProcessorCount;
    bool ok = true;
    ok = ok && cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) == cudaSuccess;
    c->own_stream = true;
    ok = ok && cudaMalloc(&c->ws_dev, sizeof(WinState)) == cudaSuccess;
    ok = ok && cudaMallocHost(&c->ws_host, sizeof(WinState)) == cudaSuccess;
    ok = ok && cudaMalloc(&c->iteration_dev, sizeof(int)) == cudaSuccess;
    // solve buffers: 4 + 1 + 1 + 1 matrices (n x n) and 6 vectors
    const size_t nn = (size_t) MAXN * MAXN;
    ok = ok && cudaMalloc(&c->solve_mem, sizeof(double) * (7 * nn + 8 * MAXN)) == cudaSuccess;
    ok = ok && tracker_alloc(c);
    if (!ok) { fprintf(stderr, "ldso_b200: context allocation failed: %s\n", cudaGetErrorString(cudaGetLastError())); delete c; return nullptr; }
    cudaMemset(c->solve_mem, 0, sizeof(double) * (7 * nn + 8 * MAXN));
    cudaMemset(c->trk.counter, 0, sizeof(unsigned));
    cudaMemset(c->iteration_dev, 0, sizeof(int));
    cudaMemset(c->ws_dev, 0, sizeof(WinState));
    memset(c->ws_host, 0, sizeof(WinState));
    double *p = c->solve_mem;
    c->sb.H_A = p; p += nn; c->sb.H_sc = p; p += nn; c->sb.HM = p; p += nn; c->sb.Pns = p; p += nn;
    c->sb.A0g = p; p += nn; c->sb.HSg = p; p += nn;     // assembled system handed from K2b to K3
    // lastHS | lastbS | lastX are contiguous: get_last_solution reads them back with one copy
    c->sb.lastHS = p; p += nn; c->sb.lastbS = p; p += MAXN; c->sb.lastX = p; p += MAXN;
    c->sb.b_A = p; p += MAXN; c->sb.b_sc = p; p += MAXN; c->sb.bM = p; p += MAXN;
    c->sb.dg = p; p += MAXN; c->sb.bFg = p; p += MAXN;
    ok = cudaMallocHost(&c->sol_host, sizeof(double) * (nn + 3 * MAXN)) == cudaSuccess;      // [lastHS | lastbS | lastX | scalars]
    if (!ok) { fprintf(stderr, "ldso_b200: pinned allocation failed\n"); delete c; return nullptr; }
    read_timing_env(c);
    c->use_pdl = getenv("LDSO_B200_NO_PDL") == nullptr;
    cudaEventCreateWithFlags(&c->frames_copied, cudaEventDisableTiming);
    ba_set_kernel_attributes();
    return c;
}

extern "C" void ldso_b200_destroy(ldso_b200_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->ktime && !c->kt.empty()) {
        double us[KT_N]; int cnt[KT_N];
        kt_collect(c, us, cnt);
        for (int i = 0; i < KT_N; i++)
            if (cnt[i]) fprintf(stderr, "[ldso_b200 ktime] %-12s n=%6d avg=%8.2f us\n", KT_NAMES[i], cnt[i], us[i]);
    }
    if (c->gn_graph) cudaGraphExecDestroy(c->gn_graph);
    free_window(c);
    for (int s = 0; s < NSLOTS; s++) for (int l = 0; l < MAXLVL; l++) if (c->img[s][l]) cudaFree(c->img[s][l]);
    for (int l = 0; l < MAXLVL; l++) for (int k = 0; k < 4; k++) if (c->trk.pc[l][k]) cudaFree(c->trk.pc[l][k]);
    for (int l = 0; l < MAXLVL; l++) { if (c->cd.id[l]) cudaFree(c->cd.id[l]); if (c->cd.ws[l]) cudaFree(c->cd.ws[l]); if (c->cd.bak[l]) cudaFree(c->cd.bak[l]); if (c->cd.pos[l]) cudaFree(c->cd.pos[l]); }
    if (c->cd.rows) cudaFree(c->cd.rows);
    if (c->cd.tot) cudaFree(c->cd.tot);
    if (c->cd.in) cudaFree(c->cd.in);
    if (c->scratch) cudaFree(c->scratch);
    if (c->ws_dev) cudaFree(c->ws_dev);
    if (c->ws_host) cudaFreeHost(c->ws_host);
    if (c->sol_host) cudaFreeHost(c->sol_host);
    if (c->scr.actsel_pin) cudaFreeHost(c->scr.actsel_pin);
    if (c->scr.buf) cudaFree(c->scr.buf);
    for (int r = 0; r < K2R_MAX_PEERS; r++) if (c->peer.opened[r]) cudaIpcCloseMemHandle(c->peer.opened[r]);
    if (c->peer.local) cudaFree(c->peer.local);
    if (c->peer.words) cudaFree(c->peer.words);
    if (c->peer.red_sum) cudaFree(c->peer.red_sum);
    if (c->iteration_dev) cudaFree(c->iteration_dev);
    if (c->solve_mem) cudaFree(c->solve_mem);
    if (c->trk.partials) cudaFree(c->trk.partials);
    if (c->trk.counter) cudaFree(c->trk.counter);
    if (c->trk.out_dev) cudaFree(c->trk.out_dev);
    if (c->trk.track_out) cudaFree(c->trk.track_out);
    if (c->own_stream && c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

extern "C" const char *ldso_b200_last_error(const ldso_b200_ctx *c) { return c ? c->err.c_str() : "null context"; }
extern "C" long long ldso_b200_launch_count(const ldso_b200_ctx *c) { return c ? c->launches : 0; }

extern "C" int ldso_b200_set_stream(ldso_b200_ctx *c, void *cuda_stream) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    if (c->own_stream && c->stream) { cudaStreamSynchronize(c->stream); cudaStreamDestroy(c->stream); }
    c->stream = (cudaStream_t) cuda_stream;
    c->own_stream = false;
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_synchronize(ldso_b200_ctx *c) {
    if (!c) return LDSO_B200_ERR_ARG;
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

// ---------------------------------------------------------------------------------------------- images
static int ensure_slot(ldso_b200_ctx *c, int slot) {
    if (slot < 0 || slot >= NSLOTS) return c->fail(LDSO_B200_ERR_ARG, "image slot out of range");
    for (int l = 0; l < c->levels; l++)
        if (!c->img[slot][l]) CUDA_CHECK_RET(c, cudaMalloc(&c->img[slot][l], sizeof(float4) * (size_t) c->lw[l] * c->lh[l]));
    if (!c->scratch) {
        c->scratch_floats = (size_t) c->w * c->h * 3;
        CUDA_CHECK_RET(c, cudaMalloc(&c->scratch, sizeof(float) * c->scratch_floats));
    }
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_upload_frame(ldso_b200_ctx *c, int slot, const float *const *dIp, int n_levels) {
    if (!c || !dIp) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    if (n_levels != c->levels) return c->fail(LDSO_B200_ERR_ARG, "n_levels != pyr_levels of the context");
    int rc = ensure_slot(c, slot);
    if (rc) return rc;
    for (int l = 0; l < c->levels; l++) {
        const int npx = c->lw[l] * c->lh[l];
        CUDA_CHECK_RET(c, cudaMemcpyAsync(c->scratch, dIp[l], sizeof(float) * 3 * npx, cudaMemcpyHostToDevice, c->stream));
        k_repack_aos3<<<(npx + 255) / 256, 256, 0, c->stream>>>(c->scratch, c->img[slot][l], npx);
        LAUNCH_CHECK(c);
        // the staging buffer is reused by the next level: the copies are stream-ordered, but the host buffer
        // of a pageable cudaMemcpyAsync is consumed before the call returns, so this is safe.
    }
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

int make_images_impl(ldso_b200_ctx *c, int slot, const float *color, bool wait_copy) {
    if (!c || !color) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    int rc = ensure_slot(c, slot);
    if (rc) return rc;
    CUDA_CHECK_RET(c, cudaMemcpyAsync(c->scratch, color, sizeof(float) * c->w * c->h, cudaMemcpyHostToDevice, c->stream));
    if (!c->copy_done) CUDA_CHECK_RET(c, cudaEventCreateWithFlags(&c->copy_done, cudaEventDisableTiming));
    CUDA_CHECK_RET(c, cudaEventRecord(c->copy_done, c->stream));
    for (int l = 0; l < c->levels; l++) {
        const int npx = c->lw[l] * c->lh[l];
        k_pyr_level<<<(npx + 255) / 256, 256, 0, c->stream>>>(c->scratch, l == 0 ? nullptr : c->img[slot][l - 1], c->img[slot][l],
                                                                c->lw[l], c->lh[l], l == 0 ? 0 : c->lw[l - 1]);
        LAUNCH_CHECK(c);
    }
    // the caller's buffer is free once the copy has landed; the pyramid kernels keep running asynchronously
    if (wait_copy) CUDA_CHECK_RET(c, cudaEventSynchronize(c->copy_done));
    return LDSO_B200_OK;
}
extern "C" int ldso_b200_make_images(ldso_b200_ctx *c, int slot, const float *color) { return make_images_impl(c, slot, color, true); }

extern "C" int ldso_b200_download_frame_level(ldso_b200_ctx *c, int slot, int lvl, float *out) {
    if (!c || !out || slot < 0 || slot >= NSLOTS || lvl < 0 || lvl >= c->levels || !c->img[slot][lvl]) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    const int npx = c->lw[lvl] * c->lh[lvl];
    k_unpack_aos3<<<(npx + 255) / 256, 256, 0, c->stream>>>(c->img[slot][lvl], c->scratch, npx);
    LAUNCH_CHECK(c);
    RET_IF(d2h(c, out, c->scratch, sizeof(float) * 3 * npx));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

// ---------------------------------------------------------------------------------------------- one-shot scratch
int reserve_scratch(ldso_b200_ctx *c, size_t bytes) {
    if (bytes <= c->scr.cap) return LDSO_B200_OK;
    if (c->scr.buf) cudaFree(c->scr.buf);
    c->scr.buf = nullptr; c->scr.cap = 0;
    CUDA_CHECK_RET(c, cudaMalloc(&c->scr.buf, bytes));
    c->scr.cap = bytes;
    return LDSO_B200_OK;
}

// Per-kernel CUDA-event timing of the GN loop (bench.py's roofline leg): enable != 0 starts collecting (graphs off),
// enable == 0 stops and returns the average duration in microseconds of K1, K2a, K2b, K3 since it was enabled.
extern "C" int ldso_b200_kernel_times(ldso_b200_ctx *c, int enable, double out_us[5]) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    double us[KT_N]; int cnt[KT_N];
    kt_collect(c, us, cnt);
    if (enable) {
        c->ktime = true;
        c->use_graph = false;
        return LDSO_B200_OK;
    }
    read_timing_env(c);
    if (out_us) for (int i = 0; i < 5; i++) out_us[i] = us[i];
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_debug_res_to_zero(ldso_b200_ctx *c, float *out8) {
    if (!c || !out8 || !c->have_window) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(d2h(c, out8, c->d.res_toZero, 32 * (size_t) c->d.nR));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_debug_clocks(ldso_b200_ctx *c, long long *out32) {
    if (!c || !out32) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    // out: 80 values = WinState::dbg[0..63] then DevWindow::dbg[0..15]
    RET_IF(d2h(c, out32, c->ws_dev->dbg, sizeof(long long) * 64));
    if (c->d.dbg) RET_IF(d2h(c, out32 + 64, c->d.dbg, sizeof(long long) * 16));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_debug_cta_spans(ldso_b200_ctx *c, long long *out, int cap_items) {
    if (!c || !out || !c->d.dbg) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    const int n = std::min(cap_items, c->d.nItems);
    RET_IF(d2h(c, out, c->d.dbg + 32, sizeof(long long) * 3 * n));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return n;
}

extern "C" int ldso_b200_get_nullspace_projector(ldso_b200_ctx *c, double *P) {
    if (!c || !c->have_frames || !P) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    RET_IF(d2h(c, P, c->sb.Pns, sizeof(double) * c->n * c->n));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}
