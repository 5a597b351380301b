// ldso_b200 C ABI implementation (include/ldso_b200.h), bundle adjustment: the window arena, frames, marginalisation prior,
// the piecewise entry points, the fused Gauss-Newton loop and its CUDA graph, the read-back mirror, optimize_from_host_* and
// the shard / peer exchange.
#include "context.h"
#include "host_math.h"
#include "ba_k1.cuh"
#include "ba_k2.cuh"
#include "ba_k3.cuh"

static_assert(K1_THREADS / 32 == MAXF, "phase B maps one warp to one target frame");

void ba_set_kernel_attributes() {
    cudaFuncSetAttribute(k1_linearize_accumulate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) k1_smem_bytes(64));
    cudaFuncSetAttribute(k3_solve_step, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) K3_SMEM_BYTES);
    cudaFuncSetAttribute(k2b_stitch, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) K2B_SMEM_BYTES);
}

// ---------------------------------------------------------------------------------------------- window
static void free_derived(ldso_b200_ctx *c) {
    for (void *p : c->derived_allocs) cudaFree(p);
    c->derived_allocs.clear();
    c->d.items = nullptr; c->d.host_item_begin = nullptr; c->d.res_newest_slot = nullptr;
    c->d.partials = nullptr; c->d.item_stats = nullptr; c->d.red = nullptr; c->d.dbg = nullptr;
}

void free_window(ldso_b200_ctx *c) {
    for (void *p : c->win_allocs) cudaFree(p);
    c->win_allocs.clear();
    free_derived(c);
    if (c->arena_dev) { cudaFree(c->arena_dev); c->arena_dev = nullptr; }
    if (c->arena_host) { cudaFreeHost(c->arena_host); c->arena_host = nullptr; }
    invalidate_results(c);
    c->gn_graph_valid = false;
    c->have_window = false;
}

template<typename T>
static int dev_alloc(ldso_b200_ctx *c, T **p, size_t count, std::vector<void *> *owner = nullptr) {
    void *q = nullptr;
    CUDA_CHECK_RET(c, cudaMalloc(&q, sizeof(T) * std::max<size_t>(count, 128)));   // empty windows still get valid buffers
    (owner ? *owner : c->win_allocs).push_back(q);
    *p = (T *) q;
    return 0;
}

// Window memory: ONE device arena + ONE pinned host mirror with the same layout.
//   [topology | inputs ......................... | pt_idepth pt_idepth_zero | results ............ ]
//    ^ uploaded only when the CSR changes         ^---- upload range ------^
//                                                 ^----------- download range (one D2H) ----------^
// so a set_window is one pack + one cudaMemcpyAsync + one memset, and reading points/residuals back is one copy.
static int alloc_window(ldso_b200_ctx *c, int nP, int nR) {
    DevWindow &d = c->d;
    Arena A;
    const size_t nPs = std::max(nP, 32), nRs = std::max(nR, 32);
    auto &L = c->lay;
    L.pt_host = A.take(4 * nPs); L.pt_res_begin = A.take(4 * (nPs + 1)); L.res_point = A.take(4 * nRs); L.res_target = A.take(4 * nRs);
    L.topo_end = A.off;
    L.pt_u = A.take(4 * nPs); L.pt_v = A.take(4 * nPs); L.pt_color = A.take(32 * nPs); L.pt_weights = A.take(32 * nPs);
    L.pt_priorF = A.take(4 * nPs); L.pt_idepth_backup = A.take(4 * nPs); L.res_lin = A.take(nRs);
    L.res_state = A.take(nRs);
    L.dl_begin = A.off;
    L.pt_idepth = A.take(4 * nPs); L.pt_idepth_zero = A.take(4 * nPs);
    L.ul_end = A.off;
    L.pt_step = A.take(4 * nPs); L.pt_HdiF = A.take(4 * nPs); L.pt_bdSumF = A.take(4 * nPs); L.pt_Hdd = A.take(4 * nPs);
    L.pt_bd = A.take(4 * nPs); L.pt_Hcd = A.take(16 * nPs);
    L.res_new_state = A.take(nRs); L.res_active = A.take(nRs); L.res_energy = A.take(4 * nRs); L.res_new_energy = A.take(4 * nRs);
    L.res_new_energy_wo = A.take(4 * nRs);
    L.dl_light_end = A.off;
    L.res_JpJdF = A.take(32 * nRs);
    L.dl_end = A.off;
    L.res_JpJdF_new = A.take(32 * nRs);
    L.total = A.off;
    // res_state is both an input and a result: it sits right before dl_begin and is fetched separately (tiny)
    CUDA_CHECK_RET(c, cudaMalloc(&c->arena_dev, L.total));
    CUDA_CHECK_RET(c, cudaMallocHost(&c->arena_host, L.total));
    memset(c->arena_host, 0, L.total);
    char *B = c->arena_dev;
    d.pt_host = (int *) (B + L.pt_host); d.pt_res_begin = (int *) (B + L.pt_res_begin);
    d.res_point = (int *) (B + L.res_point); d.res_target = (int *) (B + L.res_target);
    d.pt_u = (float *) (B + L.pt_u); d.pt_v = (float *) (B + L.pt_v); d.pt_color = (float *) (B + L.pt_color);
    d.pt_weights = (float *) (B + L.pt_weights); d.pt_priorF = (float *) (B + L.pt_priorF);
    d.pt_idepth_backup = (float *) (B + L.pt_idepth_backup); d.res_lin = (uint8_t *) (B + L.res_lin);
    d.res_state = (uint8_t *) (B + L.res_state);
    d.pt_idepth = (float *) (B + L.pt_idepth); d.pt_idepth_zero = (float *) (B + L.pt_idepth_zero);
    d.pt_step = (float *) (B + L.pt_step); d.pt_HdiF = (float *) (B + L.pt_HdiF); d.pt_bdSumF = (float *) (B + L.pt_bdSumF);
    d.pt_Hdd = (float *) (B + L.pt_Hdd); d.pt_bd = (float *) (B + L.pt_bd); d.pt_Hcd = (float *) (B + L.pt_Hcd);
    d.res_new_state = (uint8_t *) (B + L.res_new_state); d.res_active = (uint8_t *) (B + L.res_active);
    d.res_energy = (float *) (B + L.res_energy); d.res_new_energy = (float *) (B + L.res_new_energy);
    d.res_new_energy_wo = (float *) (B + L.res_new_energy_wo); d.res_JpJdF = (float *) (B + L.res_JpJdF);
    d.res_JpJdF_new = (float *) (B + L.res_JpJdF_new);
    // big arrays only the piecewise API / tests touch
    int rc = 0;
    rc |= dev_alloc(c, &d.res_J, (size_t) nR * 74);
    rc |= dev_alloc(c, &d.res_proj, (size_t) nR * 16); rc |= dev_alloc(c, &d.res_cpt, (size_t) nR * 3);
    rc |= dev_alloc(c, &d.res_toZero, (size_t) nR * 8);
    rc |= dev_alloc(c, &c->pt_sel_dev, nP);
    return rc ? LDSO_B200_ERR_CUDA : LDSO_B200_OK;
}

extern "C" int ldso_b200_set_window(ldso_b200_ctx *c, const ldso_b200_window *win) {
    if (!c || !win) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    const int nP = win->nPoints, nR = win->nResiduals;
    if (nP < 0 || nR < 0) return c->fail(LDSO_B200_ERR_ARG, "negative sizes");
    for (int p = 0; p < nP; p++) {
        if (win->pt_host[p] < 0 || win->pt_host[p] >= MAXF) return c->fail(LDSO_B200_ERR_ARG, "pt_host out of range");
        if (p > 0 && win->pt_host[p] < win->pt_host[p - 1]) return c->fail(LDSO_B200_ERR_ARG, "points must be ordered by host frame");
        if (win->res_begin[p + 1] < win->res_begin[p]) return c->fail(LDSO_B200_ERR_ARG, "res_begin must be non-decreasing");
        if (win->res_begin[p + 1] - win->res_begin[p] > MAXF) return c->fail(LDSO_B200_ERR_ARG, "more than MAX_FRAMES residuals on a point");
    }
    if (nP > 0 && (win->res_begin[0] != 0 || win->res_begin[nP] != nR)) return c->fail(LDSO_B200_ERR_ARG, "res_begin does not cover the residual arrays");
    for (int r = 0; r < nR; r++) if (win->res_target[r] < 0 || win->res_target[r] >= MAXF) return c->fail(LDSO_B200_ERR_ARG, "res_target out of range");
    if (c->window_copied) CUDA_CHECK_RET(c, cudaEventSynchronize(c->window_copied));     // the pinned mirror may still be in flight
    RET_IF(wait_results(c));                                                              // ... or be the target of a queued read-back
    DevWindow &d = c->d;
    const bool same_topology = c->have_window && d.nP == nP && d.nR == nR && (int) c->h_pt_host.size() == nP && nP > 0 &&
                               std::equal(win->pt_host, win->pt_host + nP, c->h_pt_host.begin()) &&
                               std::equal(win->res_begin, win->res_begin + nP + 1, c->h_res_begin.begin()) &&
                               std::equal(win->res_target, win->res_target + nR, c->h_res_target.begin());
    auto &L = c->lay;
    if (!same_topology) {
        free_window(c);
        memset(&d, 0, sizeof(d));
        d.nP = nP; d.nR = nR;
        c->h_pt_host.assign(win->pt_host, win->pt_host + nP);
        c->h_res_begin.assign(win->res_begin, win->res_begin + nP + 1);
        if (nP == 0) c->h_res_begin.assign(1, 0);
        c->h_res_target.assign(win->res_target, win->res_target + nR);
        int rc = alloc_window(c, nP, nR);
        if (rc) return rc;
        d.newest_offset = 0;
        d.newest_total = -1;   // derived
        c->derived_dirty = true;
        char *H = c->arena_host;
        memcpy(H + L.pt_host, win->pt_host, 4 * (size_t) nP);
        memcpy(H + L.pt_res_begin, c->h_res_begin.data(), 4 * ((size_t) nP + 1));
        int *rp = (int *) (H + L.res_point);
        for (int p = 0; p < nP; p++) for (int r = c->h_res_begin[p]; r < c->h_res_begin[p + 1]; r++) rp[r] = p;
        memcpy(H + L.res_target, win->res_target, 4 * (size_t) nR);
    }
    // ---- pack the per-call inputs into the pinned mirror
    char *H = c->arena_host;
    memcpy(H + L.pt_u, win->pt_u, 4 * (size_t) nP); memcpy(H + L.pt_v, win->pt_v, 4 * (size_t) nP);
    memcpy(H + L.pt_color, win->pt_color, 32 * (size_t) nP); memcpy(H + L.pt_weights, win->pt_weights, 32 * (size_t) nP);
    float *priorF = (float *) (H + L.pt_priorF);
    for (int p = 0; p < nP; p++)   // PointHessian::takeData (PointHessian.h:112-117)
        priorF[p] = (win->pt_has_prior && win->pt_has_prior[p]) ? c->S.idepthFixPrior * SCALE_IDEPTH * SCALE_IDEPTH : 0.f;
    memcpy(H + L.pt_idepth_backup, win->pt_idepth, 4 * (size_t) nP);
    if (win->res_is_linearized) memcpy(H + L.res_lin, win->res_is_linearized, nR); else memset(H + L.res_lin, 0, std::max(nR, 1));
    c->has_lin = false;
    if (win->res_is_linearized) for (int r = 0; r < nR; r++) if (win->res_is_linearized[r]) { c->has_lin = true; break; }
    if (win->res_state) memcpy(H + L.res_state, win->res_state, nR); else memset(H + L.res_state, LDSO_B200_RES_IN, std::max(nR, 1));
    memcpy(H + L.pt_idepth, win->pt_idepth, 4 * (size_t) nP); memcpy(H + L.pt_idepth_zero, win->pt_idepth_zero, 4 * (size_t) nP);
    const size_t ul_begin = same_topology ? L.topo_end : 0;
    CUDA_CHECK_RET(c, cudaMemcpyAsync(c->arena_dev + ul_begin, H + ul_begin, L.ul_end - ul_begin, cudaMemcpyHostToDevice, c->stream));
    if (!c->window_copied) CUDA_CHECK_RET(c, cudaEventCreateWithFlags(&c->window_copied, cudaEventDisableTiming));
    CUDA_CHECK_RET(c, cudaEventRecord(c->window_copied, c->stream));
    CUDA_CHECK_RET(c, cudaMemsetAsync(c->arena_dev + L.ul_end, 0, L.total - L.ul_end, c->stream));    // all result/state arrays
    if (win->res_toZeroF && nR > 0) CUDA_CHECK_RET(c, cudaMemcpyAsync(d.res_toZero, win->res_toZeroF, 32 * (size_t) nR, cudaMemcpyHostToDevice, c->stream));
    if (!same_topology) CUDA_CHECK_RET(c, cudaMemsetAsync(d.res_J, 0, sizeof(float) * 74 * (size_t) std::max(nR, 1), c->stream));
    if (win->res_toZeroF) CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));   // pageable source
    invalidate_results(c);
    c->solve_ready = false; c->restitch_ok = false;
    c->have_window = true;
    return LDSO_B200_OK;
}

int build_derived(ldso_b200_ctx *c) {
    if (!c->have_window || !c->have_frames) return c->fail(LDSO_B200_ERR_STATE, "set_frames and set_window must both be called first");
    if (!c->derived_dirty) return LDSO_B200_OK;
    DevWindow &d = c->d;
    const int nP = d.nP, nR = d.nR, nF = c->nF;
    for (int p = 0; p < nP; p++) if (c->h_pt_host[p] >= nF) return c->fail(LDSO_B200_ERR_ARG, "pt_host >= nFrames");
    for (int r = 0; r < nR; r++) if (c->h_res_target[r] >= nF) return c->fail(LDSO_B200_ERR_ARG, "res_target >= nFrames");
    // two co-resident CTAs per SM hide each other's phase latencies (K1 is a chain of short, barrier-separated phases)
    // ... and large windows are cut into whole waves of 2*SMs items (at most 64 points each: the records of an item live in
    // shared memory), so that the last wave is as full as the first
    const int slots = 2 * std::max(c->sm_count, 1);
    const int waves = std::max(1, (nP + 64 * slots - 1) / (64 * slots));
    const int target_items = waves * slots;
    int ppi = (nP + target_items - 1) / target_items;
    ppi = std::max(4, std::min(64, ppi));
    d.pts_per_item = ppi;
    c->k1_smem = k1_smem_bytes(ppi);
    std::vector<int4> items;
    std::vector<int> hib(MAXF + 1, 0);
    int p = 0;
    for (int h = 0; h < MAXF; h++) {
        hib[h] = (int) items.size();
        while (p < nP && c->h_pt_host[p] == h) {
            int e = p;
            while (e < nP && c->h_pt_host[e] == h && e - p < ppi) e++;
            items.push_back(make_int4(h, p, e, 0));
            p = e;
        }
    }
    hib[MAXF] = (int) items.size();
    d.nItems = (int) items.size();
    std::vector<int> slot(nR, -1);
    int ns = 0;
    for (int r = 0; r < nR; r++) if (c->h_res_target[r] == nF - 1) slot[r] = ns++;
    const int local_newest = ns;
    if (d.newest_total < 0 || !c->multi) { d.newest_total = local_newest; d.newest_offset = 0; }
    for (int r = 0; r < nR; r++) if (slot[r] >= 0) slot[r] += d.newest_offset;

    int4 *items_dev; int *hib_dev, *slot_dev;
    int rc = 0;
    // the previous derived buffers (same window, other nF / shard description) may still be read by queued kernels
    if (!c->derived_allocs.empty()) { CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream)); free_derived(c); }
    std::vector<void *> *own = &c->derived_allocs;
    rc |= dev_alloc(c, &items_dev, items.size(), own); rc |= dev_alloc(c, &hib_dev, MAXF + 1, own); rc |= dev_alloc(c, &slot_dev, nR, own);
    rc |= dev_alloc(c, &d.partials, (size_t) std::max(d.nItems, 1) * PART_STRIDE, own);
    rc |= dev_alloc(c, &d.item_stats, (size_t) std::max(d.nItems, 1) * 4, own);
    rc |= dev_alloc(c, &d.red, (size_t) RED_SELECT + std::max(d.newest_total, 1) + 16, own);
    rc |= dev_alloc(c, &d.dbg, 32 + 3 * (size_t) std::max(d.nItems, 1), own);
    if (rc) return LDSO_B200_ERR_CUDA;
    rc |= h2d(c, items_dev, items.data(), sizeof(int4) * items.size());
    rc |= h2d(c, hib_dev, hib.data(), sizeof(int) * (MAXF + 1));
    rc |= h2d(c, slot_dev, slot.data(), sizeof(int) * nR);
    if (rc) return LDSO_B200_ERR_CUDA;
    CUDA_CHECK_RET(c, cudaMemsetAsync(d.red, 0, sizeof(double) * ((size_t) RED_SELECT + std::max(d.newest_total, 1) + 16), c->stream));
    CUDA_CHECK_RET(c, cudaMemsetAsync(d.partials, 0, sizeof(float) * (size_t) std::max(d.nItems, 1) * PART_STRIDE, c->stream));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    if (c->peer.connected && c->peer.px.n_doubles != RED_SELECT + std::max(d.newest_total, 0))
        return c->fail(LDSO_B200_ERR_STATE, "the window's newest-frame residual count changed: the peer exchange buffers must be re-exported");
    d.items = items_dev; d.host_item_begin = hib_dev; d.res_newest_slot = slot_dev;
    c->derived_dirty = false;
    c->gn_graph_valid = false;
    return LDSO_B200_OK;
}

// ---------------------------------------------------------------------------------------------- frames
static int clear_prior(ldso_b200_ctx *c, int n) {
    CUDA_CHECK_RET(c, cudaMemsetAsync(c->sb.HM, 0, sizeof(double) * n * n, c->stream));
    CUDA_CHECK_RET(c, cudaMemsetAsync(c->sb.bM, 0, sizeof(double) * n, c->stream));
    return LDSO_B200_OK;
}
extern "C" int ldso_b200_set_frames(ldso_b200_ctx *c, int nFrames, const ldso_b200_frame_state *frames,
                                    const double calib_value_scaled[4], const double calib_value_zero[4]) {
    if (!c || !frames || !calib_value_scaled || !calib_value_zero) return LDSO_B200_ERR_ARG;
    if (nFrames < 1 || nFrames > MAXF) return c->fail(LDSO_B200_ERR_ARG, "nFrames must be in [1, LDSO_B200_MAX_FRAMES]");
    cudaSetDevice(c->device);
    // ws_host (pinned) may still be the source of the previous call's upload: wait for that copy only (not for the
    // kernels queued behind it), so that back-to-back calls overlap host packing with device work
    CUDA_CHECK_RET(c, cudaEventSynchronize(c->frames_copied));
    using namespace hostmath;
    WinState &W = *c->ws_host;
    // the adjoints and the null-space projector depend only on the evaluation points (worldToCam_evalPT, state_zero's
    // affine part, exposures): they change once per keyframe, so they are recomputed only when those inputs change
    std::vector<double> key;
    key.reserve((size_t) nFrames * 16 + 1);
    key.push_back((double) nFrames);
    for (int i = 0; i < nFrames; i++) {
        key.insert(key.end(), frames[i].evalR, frames[i].evalR + 9);
        key.insert(key.end(), frames[i].evalT, frames[i].evalT + 3);
        key.push_back(frames[i].state_zero[6]); key.push_back(frames[i].state_zero[7]); key.push_back(frames[i].ab_exposure);
    }
    const bool evalpt_cached = c->have_frames && key == c->evalpt_key;
    if (evalpt_cached) {
        // keep adHost/adTarget(/F) of the previous call; everything else is rewritten below
        memset(&W, 0, offsetof(WinState, adHost));
        memset((char *) &W + offsetof(WinState, cPrior), 0, sizeof(WinState) - offsetof(WinState, cPrior));
    } else {
        memset(&W, 0, sizeof(W));
    }
    const int nF = nFrames, n = 8 * nF + CPARS;
    const int prev_nF = c->have_frames ? c->nF : -1;
    W.nF = nF; W.n = n; W.w = c->w; W.h = c->h;
    W.wM3G = (float) (c->w - 3); W.hM3G = (float) (c->h - 3);      // GlobalCalib.cc:42-43
    W.S = c->S;
    std::vector<Pose> ev(nF);
    for (int i = 0; i < nF; i++) {
        const ldso_b200_frame_state &f = frames[i];
        if (f.image_slot < 0 || f.image_slot >= NSLOTS || !c->img[f.image_slot][0]) return c->fail(LDSO_B200_ERR_ARG, "frame image slot not uploaded");
        FrameDev &D = W.fr[i];
        memcpy(D.evalR, f.evalR, sizeof(D.evalR)); memcpy(D.evalT, f.evalT, sizeof(D.evalT));
        memcpy(D.state, f.state, sizeof(D.state)); memcpy(D.state_zero, f.state_zero, sizeof(D.state_zero));
        memcpy(D.state_backup, f.state, sizeof(D.state));
        D.frameEnergyTH = f.frameEnergyTH; W.frameEnergyTH[i] = f.frameEnergyTH; D.ab_exposure = f.ab_exposure; D.frame_id = f.frame_id; D.slot = f.image_slot;
        // FrameHessian::getPrior (FrameHessian.h:125-150), takeData (FrameHessian.cc:108-112)
        double p[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (f.frame_id == 0) {
            p[0] = p[1] = p[2] = c->S.initialTransPrior;
            p[3] = p[4] = p[5] = c->S.initialRotPrior;
            p[6] = c->S.initialAffAPrior;
            p[7] = c->S.initialAffBPrior;
        } else {
            p[6] = (c->S.affineOptModeA < 0) ? c->S.initialAffAPrior : c->S.affineOptModeA;
            p[7] = (c->S.affineOptModeB < 0) ? c->S.initialAffBPrior : c->S.affineOptModeB;
        }
        for (int k = 0; k < 8; k++) D.prior[k] = p[k];
        memcpy(ev[i].R, f.evalR, sizeof(ev[i].R)); memcpy(ev[i].t, f.evalT, sizeof(ev[i].t));
        W.img0[i] = c->img[f.image_slot][0];
        c->slots[i] = f.image_slot;
    }
    // calibration (CalibHessian::setValueScaled, CalibHessian.h:87-100)
    CalibDev &C = W.calib;
    for (int i = 0; i < 4; i++) { C.value_scaled[i] = calib_value_scaled[i]; C.value_zero[i] = calib_value_zero[i]; }
    C.value[0] = (double) (1.0f / SCALE_F) * C.value_scaled[0]; C.value[1] = (double) (1.0f / SCALE_F) * C.value_scaled[1];
    C.value[2] = (double) (1.0f / SCALE_C) * C.value_scaled[2]; C.value[3] = (double) (1.0f / SCALE_C) * C.value_scaled[3];
    for (int i = 0; i < 4; i++) C.value_backup[i] = C.value[i];
    C.fxl = (float) C.value_scaled[0]; C.fyl = (float) C.value_scaled[1]; C.cxl = (float) C.value_scaled[2]; C.cyl = (float) C.value_scaled[3];
    C.fxli = 1.0f / C.fxl; C.fyli = 1.0f / C.fyl; C.cxli = -C.cxl / C.fxl; C.cyli = -C.cyl / C.fyl;
    for (int i = 0; i < 4; i++) { C.cDeltaF[i] = (float) (C.value[i] - C.value_zero[i]); W.cPrior[i] = c->S.initialCalibHessian; }

    // EnergyFunctional::setAdjointsF (EnergyFunctional.cc:431-489)
    if (!evalpt_cached)
    for (int h = 0; h < nF; h++)
        for (int t = 0; t < nF; t++) {
            Pose hostToTarget = mul(ev[t], inv(ev[h]));
            double Adj[36];
            adjoint(hostToTarget, Adj);
            double *AH = W.adHost[h + nF * t], *AT = W.adTarget[h + nF * t];
            for (int i = 0; i < 8; i++) AH[i * 8 + i] = AT[i * 8 + i] = 1.0;
            for (int i = 0; i < 6; i++) for (int j = 0; j < 6; j++) AH[i * 8 + j] = -Adj[j * 6 + i];
            float eF = frames[h].ab_exposure, eT = frames[t].ab_exposure;
            if (eF == 0 || eT == 0) eT = eF = 1;
            const float a0h = (float) (frames[h].state_zero[6] * SCALE_A), a0t = (float) (frames[t].state_zero[6] * SCALE_A);
            const float affLL0 = expf(a0t - a0h) * eT / eF;
            AT[6 * 8 + 6] = -affLL0; AH[6 * 8 + 6] = affLL0; AT[7 * 8 + 7] = -1; AH[7 * 8 + 7] = affLL0;
            for (int j = 0; j < 8; j++) {
                for (int i = 0; i < 3; i++) { AH[i * 8 + j] *= SCALE_XI_TRANS; AT[i * 8 + j] *= SCALE_XI_TRANS; }
                for (int i = 3; i < 6; i++) { AH[i * 8 + j] *= SCALE_XI_ROT; AT[i * 8 + j] *= SCALE_XI_ROT; }
                AH[6 * 8 + j] *= SCALE_A; AT[6 * 8 + j] *= SCALE_A;
                AH[7 * 8 + j] *= SCALE_B; AT[7 * 8 + j] *= SCALE_B;
            }
            for (int i = 0; i < 64; i++) { W.adHostF[h + nF * t][i] = (float) AH[i]; W.adTargetF[h + nF * t][i] = (float) AT[i]; }
        }

    // null spaces (FrameHessian::setStateZero, FrameHessian.cc:11-42; FullSystem::getNullspaces, FullSystem.cc:1711-1760)
    // and the projector EnergyFunctional::orthogonalize applies (pose + scale, EnergyFunctional.cc:687-716)
    std::vector<double> N((size_t) n * 7, 0.0);
    if (!evalpt_cached) {
    for (int f = 0; f < nF; f++) {
        const Pose evI = inv(ev[f]);
        for (int i = 0; i < 6; i++) {
            double e[6] = {0, 0, 0, 0, 0, 0}, m[6] = {0, 0, 0, 0, 0, 0};
            e[i] = 1e-3; m[i] = -1e-3;
            double lp[6], lm[6];
            logm(mul(mul(ev[f], expm(e)), evI), lp);
            logm(mul(mul(ev[f], expm(m)), evI), lm);
            for (int r = 0; r < 6; r++) {
                double v = (lp[r] - lm[r]) / 2e-3;
                v *= (r < 3) ? (double) (1.0f / SCALE_XI_TRANS) : (double) (1.0f / SCALE_XI_ROT);
                N[(size_t) i * n + CPARS + 8 * f + r] = v;
            }
        }
        Pose P = ev[f], M = ev[f];
        for (int k = 0; k < 3; k++) { P.t[k] *= 1.00001; M.t[k] /= 1.00001; }
        double lp[6], lm[6];
        logm(mul(P, evI), lp);
        logm(mul(M, evI), lm);
        for (int r = 0; r < 6; r++) {
            double v = (lp[r] - lm[r]) / 2e-3;
            v *= (r < 3) ? (double) (1.0f / SCALE_XI_TRANS) : (double) (1.0f / SCALE_XI_ROT);
            N[(size_t) 6 * n + CPARS + 8 * f + r] = v;
        }
    }
    for (int j = 0; j < 7; j++) {   // N.col(i) = ns[i].normalized()
        double s = 0;
        for (int r = 0; r < n; r++) s += N[(size_t) j * n + r] * N[(size_t) j * n + r];
        s = sqrt(s);
        if (s > 0) for (int r = 0; r < n; r++) N[(size_t) j * n + r] /= s;
    }
    range_projector(N, n, 7, c->S.solverModeDelta, c->Pns_host);
    c->evalpt_key = key;
    }

    c->nF = nF; c->n = n;
    CUDA_CHECK_RET(c, cudaMemcpyAsync(c->ws_dev, c->ws_host, sizeof(WinState), cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK_RET(c, cudaEventRecord(c->frames_copied, c->stream));
    if (!evalpt_cached)     // pageable source: staged before the call returns
        CUDA_CHECK_RET(c, cudaMemcpyAsync(c->sb.Pns, c->Pns_host.data(), sizeof(double) * n * n, cudaMemcpyHostToDevice, c->stream));
    if (c->prior_dim == n) {
        // same frames as the prior describes (a repeated set_frames, or the window after marginalize_frame + insertFrame)
    } else if (c->prior_dim > 0 && c->prior_dim == n - 8) {
        // one keyframe appended since the prior was last touched: EnergyFunctional::insertFrame (EnergyFunctional.cc:38-44)
        CUDA_CHECK_RET(c, cudaMemcpyAsync(c->sb.A0g, c->sb.HM, sizeof(double) * (n - 8) * (n - 8), cudaMemcpyDeviceToDevice, c->stream));
        k_grow_prior<<<(n * n + 255) / 256, 256, 0, c->stream>>>(c->sb, c->sb.A0g, n);
        LAUNCH_CHECK(c);
        c->prior_dim = n;
    } else {
        RET_IF(clear_prior(c, n));
        c->prior_dim = 0;
    }
    k_frames_refresh<<<1, 128, 0, c->stream>>>(c->ws_dev);
    LAUNCH_CHECK(c);
    c->solve_ready = false; c->restitch_ok = false; c->select_pending = false;
    c->have_frames = true;
    if (prev_nF != nF) c->derived_dirty = true;    // work items / newest-frame slots depend on nF only
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_set_marg_prior(ldso_b200_ctx *c, const double *HM, const double *bM) {
    if (!c || !c->have_frames) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    const int n = c->n;
    if (HM) CUDA_CHECK_RET(c, cudaMemcpyAsync(c->sb.HM, HM, sizeof(double) * n * n, cudaMemcpyHostToDevice, c->stream));
    else CUDA_CHECK_RET(c, cudaMemsetAsync(c->sb.HM, 0, sizeof(double) * n * n, c->stream));
    if (bM) CUDA_CHECK_RET(c, cudaMemcpyAsync(c->sb.bM, bM, sizeof(double) * n, cudaMemcpyHostToDevice, c->stream));
    else CUDA_CHECK_RET(c, cudaMemsetAsync(c->sb.bM, 0, sizeof(double) * n, c->stream));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    c->solve_ready = false;      // HM/bM enter the assembled system
    c->prior_dim = (HM || bM) ? n : 0;
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_get_marg_prior(ldso_b200_ctx *c, double *HM, double *bM) {
    if (!c || !c->have_frames) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    const int n = (c->prior_dim > 0) ? c->prior_dim : c->n;      // n - 8 between marginalize_frame and the next set_frames
    RET_IF(d2h(c, HM, c->sb.HM, sizeof(double) * n * n));
    RET_IF(d2h(c, bM, c->sb.bM, sizeof(double) * n));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

// ---------------------------------------------------------------------------------------------- launches
// One launch path for the loop kernels: inside launch_gn_body the kernel is allowed to start (and run its constant-data
// prologue up to pdl_wait()) while its predecessor on the stream is still executing. name: its LDSO_B200_KTIME timer.
template<typename... KArgs, typename... Args>
static int launch_loop_kernel(ldso_b200_ctx *c, const char *name, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args... args) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = c->stream;
    cudaLaunchAttribute at[1];
    memset(at, 0, sizeof(at));
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = (c->pdl_now && c->use_pdl && !c->ktime) ? 1 : 0;
    c->kt_begin(name);
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
    c->kt_end();
    LAUNCH_CHECK(c);
    return LDSO_B200_OK;
}

static int launch_k1(ldso_b200_ctx *c, int flags, const uint8_t *sel = nullptr) {
    if (c->d.nItems == 0) return LDSO_B200_OK;
    return launch_loop_kernel(c, "k1", k1_linearize_accumulate, dim3(c->d.nItems), dim3(K1_THREADS), c->k1_smem, c->d, (const WinState *) c->ws_dev,
                              flags, sel);
}
static int launch_k2a(ldso_b200_ctx *c, int full) {
    const int nb = (MAXF * PART_USED + 63) / 64 + 1;
    RET_IF(launch_loop_kernel(c, "k2a", k2a_reduce, dim3(nb), dim3(K2A_THREADS), 0, c->d, c->ws_dev, full, c->multi ? 1 : 0));
    if (full) { c->restitch_ok = true; c->solve_ready = false; }
    return LDSO_B200_OK;
}
static int launch_k2b(ldso_b200_ctx *c, int do_stitch, int do_select, int do_assemble) {
    if (do_stitch && do_assemble && c->prior_dim != 0 && c->prior_dim != c->n)
        return c->fail(LDSO_B200_ERR_STATE, "the marginalisation prior has a different dimension than the frames (marginalize_frame): call set_frames with the remaining frames first");
    const int nb = c->nF * c->nF + c->nF + 2;
    DevWindow dw = c->d;
    if (c->peer.connected) dw.red = c->peer.red_sum;      // the stitch reads the all-reduced accumulators
    RET_IF(launch_loop_kernel(c, "k2b", k2b_stitch, dim3(nb), dim3(K2B_THREADS), K2B_SMEM_BYTES, dw, c->ws_dev, c->sb, do_stitch, do_select,
                              (int) (do_stitch && do_assemble)));
    if (do_stitch) c->solve_ready = do_assemble != 0;
    if (do_select) c->select_pending = false;
    return LDSO_B200_OK;
}
static int launch_k2r(ldso_b200_ctx *c) {
    return launch_loop_kernel(c, "k2r", k2r_peer_allreduce, dim3(c->peer.px.n_chunks), dim3(K2R_THREADS), 0, c->d, c->peer.px);
}
// K3(SOLVE) consumes what K2b(do_assemble) left behind; re-stitch if only the prior changed in between
static int ensure_solve_ready(ldso_b200_ctx *c) {
    if (c->solve_ready) return LDSO_B200_OK;
    if (!c->restitch_ok) return c->fail(LDSO_B200_ERR_STATE, "no stitched system for the current window state: call optimize_begin / solve_system first");
    return launch_k2b(c, 1, 0, 1);
}
static int launch_k3(ldso_b200_ctx *c, int flags) {
    const double *sel_red = c->peer.connected ? c->peer.red_sum : c->d.red;
    return launch_loop_kernel(c, "k3", k3_solve_step, dim3((flags & K3F_SELECT) ? 2 : 1), dim3(K3_THREADS), K3_SMEM_BYTES, c->ws_dev, c->sb, flags,
                              c->iteration_dev, sel_red, std::max(c->d.newest_total, 0), c->d.dbg);
}
static int read_energy(ldso_b200_ctx *c, double *energy_out) {
    if (!energy_out) return LDSO_B200_OK;
    RET_IF(d2h(c, energy_out, &c->ws_dev->energy, sizeof(double)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}
static int set_iteration(ldso_b200_ctx *c, int it) {
    CUDA_CHECK_RET(c, cudaMemcpyAsync(c->iteration_dev, &it, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    return LDSO_B200_OK;
}
static int clear_select(ldso_b200_ctx *c) {   // multi-GPU: slots owned by other ranks must be zero before the all-reduce
    if (c->multi && c->d.newest_total > 0)
        CUDA_CHECK_RET(c, cudaMemsetAsync(c->d.red + RED_SELECT, 0, sizeof(double) * c->d.newest_total, c->stream));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_linearize_all(ldso_b200_ctx *c, int fixLinearization, int flags, double *energy_out) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    (void) flags;   // the piecewise path always keeps the full Jacobian: solve_system rebuilds its records from it
    RET_IF(flush_select(c));
    int f = K1F_LINEARIZE | K1F_STORE_J;
    if (fixLinearization) f |= K1F_APPLY_RES;
    RET_IF(clear_select(c));
    RET_IF(launch_k1(c, f));
    RET_IF(launch_k2a(c, 0));
    RET_IF(launch_k2b(c, 0, 1, 0));
    return read_energy(c, energy_out);
}

extern "C" int ldso_b200_apply_res(ldso_b200_ctx *c) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    if (c->d.nR > 0) {
        k_apply_res<<<(c->d.nR + 255) / 256, 256, 0, c->stream>>>(c->d);
        LAUNCH_CHECK(c);
    }
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_backup_state(ldso_b200_ctx *c) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    RET_IF(launch_k3(c, K3F_BACKUP));
    if (c->d.nP > 0) {
        k_points<<<(c->d.nP + 255) / 256, 256, 0, c->stream>>>(c->d, c->ws_dev, 1);
        LAUNCH_CHECK(c);
    }
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_solve_system(ldso_b200_ctx *c, int iteration, double *lastHS, double *lastbS, double *lastX) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    // records from the stored Jacobians: accumulateAF (mode 0); with linearized residuals in the window, accumulateLF's terms
    // (mode 1: res_toZeroF + J delta) ride in the same pass -- solveSystemF only ever uses HA + HL and the summed point terms
    RET_IF(launch_k1(c, K1F_ACCUMULATE | ((c->has_lin ? 3 : 0) << K1F_MODE_SHIFT)));
    RET_IF(launch_k2a(c, 1));
    RET_IF(launch_k2b(c, 1, 0, 1));
    RET_IF(set_iteration(c, iteration));
    RET_IF(launch_k3(c, K3F_SOLVE));
    if (c->d.nP > 0) {
        k_points<<<(c->d.nP + 255) / 256, 256, 0, c->stream>>>(c->d, c->ws_dev, 2);
        LAUNCH_CHECK(c);
    }
    return ldso_b200_get_last_solution(c, lastHS, lastbS, lastX);
}

// pt_sel_dev[p] = 1 for the n points listed in idx, 0 for the others
static int upload_point_selection(ldso_b200_ctx *c, int n, const int32_t *idx) {
    std::vector<uint8_t> sel(std::max(c->d.nP, 1), 0);
    for (int i = 0; i < n; i++) {
        if (idx[i] < 0 || idx[i] >= c->d.nP) return c->fail(LDSO_B200_ERR_ARG, "point index out of range");
        sel[idx[i]] = 1;
    }
    CUDA_CHECK_RET(c, cudaMemcpyAsync(c->pt_sel_dev, sel.data(), c->d.nP, cudaMemcpyHostToDevice, c->stream));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

// AccumulatedTopHessianSSE::addPoint<mode> over a set of points + stitchDouble, and AccumulatedSCHessianSSE::addPoint + stitchDouble
// on the same set (AccumulatedTopHessian.cc:9-118,129-255; AccumulatedSCHessian.cc:9-119): what EnergyFunctional::accumulateAF_MT /
// accumulateLF_MT / accumulateSCF_MT and marginalizePointsF call. Records are rebuilt from the stored Jacobians (linearize_all).
// mode 0/1/2 as the reference's template argument, 3 = modes 0 and 1 in one pass. point_idx == NULL: all points. H, b WITHOUT the
// frame / calibration priors (stitchDouble(usePrior = false)); the caller adds them where the reference passes usePrior = true.
extern "C" int ldso_b200_accumulate(ldso_b200_ctx *c, int mode, int n_points, const int32_t *point_idx, int shift_prior_to_zero,
                                    double *H_top, double *b_top, double *H_sc, double *b_sc, int *nres) {
    if (!c || mode < 0 || mode > 3 || n_points < 0) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    const uint8_t *sel = nullptr;
    if (point_idx) {
        RET_IF(upload_point_selection(c, n_points, point_idx));
        sel = c->pt_sel_dev;
    }
    RET_IF(launch_k1(c, K1F_ACCUMULATE | (shift_prior_to_zero ? 0 : K1F_NO_SHIFT_PRIOR) | (mode << K1F_MODE_SHIFT), sel));
    RET_IF(launch_k2a(c, 1));
    RET_IF(launch_k2b(c, 1, 0, 0));
    c->restitch_ok = false;      // the reduced buffer describes this call's selection / mode, not the window's system
    return ldso_b200_get_system(c, H_top, b_top, H_sc, b_sc, nres);
}

extern "C" int ldso_b200_get_last_solution(ldso_b200_ctx *c, double *lastHS, double *lastbS, double *lastX) {
    if (!c || !c->have_frames) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    const int n = c->n;
    // one copy of [lastHS | lastbS | lastX] into pinned staging memory, then plain memcpy into the caller's buffers
    const size_t nn = (size_t) MAXN * MAXN;
    RET_IF(wait_results(c));
    if (!c->sol_valid) {
        RET_IF(d2h(c, c->sol_host, c->sb.lastHS, sizeof(double) * (nn + 2 * MAXN)));
        CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
        c->sol_valid = true;
    }
    if (lastHS) memcpy(lastHS, c->sol_host, sizeof(double) * n * n);
    if (lastbS) memcpy(lastbS, c->sol_host + nn, sizeof(double) * n);
    if (lastX) memcpy(lastX, c->sol_host + nn + MAXN, sizeof(double) * n);
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_get_system(ldso_b200_ctx *c, double *H_A, double *b_A, double *H_sc, double *b_sc, int *resInA) {
    if (!c || !c->have_frames) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    const int n = c->n;
    RET_IF(d2h(c, H_A, c->sb.H_A, sizeof(double) * n * n));
    RET_IF(d2h(c, b_A, c->sb.b_A, sizeof(double) * n));
    RET_IF(d2h(c, H_sc, c->sb.H_sc, sizeof(double) * n * n));
    RET_IF(d2h(c, b_sc, c->sb.b_sc, sizeof(double) * n));
    RET_IF(d2h(c, resInA, &c->ws_dev->resInA, sizeof(int)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_do_step(ldso_b200_ctx *c, int *canbreak) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    k_sum_nid<<<1, 256, 0, c->stream>>>(c->d, c->ws_dev);
    LAUNCH_CHECK(c);
    RET_IF(launch_k3(c, K3F_STEP));
    if (c->d.nP > 0) {
        k_points<<<(c->d.nP + 255) / 256, 256, 0, c->stream>>>(c->d, c->ws_dev, 4);
        LAUNCH_CHECK(c);
    }
    if (canbreak) {
        RET_IF(d2h(c, canbreak, &c->ws_dev->canbreak, sizeof(int)));
        CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    }
    return LDSO_B200_OK;
}

// FullSystem::flagPointsForRemoval's re-linearisation of the points to marginalise (FullSystem.cc:1241-1249:
// resetOOB, linearize, applyRes(true), fixLinearizationF) followed by EnergyFunctional::marginalizePointsF
// (EnergyFunctional.cc:165-222): priorF *= prior_fac, addPoint<2> + SC addPoint(p, false), stitchDouble without priors,
// HM += margWeightFac (M - Msc), bM likewise. The caller then drops the points from its window.
extern "C" int ldso_b200_marginalize_points(ldso_b200_ctx *c, int n, const int32_t *point_idx, float prior_fac, int *resInM) {
    if (!c || n < 0 || (n > 0 && !point_idx)) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    RET_IF(upload_point_selection(c, n, point_idx));
    RET_IF(flush_select(c));
    RET_IF(launch_k1(c, K1F_LINEARIZE | K1F_STORE_J | K1F_APPLY_RES | K1F_RESET_OOB, c->pt_sel_dev));
    if (c->d.nR > 0) {
        k_fix_linearization<<<(c->d.nR + 255) / 256, 256, 0, c->stream>>>(c->d, c->ws_dev, c->pt_sel_dev);
        LAUNCH_CHECK(c);
        k_scale_prior<<<(c->d.nP + 255) / 256, 256, 0, c->stream>>>(c->d, c->pt_sel_dev, prior_fac);
        LAUNCH_CHECK(c);
    }
    c->has_lin = c->has_lin || n > 0;
    RET_IF(launch_k1(c, K1F_ACCUMULATE | K1F_NO_SHIFT_PRIOR | (2 << K1F_MODE_SHIFT), c->pt_sel_dev));
    RET_IF(launch_k2a(c, 1));
    RET_IF(launch_k2b(c, 1, 0, 0));
    c->restitch_ok = false;      // the reduced buffer now holds the mode-2 (marginalisation) accumulators
    c->prior_dim = c->n;
    const int nn = c->n;
    k_add_marg<<<(nn * nn + 255) / 256, 256, 0, c->stream>>>(c->sb, nn, (double) c->S.margWeightFac);
    LAUNCH_CHECK(c);
    if (resInM) {
        RET_IF(d2h(c, resInM, &c->ws_dev->resInA, sizeof(int)));
        CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    }
    return LDSO_B200_OK;
}

// EnergyFunctional::calcLEnergyF_MT / calcMEnergyF (EnergyFunctional.cc:353-378): the prior + linearised-residual energy and the
// marginalisation energy at the current state (FullSystem::optimize reads both around every step, FullSystem.cc:1697-1703).
extern "C" int ldso_b200_calc_energies(ldso_b200_ctx *c, double *energyL, double *energyM) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    if (c->prior_dim != 0 && c->prior_dim != c->n) return c->fail(LDSO_B200_ERR_STATE, "prior dimension does not match the frames: call set_frames first");
    const int nb = std::max(1, (c->d.nP + KEN_THREADS - 1) / KEN_THREADS);
    Arena A;
    const size_t o_part = A.take(sizeof(double) * nb), o_out = A.take(sizeof(double) * 2), o_cnt = A.take(sizeof(unsigned));
    RET_IF(reserve_scratch(c, A.off));
    double *part = (double *) (c->scr.buf + o_part), *out = (double *) (c->scr.buf + o_out);
    unsigned *counter = (unsigned *) (c->scr.buf + o_cnt);
    CUDA_CHECK_RET(c, cudaMemsetAsync(counter, 0, sizeof(unsigned), c->stream));
    k_calc_energies<<<nb, KEN_THREADS, 0, c->stream>>>(c->d, c->ws_dev, c->sb, part, counter, out);
    LAUNCH_CHECK(c);
    double h[2];
    RET_IF(d2h(c, h, out, sizeof(h)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    if (energyL) *energyL = h[0];
    if (energyM) *energyM = h[1];
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_marginalize_frame(ldso_b200_ctx *c, int frame_idx, int *new_dim) {
    if (!c || !c->have_frames) return LDSO_B200_ERR_STATE;
    if (frame_idx < 0 || frame_idx >= c->nF) return c->fail(LDSO_B200_ERR_ARG, "frame index out of range");
    if (c->nF < 2) return c->fail(LDSO_B200_ERR_STATE, "cannot marginalise the only frame");
    if (c->prior_dim != 0 && c->prior_dim != c->n) return c->fail(LDSO_B200_ERR_STATE, "prior dimension does not match the frames: call set_frames first");
    cudaSetDevice(c->device);
    const int n = c->n;
    if (c->prior_dim == 0) RET_IF(clear_prior(c, n));     // an all-zero prior of the current dimension
    k_marginalize_frame<<<1, KMF_THREADS, KMF_SMEM_BYTES(n), c->stream>>>(c->sb, c->ws_dev, n, frame_idx);
    LAUNCH_CHECK(c);
    c->prior_dim = n - 8;
    c->solve_ready = false; c->restitch_ok = false;
    if (new_dim) *new_dim = n - 8;
    return LDSO_B200_OK;
}

// ---------------------------------------------------------------------------------------------- fused loop
static const int K1_FUSED = K1F_LINEARIZE | K1F_ACCUMULATE | K1F_APPLY_RES;

extern "C" int ldso_b200_optimize_begin(ldso_b200_ctx *c, double *energy_out) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    RET_IF(clear_select(c));
    RET_IF(launch_k1(c, K1_FUSED | K1F_RESET_OOB));
    RET_IF(launch_k2a(c, 1));
    if (c->multi && !c->peer.connected) return LDSO_B200_OK;     // caller all-reduces, then gn_phase_b
    if (c->peer.connected) RET_IF(launch_k2r(c));
    RET_IF(launch_k2b(c, 1, 1, 1));
    return read_energy(c, energy_out);
}

// One fused Gauss-Newton iteration: K3 (solve + step, and -- second CTA -- the energy-threshold select of the PREVIOUS linearisation)
// -> K1 -> K2a -> [K2r] -> K2b (stitch + assemble). The select of the linearisation this body ends with stays pending: the next
// body's K3 runs it, or flush_select() when something else needs the threshold first.
static int launch_gn_body(ldso_b200_ctx *c) {
    struct Scope { ldso_b200_ctx *c; Scope(ldso_b200_ctx *c_) : c(c_) { c->pdl_now = true; } ~Scope() { c->pdl_now = false; } } scope(c);
    RET_IF(launch_k3(c, K3F_BACKUP | K3F_SOLVE | K3F_STEP | K3F_SELECT));
    RET_IF(launch_k1(c, K1_FUSED | K1F_APPLY_STEP));
    RET_IF(launch_k2a(c, 1));
    if (c->peer.connected) RET_IF(launch_k2r(c));
    RET_IF(launch_k2b(c, 1, 0, 1));
    c->select_pending = true;
    return LDSO_B200_OK;
}
int flush_select(ldso_b200_ctx *c) {
    if (!c->select_pending) return LDSO_B200_OK;
    c->select_pending = false;
    const bool sr = c->solve_ready;
    RET_IF(launch_k2b(c, 0, 1, 0));
    c->solve_ready = sr;
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_gn_iterations(ldso_b200_ctx *c, int first_iteration, int n_iterations) {
    if (!c) return LDSO_B200_ERR_ARG;
    if (c->multi && !c->peer.connected) return c->fail(LDSO_B200_ERR_STATE, "sharded context without peer exchange: use gn_phase_a / all-reduce / gn_phase_b, or peer_export + peer_connect");
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    RET_IF(ensure_solve_ready(c));
    RET_IF(set_iteration(c, first_iteration));     // K3 reads the iteration number from device memory and increments it
    if (c->use_graph && c->d.nItems > 0) {
        if (!c->gn_graph_valid) {
            if (c->gn_graph) { cudaGraphExecDestroy(c->gn_graph); c->gn_graph = nullptr; }
            cudaGraph_t g = nullptr;
            if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
                // e.g. the legacy default stream cannot be captured: run the plain launches instead
                cudaGetLastError();
                c->use_graph = false;
                for (int i = 0; i < n_iterations; i++) RET_IF(launch_gn_body(c));
                return LDSO_B200_OK;
            }
            const long long l0 = c->launches;
            int rc = launch_gn_body(c);
            cudaError_t e = cudaStreamEndCapture(c->stream, &g);
            c->launches = l0;
            if (rc == 0 && e == cudaSuccess) {
                e = cudaGraphInstantiate(&c->gn_graph, g, 0);
                if (e != cudaSuccess) c->gn_graph = nullptr;
            }
            if (g) cudaGraphDestroy(g);
            if (rc || e != cudaSuccess) {
                cudaGetLastError();
                if (c->use_pdl) {        // programmatic edges not capturable here: same graph with full dependencies
                    c->use_pdl = false;
                    return ldso_b200_gn_iterations(c, first_iteration, n_iterations);
                }
                if (rc) return rc;
                return c->fail_cuda(e, "CUDA graph capture of the GN iteration", __FILE__, __LINE__);
            }
            c->gn_graph_valid = true;
        }
        for (int i = 0; i < n_iterations; i++) {
            CUDA_CHECK_RET(c, cudaGraphLaunch(c->gn_graph, c->stream));
            c->launches += c->peer.connected ? 5 : 4;
            c->select_pending = true;
            invalidate_results(c);
        }
        return LDSO_B200_OK;
    }
    for (int i = 0; i < n_iterations; i++) RET_IF(launch_gn_body(c));
    return LDSO_B200_OK;
}

// Queue one whole FullSystem::optimize (uploads, prologue, n iterations, result read-back into pinned staging) on the context's
// stream and return WITHOUT waiting. The caller's buffers (io->image, frames, window arrays) are consumed before this returns except
// io->image, which must stay valid until the matching _wait. Two contexts fed alternately overlap one window's uploads with the
// other's kernels (bench.py's pipelined end-to-end leg); a single context just splits the call at its only synchronisation point.
extern "C" int ldso_b200_optimize_from_host_submit(ldso_b200_ctx *c, const ldso_b200_fused_io *io) {
    if (!c || !io || !io->frames || !io->window || !io->calib_value_scaled || !io->calib_value_zero) return LDSO_B200_ERR_ARG;
    if (io->n_iterations < 0) return c->fail(LDSO_B200_ERR_ARG, "negative iteration count");
    // the image first: 1.2 MB over PCIe, in flight while the host packs the frame states and the window
    if (io->image) RET_IF(make_images_impl(c, io->image_slot, io->image, false));
    RET_IF(ldso_b200_set_frames(c, io->nFrames, io->frames, io->calib_value_scaled, io->calib_value_zero));
    RET_IF(ldso_b200_set_window(c, io->window));
    RET_IF(ldso_b200_optimize_begin(c, nullptr));
    if (io->n_iterations > 0) RET_IF(ldso_b200_gn_iterations(c, io->first_iteration, io->n_iterations));
    RET_IF(ldso_b200_prefetch_results(c));
    // the two scalars ride behind the prefetch into pinned staging (sol_host has MAXN spare doubles behind lastX)
    const size_t nn = (size_t) MAXN * MAXN;
    RET_IF(d2h(c, c->sol_host + nn + 2 * MAXN, &c->ws_dev->energy, sizeof(double)));
    RET_IF(d2h(c, c->sol_host + nn + 2 * MAXN + 1, &c->ws_dev->canbreak, sizeof(int)));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_optimize_from_host_wait(ldso_b200_ctx *c, const ldso_b200_fused_io *io) {
    if (!c || !io) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));       // one wait covers everything (and frees the caller's image buffer)
    const size_t nn = (size_t) MAXN * MAXN;
    if (io->energy) *io->energy = c->sol_host[nn + 2 * MAXN];
    if (io->canbreak) memcpy(io->canbreak, c->sol_host + nn + 2 * MAXN + 1, sizeof(int));
    if (io->lastHS || io->lastbS || io->lastX) RET_IF(ldso_b200_get_last_solution(c, io->lastHS, io->lastbS, io->lastX));
    if (io->pt_idepth || io->pt_step || io->pt_HdiF)
        RET_IF(ldso_b200_get_points(c, io->pt_idepth, nullptr, io->pt_step, io->pt_HdiF, nullptr, nullptr, nullptr, nullptr));
    if (io->res_state || io->res_new_state || io->res_energy)
        RET_IF(ldso_b200_get_residuals(c, io->res_state, io->res_new_state, io->res_energy, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_optimize_from_host(ldso_b200_ctx *c, const ldso_b200_fused_io *io) {
    RET_IF(ldso_b200_optimize_from_host_submit(c, io));
    return ldso_b200_optimize_from_host_wait(c, io);
}

extern "C" int ldso_b200_reduce_buffer(ldso_b200_ctx *c, void **buf_dev, size_t *n_doubles) {
    if (!c || !buf_dev || !n_doubles) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    *buf_dev = c->d.red;
    *n_doubles = (size_t) RED_SELECT + std::max(c->d.newest_total, 0);
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_set_shard(ldso_b200_ctx *c, int newest_slot_offset, int newest_total) {
    if (!c) return LDSO_B200_ERR_ARG;
    if (newest_slot_offset < 0 || newest_total < newest_slot_offset) return c->fail(LDSO_B200_ERR_ARG, "bad shard description");
    c->multi = true;
    c->d.newest_offset = newest_slot_offset;
    c->d.newest_total = newest_total;
    c->derived_dirty = true;
    return LDSO_B200_OK;
}

// ---- peer-memory exchange: export this rank's block, map the peers', then gn_iterations / optimize_begin run the whole
// sharded iteration on the device (K3 -> K1 -> K2a -> K2r -> K2b) with no NCCL call and no host round trip
extern "C" int ldso_b200_peer_export(ldso_b200_ctx *c, void *ipc_handle_64) {
    if (!c || !ipc_handle_64) return LDSO_B200_ERR_ARG;
    if (!c->multi) return c->fail(LDSO_B200_ERR_STATE, "peer_export needs set_shard first");
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    const int n = RED_SELECT + std::max(c->d.newest_total, 0);
    const int nch = (n + K2R_THREADS - 1) / K2R_THREADS;
    if (c->peer.connected || c->peer.local) return c->fail(LDSO_B200_ERR_STATE, "peer exchange already set up for this context");
    const size_t bytes = sizeof(uint4) * (2 * K2R_MAX_PEERS + 2) * (size_t) n;      // the inbox: [2 parities][8 senders][n] 16-byte slots + the all-gather region [2][n]
    CUDA_CHECK_RET(c, cudaMalloc(&c->peer.local, bytes));
    CUDA_CHECK_RET(c, cudaMalloc(&c->peer.words, sizeof(int) * 4));
    CUDA_CHECK_RET(c, cudaMalloc(&c->peer.red_sum, sizeof(double) * ((size_t) n + 16)));
    // cleared on the context's own (non-blocking) stream and completed before the handle is handed out: a peer's first push
    // and this rank's first exchange kernel must find zeroed tags
    CUDA_CHECK_RET(c, cudaMemsetAsync(c->peer.local, 0, bytes, c->stream));
    CUDA_CHECK_RET(c, cudaMemsetAsync(c->peer.words, 0, sizeof(int) * 4, c->stream));
    CUDA_CHECK_RET(c, cudaMemsetAsync(c->peer.red_sum, 0, sizeof(double) * ((size_t) n + 16), c->stream));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    memset(&c->peer.px, 0, sizeof(c->peer.px));
    c->peer.px.n_doubles = n; c->peer.px.n_chunks = nch;
    cudaIpcMemHandle_t h;
    CUDA_CHECK_RET(c, cudaIpcGetMemHandle(&h, c->peer.local));
    memcpy(ipc_handle_64, &h, 64);
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_peer_connect(ldso_b200_ctx *c, int rank, int world, const void *ipc_handles_64_each) {
    if (!c || !ipc_handles_64_each) return LDSO_B200_ERR_ARG;
    if (!c->peer.local) return c->fail(LDSO_B200_ERR_STATE, "peer_connect needs peer_export first");
    if (world < 1 || world > K2R_MAX_PEERS || rank < 0 || rank >= world) return c->fail(LDSO_B200_ERR_ARG, "rank/world out of range (max 8 peers)");
    cudaSetDevice(c->device);
    for (int r = 0; r < world; r++) {
        char *base = c->peer.local;
        if (r != rank) {
            cudaIpcMemHandle_t h;
            memcpy(&h, (const char *) ipc_handles_64_each + 64 * r, 64);
            void *p = nullptr;
            CUDA_CHECK_RET(c, cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
            c->peer.opened[r] = p;
            base = (char *) p;
        }
        c->peer.px.inbox[r] = (uint4 *) base;
    }
    c->peer.px.rank = rank; c->peer.px.world = world;
    c->peer.px.two_hop = (world > 2 && getenv("LDSO_B200_K2R_ONESHOT") == nullptr) ? 1 : 0;
    c->peer.px.epoch = c->peer.words; c->peer.px.done = (unsigned *) (c->peer.words + 1); c->peer.px.error = c->peer.words + 2;
    c->peer.px.out = c->peer.red_sum;
    c->peer.connected = true;
    c->gn_graph_valid = false;
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_peer_error(ldso_b200_ctx *c, int *error) {
    if (!c || !error || !c->peer.words) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(d2h(c, error, c->peer.words + 2, sizeof(int)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}


extern "C" int ldso_b200_gn_phase_a(ldso_b200_ctx *c, int iteration) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    RET_IF(clear_select(c));
    if (iteration < 0) {
        RET_IF(launch_k1(c, K1_FUSED | K1F_RESET_OOB));
    } else {
        if (!c->solve_ready) return c->fail(LDSO_B200_ERR_STATE, "gn_phase_a(iteration >= 0) needs a preceding gn_phase_b");
        RET_IF(flush_select(c));
        RET_IF(set_iteration(c, iteration));
        RET_IF(launch_k3(c, K3F_BACKUP | K3F_SOLVE | K3F_STEP));
        RET_IF(launch_k1(c, K1_FUSED | K1F_APPLY_STEP));
    }
    RET_IF(launch_k2a(c, 1));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_gn_phase_b(ldso_b200_ctx *c) {
    if (!c) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    RET_IF(launch_k2b(c, 1, 1, 1));
    return LDSO_B200_OK;
}

// ---------------------------------------------------------------------------------------------- read-back
extern "C" int ldso_b200_get_energy(ldso_b200_ctx *c, double *energy, int *canbreak) {
    if (!c || !c->have_frames) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    RET_IF(d2h(c, energy, &c->ws_dev->energy, sizeof(double)));
    RET_IF(d2h(c, canbreak, &c->ws_dev->canbreak, sizeof(int)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

// one D2H of the contiguous result range into the pinned mirror (valid until the next launch)
// Optional hint: queue the read-back of everything the getters below return (solution, point and residual arrays) into
// pinned staging memory right behind the work already on the stream, without blocking. The next getter then only waits
// for that one event instead of issuing its own copy + synchronize.
extern "C" int ldso_b200_prefetch_results(ldso_b200_ctx *c) {
    if (!c || !c->have_window || !c->have_frames) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    auto &L = c->lay;
    const size_t nn = (size_t) MAXN * MAXN;
    if (!c->mirror_valid)
        RET_IF(d2h(c, c->arena_host + L.res_state, c->arena_dev + L.res_state, L.dl_light_end - L.res_state));
    if (!c->sol_valid)
        RET_IF(d2h(c, c->sol_host, c->sb.lastHS, sizeof(double) * (nn + 2 * MAXN)));
    if (!c->results_ready) CUDA_CHECK_RET(c, cudaEventCreateWithFlags(&c->results_ready, cudaEventDisableTiming));
    CUDA_CHECK_RET(c, cudaEventRecord(c->results_ready, c->stream));
    c->results_inflight = true;
    return LDSO_B200_OK;
}
int wait_results(ldso_b200_ctx *c) {
    if (!c->results_inflight) return LDSO_B200_OK;
    CUDA_CHECK_RET(c, cudaEventSynchronize(c->results_ready));
    c->results_inflight = false;
    c->mirror_valid = true;
    c->sol_valid = true;
    return LDSO_B200_OK;
}

static int refresh_mirror(ldso_b200_ctx *c, bool full = false) {
    RET_IF(wait_results(c));
    auto &L = c->lay;
    bool copied = false;
    if (!c->mirror_valid) {
        RET_IF(d2h(c, c->arena_host + L.res_state, c->arena_dev + L.res_state, L.dl_light_end - L.res_state));
        copied = true;
    }
    if (full && !c->mirror_full_valid) {
        RET_IF(d2h(c, c->arena_host + L.dl_light_end, c->arena_dev + L.dl_light_end, L.dl_end - L.dl_light_end));
        copied = true;
    }
    if (copied) CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    c->mirror_valid = true;
    if (full) c->mirror_full_valid = true;
    return LDSO_B200_OK;
}
#define FROM_MIRROR(dst, off, bytes) do { if (dst) memcpy(dst, c->arena_host + (off), (bytes)); } while (0)

extern "C" int ldso_b200_get_points(ldso_b200_ctx *c, float *idepth, float *idepth_zero, float *step, float *HdiF,
                                    float *bdSumF, float *Hdd, float *bd, float *Hcd4) {
    if (!c || !c->have_window) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    RET_IF(refresh_mirror(c));
    const size_t nP = c->d.nP;
    auto &L = c->lay;
    FROM_MIRROR(idepth, L.pt_idepth, 4 * nP); FROM_MIRROR(idepth_zero, L.pt_idepth_zero, 4 * nP); FROM_MIRROR(step, L.pt_step, 4 * nP);
    FROM_MIRROR(HdiF, L.pt_HdiF, 4 * nP); FROM_MIRROR(bdSumF, L.pt_bdSumF, 4 * nP); FROM_MIRROR(Hdd, L.pt_Hdd, 4 * nP);
    FROM_MIRROR(bd, L.pt_bd, 4 * nP); FROM_MIRROR(Hcd4, L.pt_Hcd, 16 * nP);
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_get_residuals(ldso_b200_ctx *c, uint8_t *state_state, uint8_t *state_NewState, float *state_energy,
                                       float *state_NewEnergy, float *state_NewEnergyWithOutlier, uint8_t *isActive,
                                       float *JpJdF8, float *J74, float *projectedTo16, float *centerProjectedTo3) {
    if (!c || !c->have_window) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    RET_IF(refresh_mirror(c, JpJdF8 != nullptr));
    const size_t nR = c->d.nR;
    auto &L = c->lay;
    FROM_MIRROR(state_state, L.res_state, nR); FROM_MIRROR(state_NewState, L.res_new_state, nR); FROM_MIRROR(state_energy, L.res_energy, 4 * nR);
    FROM_MIRROR(state_NewEnergy, L.res_new_energy, 4 * nR); FROM_MIRROR(state_NewEnergyWithOutlier, L.res_new_energy_wo, 4 * nR);
    FROM_MIRROR(isActive, L.res_active, nR); FROM_MIRROR(JpJdF8, L.res_JpJdF, 32 * nR);
    if (J74 || projectedTo16 || centerProjectedTo3) {
        RET_IF(d2h(c, J74, c->d.res_J, 296 * nR));
        RET_IF(d2h(c, projectedTo16, c->d.res_proj, 64 * nR));
        RET_IF(d2h(c, centerProjectedTo3, c->d.res_cpt, 12 * nR));
        CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    }
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_get_frames(ldso_b200_ctx *c, double *state10, double *step10, float *frameEnergyTH, float *precalc40,
                                    double *adHost64, double *adTarget64, float *adHTdeltaF8, double *calib_value4) {
    if (!c || !c->have_frames) return LDSO_B200_ERR_STATE;
    cudaSetDevice(c->device);
    if (c->have_window && !c->derived_dirty) RET_IF(flush_select(c));
    RET_IF(d2h(c, c->ws_host, c->ws_dev, sizeof(WinState)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    const WinState &W = *c->ws_host;
    const int nF = W.nF;
    for (int h = 0; h < nF; h++) {
        if (state10) memcpy(state10 + 10 * h, W.fr[h].state, 80);
        if (step10) memcpy(step10 + 10 * h, W.fr[h].step, 80);
        if (frameEnergyTH) frameEnergyTH[h] = W.frameEnergyTH[h];
    }
    for (int q = 0; q < nF * nF; q++) {
        if (precalc40) {
            float *d = precalc40 + 40 * q;
            const PairRec &p = W.pair[q];
            const PairRecFull &f = W.pairFull[q];
            memcpy(d, p.R0, 36); memcpy(d + 9, p.t0, 12); memcpy(d + 12, f.RTll, 36); memcpy(d + 21, f.tTll, 12);
            memcpy(d + 24, p.KRKi, 36); memcpy(d + 33, p.Kt, 12);
            d[36] = p.aff[0]; d[37] = p.aff[1]; d[38] = p.b0; d[39] = p.distanceLL;
        }
        if (adHost64) memcpy(adHost64 + 64 * q, W.adHost[q], 512);
        if (adTarget64) memcpy(adTarget64 + 64 * q, W.adTarget[q], 512);
        if (adHTdeltaF8) memcpy(adHTdeltaF8 + 8 * q, W.adHTdeltaF[q], 32);
    }
    if (calib_value4) memcpy(calib_value4, W.calib.value, 32);
    return LDSO_B200_OK;
}

