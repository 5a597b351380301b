// ldso_b200 C ABI implementation (include/ldso_b200.h), coarse tracker: reference point cloud, evaluation, the tracking LM
// loop (single and batched) and make_coarse_depth.
#include "context.h"
#include "tracker_kernels.cuh"

// ---------------------------------------------------------------------------------------------- tracker
bool tracker_alloc(ldso_b200_ctx *c) {
    bool ok = cudaMalloc(&c->trk.partials, sizeof(float) * 1024 * TRK_NACC) == cudaSuccess;
    ok = ok && cudaMalloc(&c->trk.counter, sizeof(unsigned)) == cudaSuccess;
    ok = ok && cudaMalloc(&c->trk.out_dev, sizeof(double) * 80) == cudaSuccess;
    ok = ok && cudaMalloc(&c->trk.track_out, sizeof(TrkTrackOut)) == cudaSuccess;
    return ok;
}

// the four point-cloud arrays of level lvl hold at least n points (their contents are not kept)
static int reserve_point_cloud(ldso_b200_ctx *c, int lvl, int n) {
    if (n <= c->trk.cap[lvl]) return LDSO_B200_OK;
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    for (int k = 0; k < 4; k++) {
        if (c->trk.pc[lvl][k]) cudaFree(c->trk.pc[lvl][k]);
        CUDA_CHECK_RET(c, cudaMalloc(&c->trk.pc[lvl][k], sizeof(float) * n));
    }
    c->trk.cap[lvl] = n;
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_tracker_make_k(ldso_b200_ctx *c, float fx, float fy, float cx, float cy) {
    if (!c) return LDSO_B200_ERR_ARG;
    // CoarseTracker::makeK (CoarseTracker.cc:219-246)
    c->trk.fx[0] = fx; c->trk.fy[0] = fy; c->trk.cx[0] = cx; c->trk.cy[0] = cy;
    for (int l = 1; l < c->levels; l++) {
        c->trk.fx[l] = c->trk.fx[l - 1] * 0.5;
        c->trk.fy[l] = c->trk.fy[l - 1] * 0.5;
        c->trk.cx[l] = (c->trk.cx[0] + 0.5) / ((int) 1 << l) - 0.5;
        c->trk.cy[l] = (c->trk.cy[0] + 0.5) / ((int) 1 << l) - 0.5;
    }
    for (int l = 0; l < c->levels; l++) {
        const float K[9] = {c->trk.fx[l], 0, c->trk.cx[l], 0, c->trk.fy[l], c->trk.cy[l], 0, 0, 1};
        m33f_inverse(K, c->trk.Ki[l]);
    }
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_tracker_set_ref_level(ldso_b200_ctx *c, int lvl, int n, const float *pc_u, const float *pc_v,
                                               const float *pc_idepth, const float *pc_color) {
    if (!c || lvl < 0 || lvl >= c->levels || n < 0) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    RET_IF(reserve_point_cloud(c, lvl, n));
    const float *src[4] = {pc_u, pc_v, pc_idepth, pc_color};
    for (int k = 0; k < 4; k++)
        RET_IF(h2d(c, c->trk.pc[lvl][k], src[k], sizeof(float) * n));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    c->trk.n[lvl] = n;
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_tracker_get_ref_level(ldso_b200_ctx *c, int lvl, int *n, float *pc_u, float *pc_v, float *pc_idepth, float *pc_color) {
    if (!c || lvl < 0 || lvl >= c->levels) return LDSO_B200_ERR_ARG;
    cudaSetDevice(c->device);
    const int m = c->trk.n[lvl];
    if (n) *n = m;
    float *dst[4] = {pc_u, pc_v, pc_idepth, pc_color};
    for (int k = 0; k < 4; k++) if (dst[k] && m > 0) RET_IF(d2h(c, dst[k], c->trk.pc[lvl][k], sizeof(float) * m));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_tracker_set_frames(ldso_b200_ctx *c, float ref_aff_a, float ref_aff_b, float ref_exposure, int new_slot, float new_exposure) {
    if (!c || new_slot < 0 || new_slot >= NSLOTS || !c->img[new_slot][0]) return LDSO_B200_ERR_ARG;
    c->trk.ref_aff_a = ref_aff_a; c->trk.ref_aff_b = ref_aff_b; c->trk.ref_exposure = ref_exposure;
    c->trk.new_slot = new_slot; c->trk.new_exposure = new_exposure;
    return LDSO_B200_OK;
}

static void fill_level(ldso_b200_ctx *c, int l, TrkLevel &L) {
    L.pc_u = c->trk.pc[l][0]; L.pc_v = c->trk.pc[l][1]; L.pc_idepth = c->trk.pc[l][2]; L.pc_color = c->trk.pc[l][3];
    L.n = c->trk.n[l];
    L.img = c->img[c->trk.new_slot][l];
    L.w = c->lw[l]; L.h = c->lh[l];
    L.fx = c->trk.fx[l]; L.fy = c->trk.fy[l]; L.cx = c->trk.cx[l]; L.cy = c->trk.cy[l];
    memcpy(L.Ki, c->trk.Ki[l], sizeof(L.Ki));
}

// the arguments of k_trk_track common to both track entry points, without an abort threshold
static TrkTrackArgs track_args(ldso_b200_ctx *c, int coarsestLvl) {
    TrkTrackArgs A;
    memset(&A, 0, sizeof(A));
    for (int l = 0; l < c->levels; l++) fill_level(c, l, A.L[l]);
    A.nLevels = c->levels;
    A.ref_aff_a = c->trk.ref_aff_a; A.ref_aff_b = c->trk.ref_aff_b; A.ref_exposure = c->trk.ref_exposure; A.new_exposure = c->trk.new_exposure;
    A.huberTH = c->S.huberTH; A.coarseCutoffTH = c->S.coarseCutoffTH; A.affineOptModeA = c->S.affineOptModeA; A.affineOptModeB = c->S.affineOptModeB;
    A.coarsestLvl = coarsestLvl;
    for (int i = 0; i < 5; i++) A.minResForAbort[i] = NAN;
    return A;
}

extern "C" int ldso_b200_tracker_eval(ldso_b200_ctx *c, int lvl, const double R[9], const double t[3], float aff_a, float aff_b,
                                      float cutoffTH, double res6[6], double H[64], double b[8]) {
    if (!c || lvl < 0 || lvl >= c->levels || !R || !t || !res6) return LDSO_B200_ERR_ARG;
    if (c->trk.new_slot < 0) return c->fail(LDSO_B200_ERR_STATE, "tracker_set_frames not called");
    cudaSetDevice(c->device);
    TrkLevel L;
    fill_level(c, lvl, L);
    TrkPose P;
    float Rf[9];
    for (int i = 0; i < 9; i++) Rf[i] = (float) R[i];
    m33f_mul(Rf, L.Ki, P.RKi);
    for (int i = 0; i < 3; i++) P.t[i] = (float) t[i];
    float eF = c->trk.ref_exposure, eT = c->trk.new_exposure;
    if (eF == 0 || eT == 0) eT = eF = 1;
    const float a = expf(aff_a - c->trk.ref_aff_a) * eT / eF;
    P.affLL0 = a; P.affLL1 = aff_b - a * c->trk.ref_aff_b; P.b0 = c->trk.ref_aff_b;
    P.cutoffTH = cutoffTH; P.huberTH = c->S.huberTH;
    P.maxEnergy = 2 * c->S.huberTH * cutoffTH - c->S.huberTH * c->S.huberTH;
    int grid = std::max(1, std::min(1024, (L.n + TRK_EVAL_THREADS - 1) / TRK_EVAL_THREADS));
    k_trk_eval<<<grid, TRK_EVAL_THREADS, 0, c->stream>>>(L, P, lvl == 0 ? 1 : 0, c->trk.partials, c->trk.counter, c->trk.out_dev, (H && b) ? 1 : 0);
    LAUNCH_CHECK(c);
    double out[78];
    RET_IF(d2h(c, out, c->trk.out_dev, sizeof(out)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    memcpy(res6, out, 48);
    if (H && b) { memcpy(H, out + 6, 512); memcpy(b, out + 70, 64); }
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_tracker_track(ldso_b200_ctx *c, double R[9], double t[3], float *aff_a, float *aff_b, int coarsestLvl,
                                       const double minResForAbort[5], double lastResiduals[5], double lastFlowIndicators[3], int *ok) {
    if (!c || !R || !t || !aff_a || !aff_b || !ok) return LDSO_B200_ERR_ARG;
    if (coarsestLvl < 0 || coarsestLvl >= 5 || coarsestLvl >= c->levels) return c->fail(LDSO_B200_ERR_ARG, "coarsestLvl out of range");
    if (c->trk.new_slot < 0) return c->fail(LDSO_B200_ERR_STATE, "tracker_set_frames not called");
    cudaSetDevice(c->device);
    TrkTrackArgs A = track_args(c, coarsestLvl);
    memcpy(A.R, R, 72); memcpy(A.t, t, 24);
    A.aff_a = *aff_a; A.aff_b = *aff_b;
    if (minResForAbort) memcpy(A.minResForAbort, minResForAbort, sizeof(A.minResForAbort));
    k_trk_track<<<1, TRK_TRACK_THREADS, 0, c->stream>>>(A, c->trk.track_out, nullptr);
    LAUNCH_CHECK(c);
    TrkTrackOut o;
    RET_IF(d2h(c, &o, c->trk.track_out, sizeof(o)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    memcpy(R, o.R, 72); memcpy(t, o.t, 24);
    *aff_a = o.aff_a; *aff_b = o.aff_b;
    if (lastResiduals) memcpy(lastResiduals, o.lastResiduals, 40);
    if (lastFlowIndicators) memcpy(lastFlowIndicators, o.lastFlowIndicators, 24);
    *ok = o.ok;
    return LDSO_B200_OK;
}

// FullSystem::trackNewCoarse's hypothesis loop (FullSystem.cc:290-357) as ONE launch: n starting poses (the constant-motion,
// double-motion, half-motion, zero-motion guesses and the 26 x 3 small rotations), each tracked by its own CTA through all levels,
// all without an abort threshold (the reference passes the best residuals so far as minResForAbort to the later tries: a pruning
// of work that a parallel batch does not need). The caller applies the reference's acceptance rule to the n results.
extern "C" int ldso_b200_tracker_track_batch(ldso_b200_ctx *c, int n, const double *R9_each, const double *t3_each, const float *aff2_each, int coarsestLvl,
                                             double *R9_out, double *t3_out, float *aff2_out, double *lastResiduals5_each, double *lastFlow3_each, int *ok_each) {
    if (!c || n <= 0 || !R9_each || !t3_each || !aff2_each || !ok_each) return LDSO_B200_ERR_ARG;
    if (n > 128) return c->fail(LDSO_B200_ERR_ARG, "at most 128 hypotheses per batch");
    if (coarsestLvl < 0 || coarsestLvl >= 5 || coarsestLvl >= c->levels) return c->fail(LDSO_B200_ERR_ARG, "coarsestLvl out of range");
    if (c->trk.new_slot < 0) return c->fail(LDSO_B200_ERR_STATE, "tracker_set_frames not called");
    cudaSetDevice(c->device);
    const TrkTrackArgs A = track_args(c, coarsestLvl);
    Arena L;
    const size_t o_hyp = L.take(sizeof(TrkHypothesis) * (size_t) n), o_out = L.take(sizeof(TrkTrackOut) * (size_t) n);
    RET_IF(reserve_scratch(c, L.off));
    TrkHypothesis *dh = (TrkHypothesis *) (c->scr.buf + o_hyp);
    TrkTrackOut *dout = (TrkTrackOut *) (c->scr.buf + o_out);
    std::vector<TrkHypothesis> hh(n);
    for (int i = 0; i < n; i++) {
        memcpy(hh[i].R, R9_each + 9 * i, 72); memcpy(hh[i].t, t3_each + 3 * i, 24);
        hh[i].aff_a = aff2_each[2 * i]; hh[i].aff_b = aff2_each[2 * i + 1];
    }
    RET_IF(h2d(c, dh, hh.data(), sizeof(TrkHypothesis) * n));
    k_trk_track<<<n, TRK_TRACK_THREADS, 0, c->stream>>>(A, dout, dh);
    LAUNCH_CHECK(c);
    std::vector<TrkTrackOut> ho(n);
    RET_IF(d2h(c, ho.data(), dout, sizeof(TrkTrackOut) * n));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    for (int i = 0; i < n; i++) {
        if (R9_out) memcpy(R9_out + 9 * i, ho[i].R, 72);
        if (t3_out) memcpy(t3_out + 3 * i, ho[i].t, 24);
        if (aff2_out) { aff2_out[2 * i] = ho[i].aff_a; aff2_out[2 * i + 1] = ho[i].aff_b; }
        if (lastResiduals5_each) memcpy(lastResiduals5_each + 5 * i, ho[i].lastResiduals, 40);
        if (lastFlow3_each) memcpy(lastFlow3_each + 3 * i, ho[i].lastFlowIndicators, 24);
        ok_each[i] = ho[i].ok;
    }
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_tracker_make_coarse_depth(ldso_b200_ctx *c, int ref_slot, int n, const float *centerProjectedTo3, const float *HdiF) {
    if (!c || n < 0 || (n > 0 && (!centerProjectedTo3 || !HdiF))) return LDSO_B200_ERR_ARG;
    if (ref_slot < 0 || ref_slot >= NSLOTS || !c->img[ref_slot][0]) return c->fail(LDSO_B200_ERR_ARG, "reference image slot not uploaded");
    if (c->lh[0] > 1024) return c->fail(LDSO_B200_ERR_ARG, "image height > 1024 not supported by the row scan");
    cudaSetDevice(c->device);
    // buffers: idepth / weightSums / weightSums_bak / pos per level, point-cloud arrays with wl*hl capacity (CoarseTracker.cc:36-45)
    for (int l = 0; l < c->levels; l++) {
        const size_t npx = (size_t) c->lw[l] * c->lh[l];
        if (!c->cd.id[l]) {
            CUDA_CHECK_RET(c, cudaMalloc(&c->cd.id[l], 4 * npx)); CUDA_CHECK_RET(c, cudaMalloc(&c->cd.ws[l], 4 * npx));
            CUDA_CHECK_RET(c, cudaMalloc(&c->cd.bak[l], 4 * npx)); CUDA_CHECK_RET(c, cudaMalloc(&c->cd.pos[l], 4 * npx));
        }
        RET_IF(reserve_point_cloud(c, l, (int) npx));
    }
    if (!c->cd.rows) { CUDA_CHECK_RET(c, cudaMalloc(&c->cd.rows, sizeof(int) * 1024)); CUDA_CHECK_RET(c, cudaMalloc(&c->cd.tot, sizeof(int) * MAXLVL)); }
    if (n > c->cd.in_cap) {
        CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
        if (c->cd.in) cudaFree(c->cd.in);
        CUDA_CHECK_RET(c, cudaMalloc(&c->cd.in, sizeof(float) * 4 * (size_t) n));
        c->cd.in_cap = n;
    }
    const size_t np0 = (size_t) c->lw[0] * c->lh[0];
    CUDA_CHECK_RET(c, cudaMemsetAsync(c->cd.id[0], 0, 4 * np0, c->stream));
    CUDA_CHECK_RET(c, cudaMemsetAsync(c->cd.ws[0], 0, 4 * np0, c->stream));
    if (n > 0) {
        RET_IF(h2d(c, c->cd.in, centerProjectedTo3, sizeof(float) * 3 * n));
        RET_IF(h2d(c, c->cd.in + 3 * (size_t) n, HdiF, sizeof(float) * n));
        k_cd_scatter<<<(n + 255) / 256, 256, 0, c->stream>>>(n, c->cd.in, c->cd.in + 3 * (size_t) n, c->cd.id[0], c->cd.ws[0], c->lw[0], c->lh[0]);
        LAUNCH_CHECK(c);
    }
    for (int l = 1; l < c->levels; l++) {
        const int npx = c->lw[l] * c->lh[l];
        k_cd_down<<<(npx + 255) / 256, 256, 0, c->stream>>>(c->cd.id[l - 1], c->cd.ws[l - 1], c->cd.id[l], c->cd.ws[l], c->lw[l], c->lh[l], c->lw[l - 1]);
        LAUNCH_CHECK(c);
    }
    for (int l = 0; l < c->levels; l++) {
        const int npx = c->lw[l] * c->lh[l];
        CUDA_CHECK_RET(c, cudaMemcpyAsync(c->cd.bak[l], c->cd.ws[l], 4 * (size_t) npx, cudaMemcpyDeviceToDevice, c->stream));
        k_cd_dilate<<<(npx + 255) / 256, 256, 0, c->stream>>>(c->cd.id[l], c->cd.ws[l], c->cd.bak[l], c->lw[l], c->lh[l], l < 2 ? 1 : 0);
        LAUNCH_CHECK(c);
    }
    for (int l = 0; l < c->levels; l++) {
        const int npx = c->lw[l] * c->lh[l];
        k_cd_rowcount<<<c->lh[l], 128, 0, c->stream>>>(c->cd.id[l], c->cd.ws[l], c->img[ref_slot][l], c->lw[l], c->lh[l], c->cd.pos[l], c->cd.rows);
        LAUNCH_CHECK(c);
        k_cd_rowscan<<<1, 1024, 0, c->stream>>>(c->cd.rows, c->lh[l], c->cd.tot + l);
        LAUNCH_CHECK(c);
        k_cd_emit<<<(npx + 255) / 256, 256, 0, c->stream>>>(c->cd.id[l], c->cd.ws[l], c->img[ref_slot][l], c->cd.pos[l], c->cd.rows, c->lw[l], c->lh[l],
                                                             c->trk.pc[l][0], c->trk.pc[l][1], c->trk.pc[l][2], c->trk.pc[l][3]);
        LAUNCH_CHECK(c);
    }
    int tot[MAXLVL];
    RET_IF(d2h(c, tot, c->cd.tot, sizeof(int) * c->levels));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    for (int l = 0; l < c->levels; l++) c->trk.n[l] = tot[l];
    return LDSO_B200_OK;
}

