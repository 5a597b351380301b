// ldso_b200 C ABI implementation (include/ldso_b200.h), immature points and the initializer: immature_init, trace_immature,
// optimize_immature, select_activation and init_calc_res. Their kernels are compiled in trace.cu (see trace_types.h).
#include "context.h"
#include "trace_types.h"

// ---------------------------------------------------------------------------------------------- immature points
static TraceSettingsDev trace_settings(const ldso_b200_ctx *c) {
    TraceSettingsDev T;
    T.maxPixSearch = c->S.maxPixSearch; T.outlierTH = c->S.outlierTH; T.outlierTHSumComponent = c->S.outlierTHSumComponent;
    T.huberTH = c->S.huberTH; T.overallEnergyTHWeight = c->S.overallEnergyTHWeight;
    T.minTraceTestRadius = c->S.minTraceTestRadius; T.trace_GNIterations = c->S.trace_GNIterations;
    T.trace_stepsize = c->S.trace_stepsize; T.trace_GNThreshold = c->S.trace_GNThreshold;
    T.trace_extraSlackOnTH = c->S.trace_extraSlackOnTH; T.trace_slackInterval = c->S.trace_slackInterval;
    T.trace_minImprovementFactor = c->S.trace_minImprovementFactor;
    return T;
}

extern "C" int ldso_b200_immature_init(ldso_b200_ctx *c, int host_slot, int n, const float *u, const float *v, float *color8,
                                       float *weights8, float *gradH4, float *energyTH) {
    if (!c || n < 0 || (n > 0 && (!u || !v || !color8 || !weights8 || !gradH4 || !energyTH))) return LDSO_B200_ERR_ARG;
    if (host_slot < 0 || host_slot >= NSLOTS || !c->img[host_slot][0]) return c->fail(LDSO_B200_ERR_ARG, "host image slot not uploaded");
    if (n == 0) return LDSO_B200_OK;
    cudaSetDevice(c->device);
    const size_t N = (size_t) n;
    Arena L;
    const size_t o_u = L.take(4 * N), o_v = L.take(4 * N), o_out = L.take(4 * 21 * N);      // out: color8 weights8 gradH4 energyTH
    RET_IF(reserve_scratch(c, L.off));
    char *B = c->scr.buf;
    float *dc = (float *) (B + o_out), *dw = dc + 8 * N, *dg = dw + 8 * N, *de = dg + 4 * N;
    RET_IF(h2d(c, B + o_u, u, 4 * N));
    RET_IF(h2d(c, B + o_v, v, 4 * N));
    CUDA_CHECK_RET(c, cudaMemsetAsync(dc, 0, sizeof(float) * N * 21, c->stream));
    launch_immature_init(n, c->img[host_slot][0], c->w, (float *) (B + o_u), (float *) (B + o_v), trace_settings(c), dc, dw, dg, de, c->stream);
    LAUNCH_CHECK(c);
    RET_IF(d2h(c, color8, dc, 32 * N)); RET_IF(d2h(c, weights8, dw, 32 * N)); RET_IF(d2h(c, gradH4, dg, 16 * N)); RET_IF(d2h(c, energyTH, de, 4 * N));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_trace_immature(ldso_b200_ctx *c, int new_slot, const ldso_b200_immature *p, int n_hosts, const float *KRKi9,
                                        const float *Kt3, const float *aff2) {
    if (!c || !p || !KRKi9 || !Kt3 || !aff2 || n_hosts < 1) return LDSO_B200_ERR_ARG;
    if (new_slot < 0 || new_slot >= NSLOTS || !c->img[new_slot][0]) return c->fail(LDSO_B200_ERR_ARG, "image slot of the traced frame not uploaded");
    const int n = p->n;
    if (n < 0) return c->fail(LDSO_B200_ERR_ARG, "negative candidate count");
    if (n == 0) return LDSO_B200_OK;
    if (!p->u || !p->v || !p->host || !p->color8 || !p->weights8 || !p->gradH4 || !p->energyTH || !p->idepth_min || !p->idepth_max ||
        !p->quality || !p->lastTraceStatus || !p->lastTraceUV2 || !p->lastTracePixelInterval) return c->fail(LDSO_B200_ERR_ARG, "null candidate array");
    for (int i = 0; i < n; i++) if (p->host[i] < 0 || p->host[i] >= n_hosts) return c->fail(LDSO_B200_ERR_ARG, "candidate host index out of range");
    cudaSetDevice(c->device);
    const size_t N = (size_t) n, H = (size_t) n_hosts;
    Arena L;
    const size_t o_u = L.take(4 * N), o_v = L.take(4 * N), o_c = L.take(32 * N), o_w = L.take(32 * N), o_g = L.take(16 * N), o_e = L.take(4 * N),
                 o_min = L.take(4 * N), o_max = L.take(4 * N), o_q = L.take(4 * N), o_uv = L.take(8 * N), o_iv = L.take(4 * N), o_h = L.take(4 * N),
                 o_s = L.take(4 * N), o_K = L.take(36 * H), o_t = L.take(12 * H), o_a = L.take(8 * H);
    RET_IF(reserve_scratch(c, L.off));
    char *B = c->scr.buf;
    RET_IF(h2d(c, B + o_u, p->u, 4 * N)); RET_IF(h2d(c, B + o_v, p->v, 4 * N)); RET_IF(h2d(c, B + o_c, p->color8, 32 * N));
    RET_IF(h2d(c, B + o_w, p->weights8, 32 * N)); RET_IF(h2d(c, B + o_g, p->gradH4, 16 * N)); RET_IF(h2d(c, B + o_e, p->energyTH, 4 * N));
    RET_IF(h2d(c, B + o_min, p->idepth_min, 4 * N)); RET_IF(h2d(c, B + o_max, p->idepth_max, 4 * N)); RET_IF(h2d(c, B + o_q, p->quality, 4 * N));
    RET_IF(h2d(c, B + o_uv, p->lastTraceUV2, 8 * N)); RET_IF(h2d(c, B + o_iv, p->lastTracePixelInterval, 4 * N));
    RET_IF(h2d(c, B + o_h, p->host, 4 * N)); RET_IF(h2d(c, B + o_s, p->lastTraceStatus, 4 * N));
    RET_IF(h2d(c, B + o_K, KRKi9, 36 * H)); RET_IF(h2d(c, B + o_t, Kt3, 12 * H)); RET_IF(h2d(c, B + o_a, aff2, 8 * H));
    TraceArgs A;
    A.n = n; A.w = c->w; A.h = c->h; A.img = c->img[new_slot][0]; A.S = trace_settings(c);
    A.u = (float *) (B + o_u); A.v = (float *) (B + o_v); A.color8 = (float *) (B + o_c); A.weights8 = (float *) (B + o_w);
    A.gradH4 = (float *) (B + o_g); A.energyTH = (float *) (B + o_e); A.host = (int *) (B + o_h);
    A.KRKi9 = (float *) (B + o_K); A.Kt3 = (float *) (B + o_t); A.aff2 = (float *) (B + o_a);
    A.idepth_min = (float *) (B + o_min); A.idepth_max = (float *) (B + o_max); A.quality = (float *) (B + o_q); A.status = (int *) (B + o_s);
    A.uv2 = (float *) (B + o_uv); A.interval = (float *) (B + o_iv);
    launch_trace_on(A, c->stream);
    LAUNCH_CHECK(c);
    RET_IF(d2h(c, p->idepth_min, A.idepth_min, 4 * N)); RET_IF(d2h(c, p->idepth_max, A.idepth_max, 4 * N)); RET_IF(d2h(c, p->quality, A.quality, 4 * N));
    RET_IF(d2h(c, p->lastTraceStatus, A.status, 4 * N)); RET_IF(d2h(c, p->lastTraceUV2, A.uv2, 8 * N));
    RET_IF(d2h(c, p->lastTracePixelInterval, A.interval, 4 * N));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

extern "C" int ldso_b200_optimize_immature(ldso_b200_ctx *c, int n, const float *u, const float *v, const int32_t *host, const float *idepth_min,
                                           const float *idepth_max, const float *color8, const float *weights8, const float *energyTH,
                                           int min_obs, int32_t *ok, float *idepth, uint8_t *res_state) {
    if (!c || n < 0) return LDSO_B200_ERR_ARG;
    if (!c->have_frames) return c->fail(LDSO_B200_ERR_STATE, "optimize_immature needs set_frames first");
    if (n == 0) return LDSO_B200_OK;
    if (!u || !v || !host || !idepth_min || !idepth_max || !color8 || !weights8 || !energyTH || !ok || !idepth || !res_state)
        return c->fail(LDSO_B200_ERR_ARG, "null candidate array");
    const int nF = c->nF;
    if (nF < 2) return c->fail(LDSO_B200_ERR_STATE, "optimize_immature needs at least two frames");
    for (int i = 0; i < n; i++) if (host[i] < 0 || host[i] >= nF) return c->fail(LDSO_B200_ERR_ARG, "candidate host index out of range");
    cudaSetDevice(c->device);
    const size_t N = (size_t) n;
    Arena L;
    const size_t o_u = L.take(4 * N), o_v = L.take(4 * N), o_min = L.take(4 * N), o_max = L.take(4 * N), o_c = L.take(32 * N), o_w = L.take(32 * N),
                 o_e = L.take(4 * N), o_h = L.take(4 * N), o_ok = L.take(4 * N), o_id = L.take(4 * N), o_st = L.take(N * nF);
    RET_IF(reserve_scratch(c, L.off));
    char *B = c->scr.buf;
    RET_IF(h2d(c, B + o_u, u, 4 * N)); RET_IF(h2d(c, B + o_v, v, 4 * N)); RET_IF(h2d(c, B + o_min, idepth_min, 4 * N));
    RET_IF(h2d(c, B + o_max, idepth_max, 4 * N)); RET_IF(h2d(c, B + o_c, color8, 32 * N)); RET_IF(h2d(c, B + o_w, weights8, 32 * N));
    RET_IF(h2d(c, B + o_e, energyTH, 4 * N)); RET_IF(h2d(c, B + o_h, host, 4 * N));
    launch_optimize_immature(n, c->ws_dev, (float *) (B + o_u), (float *) (B + o_v), (int *) (B + o_h), (float *) (B + o_min), (float *) (B + o_max),
                             (float *) (B + o_c), (float *) (B + o_w), (float *) (B + o_e), min_obs, (int *) (B + o_ok), (float *) (B + o_id),
                             (unsigned char *) (B + o_st), c->stream);
    LAUNCH_CHECK(c);
    RET_IF(d2h(c, ok, B + o_ok, 4 * N)); RET_IF(d2h(c, idepth, B + o_id, 4 * N)); RET_IF(d2h(c, res_state, B + o_st, N * nF));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    return LDSO_B200_OK;
}

// FullSystem::activatePointsMT's selection (FullSystem.cc:1076-1150): distance map of the window's points in the newest keyframe,
// then the greedy pass over the candidates. One kernel, one CTA (the pass is order-dependent by construction).
extern "C" int ldso_b200_select_activation(ldso_b200_ctx *c, int newest_frame, float current_min_act_dist, float min_trace_quality, int n,
                                           const float *u, const float *v, const int32_t *host, const float *idepth_min, const float *idepth_max,
                                           const int32_t *lastTraceStatus, const float *lastTracePixelInterval, const float *quality,
                                           const float *my_type, const uint8_t *frame_flagged, uint8_t *action, float *dist_map) {
    if (!c || n < 0) return LDSO_B200_ERR_ARG;
    if (!c->have_frames || !c->have_window) return c->fail(LDSO_B200_ERR_STATE, "select_activation needs set_frames and set_window first");
    const int nF = c->nF;
    if (newest_frame < 0 || newest_frame >= nF) return c->fail(LDSO_B200_ERR_ARG, "newest_frame out of range");
    if (n > 0 && (!u || !v || !host || !idepth_min || !idepth_max || !lastTraceStatus || !lastTracePixelInterval || !quality || !my_type || !action))
        return c->fail(LDSO_B200_ERR_ARG, "null candidate array");
    if (!frame_flagged) return c->fail(LDSO_B200_ERR_ARG, "frame_flagged must hold one byte per frame");
    for (int i = 0; i < n; i++) if (host[i] < 0 || host[i] >= nF || host[i] == newest_frame) return c->fail(LDSO_B200_ERR_ARG, "candidate host must be a window frame other than the newest");
    cudaSetDevice(c->device);
    RET_IF(build_derived(c));
    const int w1 = c->w >> 1, h1 = c->h >> 1;
    const size_t N = (size_t) std::max(n, 1), cells = (size_t) w1 * h1, map_bytes = (cells + 3) & ~(size_t) 3;
    // the nine candidate arrays (u v idmin idmax quality interval my_type status host, N words each) are ONE block: they travel
    // in one copy from a pinned staging block laid out the same way
    Arena L;
    const size_t o_front0 = L.take(4 * cells), o_front1 = L.take(4 * cells), o_in = L.take(4 * 9 * N), o_idx = L.take(4 * N),
                 o_frac = L.take(4 * N), o_thresh = L.take(4 * N), o_map = L.take(map_bytes), o_act = L.take(N), o_flag = L.take(MAXF),
                 o_dbg = L.take(sizeof(long long) * 4);
    RET_IF(reserve_scratch(c, L.off));
    char *B = c->scr.buf;
    ActSelArgs A;
    A.ws = c->ws_dev; A.newest = newest_frame; A.w1 = w1; A.h1 = h1;
    A.nP = c->d.nP; A.pt_host = c->d.pt_host; A.pt_u = c->d.pt_u; A.pt_v = c->d.pt_v; A.pt_idepth = c->d.pt_idepth;
    A.n = n;
    A.front0 = (int *) (B + o_front0); A.front1 = (int *) (B + o_front1);
    const float *in = (const float *) (B + o_in);
    A.u = in; A.v = in + N; A.idmin = in + 2 * N; A.idmax = in + 3 * N; A.quality = in + 4 * N; A.interval = in + 5 * N; A.my_type = in + 6 * N;
    A.status = (const int *) (in + 7 * N); A.host = (const int *) (in + 8 * N);
    A.pre_idx = (int *) (B + o_idx); A.pre_frac = (float *) (B + o_frac); A.pre_thresh = (float *) (B + o_thresh);
    A.map = (unsigned char *) (B + o_map); A.action = (unsigned char *) (B + o_act); A.flagged = (unsigned char *) (B + o_flag);
    A.map_bytes = (int) map_bytes;
    A.currentMinActDist = current_min_act_dist; A.minTraceQuality = min_trace_quality;
    // the kernel also has a global-memory map path (use_smem = 0) for larger images; it has not been exercised on hardware yet, so
    // larger images are refused rather than served by an unvalidated path (level 1 of 1240x376 needs 114 KB)
    if (map_bytes > 200 * 1024) return c->fail(LDSO_B200_ERR_ARG, "select_activation: level-1 image larger than 200 KB (one byte per pixel must fit in shared memory)");
    A.use_smem = 1;
    // the nine candidate arrays and the frame flags are staged in one pinned block
    const size_t in_words = 9 * N, in_bytes = 4 * in_words, stage_bytes = in_bytes + N + MAXF + 16;
    if (stage_bytes > c->scr.actsel_pin_cap) {
        if (c->scr.actsel_pin) cudaFreeHost(c->scr.actsel_pin);
        c->scr.actsel_pin = nullptr; c->scr.actsel_pin_cap = 0;
        CUDA_CHECK_RET(c, cudaHostAlloc((void **) &c->scr.actsel_pin, stage_bytes * 2, cudaHostAllocDefault));
        c->scr.actsel_pin_cap = stage_bytes * 2;
    }
    {
        unsigned char *hp = c->scr.actsel_pin;
        const void *src[9] = {u, v, idepth_min, idepth_max, quality, lastTracePixelInterval, my_type, lastTraceStatus, host};
        for (int k = 0; k < 9; k++) if (n > 0) memcpy(hp + 4 * N * k, src[k], 4 * (size_t) n);
        RET_IF(h2d(c, B + o_in, hp, in_bytes));
        memcpy(hp + in_bytes, frame_flagged, (size_t) nF);
        RET_IF(h2d(c, B + o_flag, hp + in_bytes, (size_t) nF));
    }
    A.dbg = c->ktime ? (long long *) (B + o_dbg) : nullptr;
    c->kt_begin("actsel");
    launch_activation_select(A, c->stream);
    c->kt_end();
    LAUNCH_CHECK(c);
    unsigned char *hact = c->scr.actsel_pin + in_bytes + MAXF + 8;
    if (n > 0) RET_IF(d2h(c, hact, A.action, (size_t) n));
    if (dist_map) {
        c->scr.map_host.resize(map_bytes);
        RET_IF(d2h(c, c->scr.map_host.data(), A.map, map_bytes));
    }
    long long stamps[4] = {0, 0, 0, 0};
    if (A.dbg) RET_IF(d2h(c, stamps, A.dbg, sizeof(stamps)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    if (n > 0) memcpy(action, hact, (size_t) n);
    if (A.dbg) fprintf(stderr, "[ldso_b200 actsel] cycles: map+seeds+grow %lld, candidate terms %lld, sequential pass %lld\n", stamps[1] - stamps[0],
                       stamps[2] - stamps[1], stamps[3] - stamps[2]);
    if (dist_map) for (size_t i = 0; i < cells; i++) dist_map[i] = c->scr.map_host[i] == 255 ? 1000.f : (float) c->scr.map_host[i];   // fwdWarpedIDDistFinal's values
    return LDSO_B200_OK;
}

// CoarseInitializer::calcResAndGS (src/frontend/CoarseInitializer.cc:181-405) for the points of one pyramid level. EXPERIMENTAL: written
// at the end of round 1 against the pinned oracle (oracle/initializer.cc), compiled, NOT yet run on hardware (tests/test_gpu_init.py is
// skipped unless LDSO_B200_RUN_UNVALIDATED is set).
extern "C" int ldso_b200_init_calc_res(ldso_b200_ctx *c, int first_slot, int new_slot, int lvl, const double R[9], const double t[3], const double tlog3[3],
                                       float aff_a, float aff_b, float fx0, float fy0, float cx0, float cy0, int n, const float *u, const float *v,
                                       const float *idepth_new, const float *iR, const uint8_t *isGood, const float *energy2, const float *outlierTH,
                                       float alphaK, float alphaW, float couplingWeight, uint8_t *isGood_new, float *energy_new2, float *maxstep,
                                       float *lastHessian_new, float *JbBuffer_new10, float *H64, float *b8, float *Hsc64, float *bsc8, float *res3) {
    if (!c || n <= 0 || !R || !t || !tlog3) return LDSO_B200_ERR_ARG;
    if (lvl < 0 || lvl >= c->levels) return c->fail(LDSO_B200_ERR_ARG, "pyramid level out of range");
    if (first_slot < 0 || first_slot >= NSLOTS || new_slot < 0 || new_slot >= NSLOTS || !c->img[first_slot][lvl] || !c->img[new_slot][lvl])
        return c->fail(LDSO_B200_ERR_ARG, "image slot not uploaded");
    if (!u || !v || !idepth_new || !iR || !isGood || !energy2 || !outlierTH || !isGood_new || !energy_new2 || !maxstep || !lastHessian_new ||
        !JbBuffer_new10 || !H64 || !b8 || !Hsc64 || !bsc8 || !res3) return c->fail(LDSO_B200_ERR_ARG, "null array");
    const int wl = c->w >> lvl, hl = c->h >> lvl;
    for (int i = 0; i < n; i++)      // the reference samples the first frame at (u + dx, v + dy) without a bounds check (its selector keeps a margin)
        if (!(u[i] >= 2 && v[i] >= 2 && u[i] < wl - 3 && v[i] < hl - 3)) return c->fail(LDSO_B200_ERR_ARG, "initializer point closer than the pattern radius to the image border");
    cudaSetDevice(c->device);
    // CoarseInitializer::makeK (:689-715) in double, K^-1 by Eigen's 3x3 cofactor formula
    double fx = fx0, fy = fy0, cx = cx0, cy = cy0;
    for (int level = 1; level <= lvl; ++level) { fx = fx * 0.5; fy = fy * 0.5; }
    if (lvl > 0) { cx = ((double) cx0 + 0.5) / ((int) 1 << lvl) - 0.5; cy = ((double) cy0 + 0.5) / ((int) 1 << lvl) - 0.5; }
    const double K[9] = {fx, 0, cx, 0, fy, cy, 0, 0, 1};
    double Ki[9];
    {
        const double c00 = K[4] * K[8] - K[5] * K[7], c01 = K[5] * K[6] - K[3] * K[8], c02 = K[3] * K[7] - K[4] * K[6];
        const double det = K[0] * c00 + K[1] * c01 + K[2] * c02, invdet = 1.0 / det;
        Ki[0] = c00 * invdet; Ki[3] = c01 * invdet; Ki[6] = c02 * invdet;
        Ki[1] = (K[2] * K[7] - K[1] * K[8]) * invdet; Ki[4] = (K[0] * K[8] - K[2] * K[6]) * invdet; Ki[7] = (K[1] * K[6] - K[0] * K[7]) * invdet;
        Ki[2] = (K[1] * K[5] - K[2] * K[4]) * invdet; Ki[5] = (K[2] * K[3] - K[0] * K[5]) * invdet; Ki[8] = (K[0] * K[4] - K[1] * K[3]) * invdet;
    }
    InitArgs A;
    A.n = n; A.w = wl; A.h = hl;
    A.imgRef = c->img[first_slot][lvl]; A.imgNew = c->img[new_slot][lvl];
    for (int i = 0; i < 3; i++) {
        for (int j = 0; j < 3; j++) { double s = R[i * 3] * Ki[j]; s += R[i * 3 + 1] * Ki[3 + j]; s += R[i * 3 + 2] * Ki[6 + j]; A.RKi[i * 3 + j] = (float) s; }
        A.t[i] = (float) t[i];
    }
    A.aff0 = std::exp(aff_a); A.aff1 = aff_b;
    A.fx = (float) fx; A.fy = (float) fy; A.cx = (float) cx; A.cy = (float) cy; A.huberTH = c->S.huberTH;
    // alpha energy (:336-356): the reference's EAlpha accumulator never receives a term, so it depends on the translation only
    const double tsq = t[0] * t[0] + t[1] * t[1] + t[2] * t[2];
    float alphaEnergy = (float) ((double) alphaW * ((double) 0.0f + tsq * n));
    float alphaOpt;
    if (alphaEnergy > alphaK * n) { alphaOpt = 0; alphaEnergy = alphaK * n; } else alphaOpt = alphaW;
    A.alphaOpt = alphaOpt; A.couplingWeight = couplingWeight;
    const size_t N = (size_t) n, grid = (N + INIT_THREADS / 8 - 1) / (INIT_THREADS / 8);
    Arena L;
    const size_t o_u = L.take(4 * N), o_v = L.take(4 * N), o_id = L.take(4 * N), o_iR = L.take(4 * N), o_e2 = L.take(8 * N), o_oth = L.take(4 * N),
                 o_good = L.take(N), o_good_new = L.take(N), o_res = L.take(4 * (2 + 1 + 1 + 10) * N),     // energy_new2, maxstep, lastHessian_new, Jb
                 o_part = L.take(4 * grid * INIT_NACC), o_cnt = L.take(16), o_out = L.take(sizeof(double) * INIT_NACC);
    RET_IF(reserve_scratch(c, L.off));
    char *B = c->scr.buf;
    RET_IF(h2d(c, B + o_u, u, 4 * N)); RET_IF(h2d(c, B + o_v, v, 4 * N)); RET_IF(h2d(c, B + o_id, idepth_new, 4 * N)); RET_IF(h2d(c, B + o_iR, iR, 4 * N));
    RET_IF(h2d(c, B + o_e2, energy2, 8 * N)); RET_IF(h2d(c, B + o_oth, outlierTH, 4 * N)); RET_IF(h2d(c, B + o_good, isGood, N));
    CUDA_CHECK_RET(c, cudaMemsetAsync(B + o_res, 0, 4 * (size_t) (2 + 1 + 1 + 10) * N, c->stream));
    CUDA_CHECK_RET(c, cudaMemsetAsync(B + o_cnt, 0, 16, c->stream));
    A.u = (float *) (B + o_u); A.v = (float *) (B + o_v); A.idepth_new = (float *) (B + o_id); A.iR = (float *) (B + o_iR);
    A.energy2 = (float *) (B + o_e2); A.outlierTH = (float *) (B + o_oth); A.isGood = (unsigned char *) (B + o_good);
    A.isGood_new = (unsigned char *) (B + o_good_new); A.energy_new2 = (float *) (B + o_res); A.maxstep = A.energy_new2 + 2 * N;
    A.lastHessian_new = A.maxstep + N; A.Jb = A.lastHessian_new + N;
    A.partials = (float *) (B + o_part); A.counter = (unsigned *) (B + o_cnt); A.out = (double *) (B + o_out);
    launch_init_calc_res(A, c->stream);
    LAUNCH_CHECK(c);
    double sums[INIT_NACC];
    RET_IF(d2h(c, isGood_new, A.isGood_new, N)); RET_IF(d2h(c, energy_new2, A.energy_new2, 8 * N)); RET_IF(d2h(c, maxstep, A.maxstep, 4 * N));
    RET_IF(d2h(c, lastHessian_new, A.lastHessian_new, 4 * N)); RET_IF(d2h(c, JbBuffer_new10, A.Jb, 40 * N)); RET_IF(d2h(c, sums, A.out, sizeof(sums)));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    // acc9.H / acc9SC.H -> H_out, b_out, H_out_sc, b_out_sc (:390-403)
    int k = 0;
    for (int r = 0; r < 9; r++)
        for (int cc = r; cc < 9; cc++, k++) {
            const float hv = (float) sums[k], sv = (float) sums[45 + k];
            if (cc < 8) { H64[r * 8 + cc] = H64[cc * 8 + r] = hv; Hsc64[r * 8 + cc] = Hsc64[cc * 8 + r] = sv; }
            else if (r < 8) { b8[r] = hv; bsc8[r] = sv; }
        }
    for (int i = 0; i < 3; i++) { H64[i * 8 + i] += alphaOpt * n; b8[i] += (float) tlog3[i] * alphaOpt * n; }
    res3[0] = (float) sums[90]; res3[1] = alphaEnergy; res3[2] = (float) (2 * n);      // E.num counts both loops (:211-303 and :339-347)
    return LDSO_B200_OK;
}

