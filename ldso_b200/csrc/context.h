// Private to the C ABI implementation (include/ldso_b200.h): the context every api_*.cu unit works on and the helpers they
// share. It defines no kernel, so every unit may include it; each kernel header is included by exactly one unit.
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <algorithm>
#include <cstddef>

#include "common.cuh"
#include "ba_types.h"

#define NSLOTS (2 * MAXF)

struct TrkTrackOut;

struct ldso_b200_ctx {
    int device = 0, w = 0, h = 0, levels = 0;
    int lw[MAXLVL], lh[MAXLVL];
    ldso_b200_settings S;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    std::string err;
    long long launches = 0;
    int sm_count = 148;

    float4 *img[NSLOTS][MAXLVL] = {};
    float *scratch = nullptr;          // upload staging (w*h*3 floats)
    cudaEvent_t copy_done = nullptr, frames_copied = nullptr;
    size_t scratch_floats = 0;

    // window
    DevWindow d = {};
    std::vector<void *> win_allocs;
    std::vector<void *> derived_allocs;      // work items, partials, reduced buffer: rebuilt by build_derived
    bool have_window = false, have_frames = false, derived_dirty = true;
    bool select_pending = false;     // the newest frame's energy threshold of the last fused iteration has not been computed yet (flush_select)
    bool has_lin = false;            // the window holds linearized (isLinearized) residuals: solve_system accumulates HA + HL in one pass
    std::vector<int> h_pt_host, h_res_begin, h_res_target;
    int nF = 0, n = 0;
    int slots[MAXF];
    WinState *ws_dev = nullptr;
    WinState *ws_host = nullptr;       // pinned staging copy
    SolveBufs sb = {};
    double *solve_mem = nullptr;
    double *sol_host = nullptr;      // pinned staging for get_last_solution
    // K2b(do_assemble) has produced the system K3 solves and nothing it depends on changed since
    bool solve_ready = false;
    // dimension of the device-resident marginalisation prior HM, bM (0 = all zero, any dimension): set_marg_prior,
    // marginalize_points -> n; marginalize_frame -> n - 8; set_frames keeps / grows / clears it accordingly
    int prior_dim = 0;
    // the reduced accumulators still describe the current window state (a re-stitch is enough to get solve_ready back)
    bool restitch_ok = false;
    int *iteration_dev = nullptr;
    uint8_t *pt_sel_dev = nullptr;
    char *arena_dev = nullptr, *arena_host = nullptr;
    struct Layout {
        size_t pt_host, pt_res_begin, res_point, res_target, topo_end, pt_u, pt_v, pt_color, pt_weights, pt_priorF, pt_idepth_backup,
            res_lin, res_state, dl_begin, pt_idepth, pt_idepth_zero, ul_end, pt_step, pt_HdiF, pt_bdSumF, pt_Hdd, pt_bd, pt_Hcd,
            res_new_state, res_active, res_energy, res_new_energy, res_new_energy_wo, dl_light_end, res_JpJdF, dl_end, res_JpJdF_new, total;
    } lay;
    bool mirror_valid = false;       // pinned mirror holds the current [res_state, dl_light_end) arrays
    bool mirror_full_valid = false;  // ... and the bulky [dl_light_end, dl_end) tail (JpJdF) as well
    bool sol_valid = false;          // sol_host holds the current [lastHS | lastbS | lastX]
    bool results_inflight = false;   // prefetch_results queued the read-back copies; results_ready marks their end
    cudaEvent_t results_ready = nullptr;
    std::vector<double> evalpt_key, Pns_host;
    cudaEvent_t window_copied = nullptr;
    // one GN iteration (K3 -> K1 -> K2a -> K2b) captured as a CUDA graph; re-captured when the window arena changes
    cudaGraphExec_t gn_graph = nullptr;
    bool gn_graph_valid = false;
    bool use_graph = true;
    bool use_pdl = true;             // programmatic dependent launch inside the GN iteration (env LDSO_B200_NO_PDL disables)
    bool pdl_now = false;            // set while launch_gn_body issues its four kernels
    size_t k1_smem = 0;
    bool multi = false;

    // peer-memory exchange (k2r_peer_allreduce): this rank's exported inbox, the peers' mapped inboxes, and the local
    // epoch / completion / error words
    struct Peer {
        char *local = nullptr;
        void *opened[K2R_MAX_PEERS] = {};
        int *words = nullptr;        // [0] epoch, [1] done, [2] error
        double *red_sum = nullptr;
        PeerExchange px;
        bool connected = false;
    } peer;

    // device scratch shared by the one-shot entry points (reserve_scratch), and select_activation's host staging
    struct Scratch {
        char *buf = nullptr;
        size_t cap = 0;
        unsigned char *actsel_pin = nullptr; size_t actsel_pin_cap = 0;      // pinned block of the candidate arrays
        std::vector<unsigned char> map_host;                                  // distance-map read-back
    } scr;

    // tracker: the reference point cloud per level and the two frames' photometric parameters
    struct Tracker {
        int n[MAXLVL] = {};
        float *pc[MAXLVL][4] = {};       // u, v, idepth, color
        int cap[MAXLVL] = {};
        float fx[MAXLVL], fy[MAXLVL], cx[MAXLVL], cy[MAXLVL];
        float Ki[MAXLVL][9];
        float ref_aff_a = 0, ref_aff_b = 0, ref_exposure = 1, new_exposure = 1;
        int new_slot = -1;
        float *partials = nullptr;
        unsigned *counter = nullptr;
        double *out_dev = nullptr;
        TrkTrackOut *track_out = nullptr;
    } trk;

    // coarse depth map of the tracker's reference frame (make_coarse_depth)
    struct CoarseDepth {
        float *id[MAXLVL] = {}, *ws[MAXLVL] = {}, *bak[MAXLVL] = {};
        int *pos[MAXLVL] = {};
        int *rows = nullptr, *tot = nullptr;
        float *in = nullptr;
        int in_cap = 0;
    } cd;

    // optional per-kernel CUDA-event timing of the GN loop (env LDSO_B200_KTIME=1), printed at destroy
    bool ktime = false;
    struct KT { const char *name; cudaEvent_t a, b; };
    std::vector<KT> kt;
    void kt_begin(const char *name) {
        if (!ktime) return;
        KT k; k.name = name;
        cudaEventCreate(&k.a); cudaEventCreate(&k.b);
        cudaEventRecord(k.a, stream);
        kt.push_back(k);
    }
    void kt_end() { if (ktime) cudaEventRecord(kt.back().b, stream); }

    int fail(int code, const char *msg) { err = msg; return code; }
    int fail_cuda(cudaError_t e, const char *call, const char *file, int line) {
        char buf[512];
        snprintf(buf, sizeof(buf), "CUDA error %s (%s) at %s:%d in %s", cudaGetErrorName(e), cudaGetErrorString(e), file, line, call);
        err = buf;
        return LDSO_B200_ERR_CUDA;
    }
};

// Every cached read-back (pinned mirror, solution staging, queued prefetch) is stale once device state may have changed.
inline void invalidate_results(ldso_b200_ctx *c) {
    c->mirror_valid = false; c->mirror_full_valid = false; c->sol_valid = false; c->results_inflight = false;
}

#define LAUNCH_CHECK(c)                                            \
    do {                                                           \
        (c)->launches++;                                           \
        invalidate_results(c);                                     \
        cudaError_t e__ = cudaGetLastError();                      \
        if (e__ != cudaSuccess) return (c)->fail_cuda(e__, "kernel launch", __FILE__, __LINE__); \
    } while (0)

#define RET_IF(x) do { int rc__ = (x); if (rc__) return rc__; } while (0)

// Copies on the context's stream. h2d skips an empty copy, d2h a null destination (an output the caller did not ask for).
inline int h2d(ldso_b200_ctx *c, void *dst, const void *src, size_t bytes) {
    if (bytes) CUDA_CHECK_RET(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return LDSO_B200_OK;
}
inline int d2h(ldso_b200_ctx *c, void *dst, const void *src, size_t bytes) {
    if (dst) CUDA_CHECK_RET(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    return LDSO_B200_OK;
}

// Byte offsets of the arrays of one device block, each aligned to 256 bytes: take() every array, allocate (or reserve) off
// bytes once, then turn the offsets into pointers.
struct Arena {
    size_t off = 0;
    size_t take(size_t bytes) { size_t o = off; off += (bytes + 255) & ~(size_t) 255; return o; }
};

// api_context.cu
int make_images_impl(ldso_b200_ctx *c, int slot, const float *color, bool wait_copy);
int reserve_scratch(ldso_b200_ctx *c, size_t bytes);      // c->scr.buf holds at least bytes, contents undefined
// api_ba.cu
void ba_set_kernel_attributes();
void free_window(ldso_b200_ctx *c);
int build_derived(ldso_b200_ctx *c);      // work items, newest-frame slots, partial buffers: need both the window and nF
int flush_select(ldso_b200_ctx *c);       // run a deferred setNewFrameEnergyTH select (fused loop)
int wait_results(ldso_b200_ctx *c);       // wait for a queued prefetch_results and mark its staging valid
// api_tracker.cu
bool tracker_alloc(ldso_b200_ctx *c);     // the tracker's fixed-size device buffers (create)
