// ldso_b200 C ABI implementation (include/ldso_b200.h), pose graph: posegraph_optimize.
#include "context.h"
#include "posegraph.cuh"

// ---------------------------------------------------------------------------------------------- pose graph
// Map::runPoseGraphOptimization (src/Map.cc:75-165): g2o Gauss-Newton over VertexSim3 / EdgeSim3 with numeric Jacobians, `iterations`
// rounds (25 in the reference), vertex `fixed` held (the current keyframe). The linear system of a round is solved by block-Jacobi
// preconditioned conjugate gradients to a relative residual of pcg_tol (g2o factorises it; both are exact solves of the same normal
// equations up to pcg_tol). Poses in / out as Sim3 = quaternion (w, x, y, z) with norm = scale + translation (Sophus' storage).
extern "C" int ldso_b200_posegraph_optimize(ldso_b200_ctx *c, int nV, double *q4, double *t3, int nE, const int32_t *ei, const int32_t *ej,
                                            const double *mq4, const double *mt3, const double *info49, int fixed, int iterations,
                                            double pcg_tol, int pcg_max_iter, double *chi2_out, int *pcg_iterations_total) {
    if (!c || nV < 2 || nE < 1 || !q4 || !t3 || !ei || !ej || !mq4 || !mt3 || !info49 || iterations < 0) return LDSO_B200_ERR_ARG;
    if (fixed < 0 || fixed >= nV) return c->fail(LDSO_B200_ERR_ARG, "fixed vertex out of range");
    for (int e = 0; e < nE; e++) if (ei[e] < 0 || ei[e] >= nV || ej[e] < 0 || ej[e] >= nV || ei[e] == ej[e]) return c->fail(LDSO_B200_ERR_ARG, "edge vertex index out of range");
    cudaSetDevice(c->device);
    // incidence lists (vertex -> edge * 2 + side), edge order
    std::vector<int> ib(nV + 1, 0), inc(2 * (size_t) nE);
    for (int e = 0; e < nE; e++) { ib[ei[e] + 1]++; ib[ej[e] + 1]++; }
    for (int v = 0; v < nV; v++) ib[v + 1] += ib[v];
    { std::vector<int> pos(ib.begin(), ib.end() - 1); for (int e = 0; e < nE; e++) { inc[pos[ei[e]]++] = 2 * e; inc[pos[ej[e]]++] = 2 * e + 1; } }
    const int nbv = (nV + PG_WARPS - 1) / PG_WARPS, nbe = (nE + PG_WARPS - 1) / PG_WARPS;
    // one device block
    Arena A;
    const size_t o_q = A.take(32 * (size_t) nV), o_t = A.take(24 * (size_t) nV), o_ei = A.take(4 * (size_t) nE), o_ej = A.take(4 * (size_t) nE),
                 o_mq = A.take(32 * (size_t) nE), o_mt = A.take(24 * (size_t) nE), o_info = A.take(392 * (size_t) nE), o_Hii = A.take(392 * (size_t) nE),
                 o_Hij = A.take(392 * (size_t) nE), o_Hjj = A.take(392 * (size_t) nE), o_bi = A.take(56 * (size_t) nE), o_bj = A.take(56 * (size_t) nE),
                 o_chi = A.take(8 * (size_t) nE), o_ib = A.take(4 * ((size_t) nV + 1)), o_inc = A.take(8 * (size_t) nE), o_D = A.take(392 * (size_t) nV),
                 o_Di = A.take(392 * (size_t) nV), o_b = A.take(56 * (size_t) nV), o_x = A.take(56 * (size_t) nV), o_r = A.take(56 * (size_t) nV),
                 o_z = A.take(56 * (size_t) nV), o_p0 = A.take(56 * (size_t) nV), o_p1 = A.take(56 * (size_t) nV), o_Ap = A.take(56 * (size_t) nV),
                 o_part = A.take(8 * (size_t) std::max(nbv, nbe)), o_scal = A.take(64), o_cnt = A.take(16);
    char *B = nullptr;
    CUDA_CHECK_RET(c, cudaMalloc(&B, A.off));
    struct Free { char *p; ~Free() { if (p) cudaFree(p); } } guard{B};
    CUDA_CHECK_RET(c, cudaMemsetAsync(B, 0, A.off, c->stream));
    RET_IF(h2d(c, B + o_q, q4, 32 * (size_t) nV)); RET_IF(h2d(c, B + o_t, t3, 24 * (size_t) nV));
    RET_IF(h2d(c, B + o_ei, ei, 4 * (size_t) nE)); RET_IF(h2d(c, B + o_ej, ej, 4 * (size_t) nE));
    RET_IF(h2d(c, B + o_mq, mq4, 32 * (size_t) nE)); RET_IF(h2d(c, B + o_mt, mt3, 24 * (size_t) nE)); RET_IF(h2d(c, B + o_info, info49, 392 * (size_t) nE));
    RET_IF(h2d(c, B + o_ib, ib.data(), 4 * ((size_t) nV + 1))); RET_IF(h2d(c, B + o_inc, inc.data(), 8 * (size_t) nE));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));      // pageable sources
    PgGraph g;
    g.nV = nV; g.nE = nE; g.fixed = fixed;
    g.q = (double *) (B + o_q); g.t = (double *) (B + o_t); g.ei = (const int *) (B + o_ei); g.ej = (const int *) (B + o_ej);
    g.mq = (const double *) (B + o_mq); g.mt = (const double *) (B + o_mt); g.info = (const double *) (B + o_info);
    g.Hii = (double *) (B + o_Hii); g.Hij = (double *) (B + o_Hij); g.Hjj = (double *) (B + o_Hjj); g.bi = (double *) (B + o_bi); g.bj = (double *) (B + o_bj);
    g.chi2e = (double *) (B + o_chi); g.inc_begin = (const int *) (B + o_ib); g.inc = (const int *) (B + o_inc);
    g.D = (double *) (B + o_D); g.Dinv = (double *) (B + o_Di); g.b = (double *) (B + o_b); g.x = (double *) (B + o_x); g.r = (double *) (B + o_r);
    g.z = (double *) (B + o_z); g.p0 = (double *) (B + o_p0); g.p1 = (double *) (B + o_p1); g.Ap = (double *) (B + o_Ap);
    g.part = (double *) (B + o_part); g.scal = (double *) (B + o_scal); g.counter = (unsigned *) (B + o_cnt);
    int total_cg = 0;
    const int chunk = 10;
    for (int it = 0; it <= iterations; it++) {
        k_pg_linearize<<<nbe, 32 * PG_WARPS, 0, c->stream>>>(g);
        LAUNCH_CHECK(c);
        k_pg_chi2<<<1, 256, 0, c->stream>>>(g, g.scal + 5);
        LAUNCH_CHECK(c);
        if (chi2_out) RET_IF(d2h(c, chi2_out + it, g.scal + 5, 8));
        if (it == iterations) break;
        k_pg_assemble<<<nbv, 32 * PG_WARPS, 0, c->stream>>>(g);
        LAUNCH_CHECK(c);
        double rz0 = 0.0, rz = 0.0;
        RET_IF(d2h(c, &rz0, g.scal, 8));
        CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
        rz = rz0;
        int k = 0;
        while (k < pcg_max_iter && rz > pcg_tol * pcg_tol * rz0 && rz0 > 0.0) {
            for (int j = 0; j < chunk && k < pcg_max_iter; j++, k++) {
                double *pin = (k & 1) ? g.p0 : g.p1, *pout = (k & 1) ? g.p1 : g.p0;
                k_pg_cg_a<<<nbv, 32 * PG_WARPS, 0, c->stream>>>(g, pin, pout, k == 0 ? 1 : 0);
                k_pg_cg_b<<<nbv, 32 * PG_WARPS, 0, c->stream>>>(g, pout);
                c->launches += 2;
            }
            RET_IF(d2h(c, &rz, g.scal, 8));
            CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
            if (!(rz == rz)) return c->fail(LDSO_B200_ERR_STATE, "pose graph: the normal equations are not positive definite (CG broke down)");
        }
        total_cg += k;
        k_pg_update<<<(nV + 127) / 128, 128, 0, c->stream>>>(g);
        LAUNCH_CHECK(c);
    }
    RET_IF(d2h(c, q4, g.q, 32 * (size_t) nV));
    RET_IF(d2h(c, t3, g.t, 24 * (size_t) nV));
    CUDA_CHECK_RET(c, cudaStreamSynchronize(c->stream));
    { cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) return c->fail_cuda(e__, "pose graph kernels", __FILE__, __LINE__); }
    if (pcg_iterations_total) *pcg_iterations_total = total_cg;
    return LDSO_B200_OK;
}

