// K2a (fold per-item partials in double), K2b (stitch through the adjoints + newest-frame energy threshold),
// K3 (assemble, scaled LDLT solve, orthogonalize, frame/calib step, frame-pair precalc) and the small
// piecewise kernels (applyRes, resubstitute/step on points).
#pragma once
#include "common.cuh"
#include "se3_math.cuh"
#include "ba_types.h"

// ---------------------------------------------------------------------------------------------------------
// K2a: red[h][e] = sum over the work items of host h of partial[item][e], in double
// (the reference casts its per-thread float accumulators to double before summing them,
//  AccumulatedTopHessian.cc:215-219, AccumulatedSCHessian.cc:78-83,101-105).
// The last block folds the per-item scalar statistics.
__device__ __forceinline__ void dbg_span(long long *slot_min_max, bool end) {
#ifdef LDSO_B200_PROFILE
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    if (!end) atomicMin((unsigned long long *) slot_min_max, gt);
    else atomicMax((unsigned long long *) (slot_min_max + 1), gt);
#endif
}
#define K2A_THREADS 512
#define K2A_SLICES (K2A_THREADS / 64)     // 8 threads share one output element, each folds every 8th work item
__global__ void __launch_bounds__(K2A_THREADS) k2a_reduce(DevWindow d, WinState *ws, int full, int multi) {
    pdl_launch_dependents();
    // before pdl_wait: what is constant for the window (frame count, the hosts' work-item ranges) -- two dependent L2 round trips
    // that would otherwise sit between the wait and the first partial load
    const int nF = ws->nF;
    const int el = threadIdx.x & 63, q = threadIdx.x >> 6;
    const int g = blockIdx.x * 64 + el;
    int pre_i0 = 0, pre_i1 = 0;
    if (full && blockIdx.x != gridDim.x - 1 && g < MAXF * PART_USED && g / PART_USED < nF) {
        pre_i0 = d.host_item_begin[g / PART_USED]; pre_i1 = d.host_item_begin[g / PART_USED + 1];
    }
    pdl_wait();                      // everything below reads what K1 just wrote
    if (threadIdx.x == 0) dbg_span(&ws->dbg[16], false);
    if (blockIdx.x == gridDim.x - 1) {
        // stats: warp w (<4) reduces stat w over all items
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        if (w < 4) {
            double s = 0.0;
            for (int i = lane; i < d.nItems; i += 32) s += d.item_stats[4 * i + w];
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) {
                d.red[RED_STATS + w] = s;
                if (!multi) {     // single GPU: publish now; multi GPU: K2b publishes after the all-reduce
                    if (w == 0) ws->energy = s;
                    if (w == 1) ws->resInA = (int) (s + 0.5);
                    if (w == 2) ws->sumNID = (float) s;
                    if (w == 3) ws->numID = (float) s;
                }
            }
        }
        { if (threadIdx.x == 0) dbg_span(&ws->dbg[16], true); return; }
    }
    if (!full) return;
    // 64 consecutive output elements per CTA; slice q of 8 folds items i0+q, i0+q+8, ... with all of its loads in
    // flight at once (the fold is a chain of L2 round trips otherwise); the 8 slice sums are added in a fixed order.
    __shared__ double part[K2A_SLICES][64];
    double s = 0.0;
    if (g < MAXF * PART_USED) {
        const int h = g / PART_USED, e = g - h * PART_USED;
        if (h < nF) {
            const int i0 = pre_i0, i1 = pre_i1;
            const float *p = d.partials + (size_t) (i0 + q) * PART_STRIDE + e;
            int i = i0 + q;
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
            for (; i + 3 * K2A_SLICES < i1; i += 4 * K2A_SLICES, p += 4 * K2A_SLICES * PART_STRIDE) {
                const float v0 = p[0], v1 = p[K2A_SLICES * PART_STRIDE], v2 = p[2 * K2A_SLICES * PART_STRIDE], v3 = p[3 * K2A_SLICES * PART_STRIDE];
                s0 += (double) v0; s1 += (double) v1; s2 += (double) v2; s3 += (double) v3;
            }
            float v0 = 0.f, v1 = 0.f, v2 = 0.f;
            if (i < i1) v0 = p[0];
            if (i + K2A_SLICES < i1) v1 = p[K2A_SLICES * PART_STRIDE];
            if (i + 2 * K2A_SLICES < i1) v2 = p[2 * K2A_SLICES * PART_STRIDE];
            s0 += (double) v0; s1 += (double) v1; s2 += (double) v2;
            s = (s0 + s1) + (s2 + s3);
        }
    }
    part[q][el] = s;
    __syncthreads();
    if (q == 0 && g < MAXF * PART_USED) {
        double t = part[0][el];
#pragma unroll
        for (int k = 1; k < K2A_SLICES; k++) t += part[k][el];
        d.red[g] = t;
    }
    if (threadIdx.x == 0) dbg_span(&ws->dbg[16], true);
}

// ---------------------------------------------------------------------------------------------------------
// K2r: the exchange step of the sharded Gauss-Newton iteration as ONE kernel over NVLink peer memory (no NCCL call, no host
// round trip): a push-based one-shot all-reduce of the reduced buffer with flag-in-data slots. Every rank owns an inbox
// [2 parities][8 senders][n] of 16-byte slots {lo32, tag, hi32, tag}. The thread that owns element g (1) writes its value,
// tagged with the exchange number, straight into the inbox of every peer (two 8-byte stores per slot, each atomic over
// NVLink -- no fence, no separate flag), then (2) polls its OWN inbox (local memory) until the slots of all peers carry
// this exchange's tag, and (3) adds the contributions in RANK ORDER (identical bits on every rank) into the buffer the
// stitch kernel reads. Cost: one one-way NVLink store latency plus local polling. The inbox is double-buffered by parity:
// a sender reuses a slot two exchanges later, which it cannot reach before this rank has sent the exchange in between,
// i.e. after this rank finished reading the current one.
#define K2R_THREADS 256
__device__ __forceinline__ void k2r_push(uint4 *dst, double v, unsigned e) {
    // ONE 16-byte store per slot: a warp's 32 slots leave as four 128-byte NVLink writes instead of 64 8-byte ones. A torn
    // delivery (8 + 8 bytes) is caught by the reader, which accepts a slot only when BOTH tags carry this exchange's number.
    const unsigned lo = (unsigned) __double2loint(v), hi = (unsigned) __double2hiint(v);
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(lo), "r"(e), "r"(hi), "r"(e) : "memory");
}
__device__ __forceinline__ double k2r_poll(const uint4 *src, unsigned e, bool &late) {
    unsigned a, f0, c, f1;
    int spins = 0;
    do {
        asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(a), "=r"(f0), "=r"(c), "=r"(f1) : "l"(src) : "memory");
    } while ((f0 != e || f1 != e) && ++spins < (1 << 24));          // ~ seconds; never hang the GPU
    if (f0 != e || f1 != e) late = true;
    return __hiloint2double((int) c, (int) a);
}
// world <= 2: one-shot exchange (every rank pushes its whole buffer to the peer, sums in rank order).
// world  > 2: reduce-scatter + all-gather inside the same kernel: element g belongs to rank g / len; every rank pushes its value of g
// to the OWNER only; the owner's thread g sums the contributions in rank order and pushes the total to everybody (second inbox
// region). Per rank 2 n (world-1)/world slots leave instead of n (world-1): 4x fewer bytes at 8 GPUs for one more NVLink hop.
// Every rank ends with the same bits in both schemes. A thread only ever waits for the thread of the same element on another rank.
__global__ void __launch_bounds__(K2R_THREADS) k2r_peer_allreduce(DevWindow d, PeerExchange px) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ int s_epoch;
    const int tid = threadIdx.x;
    if (tid == 0) s_epoch = *((volatile int *) px.epoch) + 1;
    __syncthreads();
    const unsigned e = (unsigned) s_epoch;
    const int par = (int) (e & 1u);
    const int g = blockIdx.x * K2R_THREADS + tid;
    const int n = px.n_doubles;
    if (g < n) {
        const double mine = d.red[g];
        bool late = false;
        double s = 0.0;
        if (!px.two_hop) {
            for (int p = 0; p < px.world; p++)
                if (p != px.rank) k2r_push(px.inbox[p] + ((size_t) (par * K2R_MAX_PEERS + px.rank) * n + g), mine, e);
            for (int r = 0; r < px.world; r++)
                s += (r == px.rank) ? mine : k2r_poll(px.inbox[px.rank] + ((size_t) (par * K2R_MAX_PEERS + r) * n + g), e, late);
        } else {
            const int len = (n + px.world - 1) / px.world, owner = g / len;
            const size_t regB = (size_t) 2 * K2R_MAX_PEERS * n;           // the all-gather inbox region behind the reduce-scatter one
            if (owner != px.rank) {
                k2r_push(px.inbox[owner] + ((size_t) (par * K2R_MAX_PEERS + px.rank) * n + g), mine, e);
                s = k2r_poll(px.inbox[px.rank] + regB + (size_t) par * n + g, e, late);
            } else {
                for (int r = 0; r < px.world; r++)
                    s += (r == px.rank) ? mine : k2r_poll(px.inbox[px.rank] + ((size_t) (par * K2R_MAX_PEERS + r) * n + g), e, late);
                for (int p = 0; p < px.world; p++)
                    if (p != px.rank) k2r_push(px.inbox[p] + regB + (size_t) par * n + g, s, e);
            }
        }
        px.out[g] = s;
        if (late) *px.error = 1;
    }
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(px.done, 1u) == gridDim.x - 1) { *px.done = 0u; *px.epoch = (int) e; }
    }
}

// ---------------------------------------------------------------------------------------------------------
// packed index of element (r,c) of the symmetric 13x13 AccumulatorApprox block [C(4)|xi(6)|ab(2)|r(1)]
__device__ __forceinline__ int packed13(int r, int c) {
    if (r > c) { int t = r; r = c; c = t; }
    if (c < 10) return r * 10 - (r * (r - 1)) / 2 + (c - r);
    if (r < 10) return 55 + 3 * r + (c - 10);
    return 85 + ((r == 10) ? (c - 10) : (r == 11) ? 3 + (c - 11) : 5);
}

// K2b: one CTA per 8x8 output block (a,b) of H_A and H_sc, nF CTAs for the calibration rows + b, one CTA for
// the calibration corner, and a last CTA for FullSystem::setNewFrameEnergyTH (FullSystem.cc:1762-1793).
// Formulas: AccumulatedTopHessian.cc:221-240 + .h:95-104 and AccumulatedSCHessian.cc:85-118 + .h:93-97,
// regrouped by output block so that no two CTAs write the same element (deterministic, no atomics).
#define K2B_THREADS 512
#define K2B_NSLOT (K2B_THREADS / 64)
#define K2B_SELCAP 30720         // newest-frame energies kept in shared memory by the select CTA (120 KB of the CTA's dynamic smem)
// staged 8x8 matrices use a row stride of 10 doubles: rows then start 20 banks apart, so both the "one row per lane
// group" and the "transposed operand" access patterns of the triple products are bank-conflict free and stay 16-byte
// aligned (with the natural stride of 8 every other row maps to the same banks: 4-way conflicts on every operand load)
#define K2B_RS 10
#define K2B_MS (8 * K2B_RS)
#define K2B_M(q, r, c) ((q) * K2B_MS + (r) * K2B_RS + (c))
#define K2B_NMAT (7 * MAXF + MAXF * MAXF + 2 * MAXF + MAXF + MAXF + 2 * MAXF + 2)
#define K2B_SMEM_DOUBLES (K2B_NMAT * K2B_MS + 2 * MAXF * 64 + K2B_NSLOT * 128)
#define K2B_SMEM_BYTES (K2B_SMEM_DOUBLES * sizeof(double))
__device__ __forceinline__ double top_elem(const double *red, int h, int t, int r13, int c13) {
    return red[h * PART_USED + PART_TOP + t * 96 + packed13(r13, c13)];
}

// FullSystem::setNewFrameEnergyTH (FullSystem.cc:1762-1793): the exact k-th order statistic of the newest frame's residual energies
// (radix select, keys in shared memory). Called by all K2B_THREADS threads of ONE CTA: the last CTA of k2b_stitch (prologue, piecewise
// API) or the second CTA of k3_solve_step, where it runs beside the solver instead of in front of it (the threshold is first read by
// the next linearisation).
__device__ void k2_select_body(const double *red, int N, WinState *ws, double *sk2, long long *dbg) {
    __shared__ unsigned hist[256];
    __shared__ unsigned hist_w[K2B_THREADS / 32][256];     // per-warp histograms (no cross-warp contention on the hot bins)
    __shared__ unsigned sel_prefix, sel_k, sel_count;
    const int tid = threadIdx.x, nF = ws->nF;

        PROF_ONLY(if (tid == 0) dbg[12] = clock64();)
                // settings (constant): requested now, consumed after the passes
        const float set_thn = ws->S.frameEnergyTHN, set_fac = ws->S.frameEnergyTHFacMedian, set_cw = ws->S.frameEnergyTHConstWeight,
                    set_ow = ws->S.overallEnergyTHWeight;
        const double *vals = red + RED_SELECT;
        unsigned *skey = (unsigned *) sk2;            // float bit patterns of the valid energies (0x80000000 = excluded)
        const bool insm = N <= K2B_SELCAP;
        if (tid == 0) { sel_count = 0; sel_prefix = 0; }
        __syncthreads();
        unsigned cnt = 0;
        for (int i0 = tid; i0 < N; i0 += 8 * K2B_THREADS) {      // 8 independent loads per trip (the values come from L2 / HBM)
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) { const int i = i0 + u * K2B_THREADS; v[u] = (i < N) ? vals[i] : -1.0; }
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int i = i0 + u * K2B_THREADS;
                const bool ok = v[u] >= 0.0;
                if (insm && i < N) skey[i] = ok ? __float_as_uint((float) v[u]) : 0x80000000u;
                cnt += ok;
            }
        }
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if ((tid & 31) == 0) atomicAdd(&sel_count, cnt);
        __syncthreads();
        const unsigned m = sel_count;
        float th;
        if (m == 0) {
            th = 12 * 12 * LDSO_B200_PATTERN;
        } else {
            if (tid == 0) sel_k = (unsigned) (int) (set_thn * (float) m);
            __syncthreads();
            for (int pass = 3; pass >= 0; pass--) {
                for (int i = tid; i < 256 * (K2B_THREADS / 32); i += K2B_THREADS) (&hist_w[0][0])[i] = 0;
                __syncthreads();
                const unsigned pref = sel_prefix;
                const unsigned himask = (pass == 3) ? 0u : (0xffffffffu << (8 * (pass + 1)));
                // energies of one frame share their leading bytes: aggregate equal bins inside the warp first
                // (one shared-memory atomic per distinct bin per warp instead of 32 serialised ones)
                for (int i0 = tid; i0 < ((N + 31) & ~31); i0 += 4 * K2B_THREADS) {     // 4 independent keys per trip
                    unsigned key[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const int i = i0 + u * K2B_THREADS;
                        key[u] = 0x80000000u;
                        if (i < N) {
                            if (insm) key[u] = skey[i];
                            else { const double v = vals[i]; key[u] = (v >= 0.0) ? __float_as_uint((float) v) : 0x80000000u; }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        const bool act = (key[u] != 0x80000000u) && ((key[u] & himask) == pref);
                        const unsigned bin = act ? ((key[u] >> (8 * pass)) & 0xffu) : 256u;
                        // equal bins are aggregated inside the warp first (one atomic per distinct bin), on the warp's own histogram
                        const unsigned mm = __match_any_sync(0xffffffffu, bin);
                        if (act && (tid & 31) == __ffs(mm) - 1) atomicAdd(&hist_w[tid >> 5][bin], (unsigned) __popc(mm));
                    }
                }
                __syncthreads();
                if (tid < 256) {
                    unsigned t = 0;
#pragma unroll
                    for (int wv = 0; wv < K2B_THREADS / 32; wv++) t += hist_w[wv][tid];
                    hist[tid] = t;
                }
                __syncthreads();
                if (tid < 32) {
                    // warp 0: lane owns 8 consecutive bins; find the bin holding rank sel_k
                    unsigned hq[8], loc = 0;
#pragma unroll
                    for (int q = 0; q < 8; q++) { hq[q] = hist[8 * tid + q]; loc += hq[q]; }
                    unsigned incl = loc;
                    for (int o = 1; o < 32; o <<= 1) {
                        const unsigned v = __shfl_up_sync(0xffffffffu, incl, o);
                        if (tid >= o) incl += v;
                    }
                    const unsigned excl = incl - loc;
                    const unsigned k0 = sel_k;
                    const bool mine = (k0 >= excl) && (k0 < incl);
                    __syncwarp();
                    if (mine) {
                        unsigned k = k0 - excl, bin = 8 * tid;
                        bool found = false;
#pragma unroll
                        for (int q = 0; q < 8; q++) {
                            if (!found) {
                                if (k < hq[q]) found = true;
                                else { k -= hq[q]; bin++; }
                            }
                        }
                        sel_k = k;
                        sel_prefix = pref | (bin << (8 * pass));
                    }
                }
                __syncthreads();
            }
            const float nthElement = sqrtf(__uint_as_float(sel_prefix));
            th = nthElement * set_fac;
            th = 26.0f * set_cw + th * (1 - set_cw);
            th = th * th;
            th *= set_ow * set_ow;
        }
        if (tid == 0) { ws->frameEnergyTH[nF - 1] = th; PROF_ONLY(dbg[13] = clock64();) }
    }

// 1x4 register tiles of the 8x8 triple products (operands staged in shared memory with row stride K2B_RS): one 8-term FMA chain per
// output, ascending index -- the same sums as one output per thread, with 20 16-byte loads per 32 FMAs instead of 64 8-byte loads
// (one output per thread is bound by shared-memory load issue, not by the FP64 pipe).
// o[c] = sum_i Arow[i] * D[i][c0 + c]        (A * D;  Dc = &D[0][c0])
__device__ __forceinline__ void k2b_tile_AD(const double *Arow, const double *Dc, double o[4]) {
    double av[8];
#pragma unroll
    for (int i = 0; i < 8; i += 2) { const double2 a = *(const double2 *) (Arow + i); av[i] = a.x; av[i + 1] = a.y; }
    o[0] = o[1] = o[2] = o[3] = 0.0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const double2 d01 = *(const double2 *) (Dc + i * K2B_RS), d23 = *(const double2 *) (Dc + i * K2B_RS + 2);
        o[0] += av[i] * d01.x; o[1] += av[i] * d01.y; o[2] += av[i] * d23.x; o[3] += av[i] * d23.y;
    }
}
// o[c] = sum_j Arow[j] * B[c0 + c][j]        (A * B^T;  Br = &B[c0][0])
__device__ __forceinline__ void k2b_tile_ABt(const double *Arow, const double *Br, double o[4]) {
    double av[8];
#pragma unroll
    for (int i = 0; i < 8; i += 2) { const double2 a = *(const double2 *) (Arow + i); av[i] = a.x; av[i + 1] = a.y; }
#pragma unroll
    for (int c = 0; c < 4; c++) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < 8; j += 2) { const double2 b = *(const double2 *) (Br + c * K2B_RS + j); s += av[j] * b.x; s += av[j + 1] * b.y; }
        o[c] = s;
    }
}
__device__ __forceinline__ void k2b_store4(double *dst, const double o[4]) {      // dst 16-byte aligned
    *(double2 *) dst = make_double2(o[0], o[1]);
    *(double2 *) (dst + 2) = make_double2(o[2], o[3]);
}
#define K2B_LAMBDA 1e-5        // SOLVER_FIX_LAMBDA (EnergyFunctional.cc:243)
__device__ __forceinline__ double k2b_delta(const WinState *ws, int c) {      // getStitchedDeltaF (EnergyFunctional.h:178-184)
    return (c < CPARS) ? (double) ws->calib.cDeltaF[c] : ws->fr[(c - CPARS) >> 3].delta[(c - CPARS) & 7];
}
__global__ void __launch_bounds__(K2B_THREADS) k2b_stitch(DevWindow d, WinState *ws, SolveBufs sb, int do_stitch, int do_select, int do_assemble) {
    pdl_launch_dependents();
    const int nF = ws->nF, n = ws->n;
    const int tid = threadIdx.x;
    const double *red = d.red;
    const int nBlocks = nF * nF;
    if ((int) blockIdx.x < nBlocks) {
        if (!do_stitch) return;
        // ---- 8x8 frame block (a,b) of H_A and H_sc. All operands (adjoints, D blocks, top blocks) are first staged
        // in shared memory with one burst of independent loads; the triple products then run from shared memory.
        extern __shared__ __align__(16) double sk2[];
        double *sAHa = sk2;                    // [nF] adHost[a + nF*j]
        double *sATa = sAHa + MAXF * K2B_MS;   // [nF] adTarget[i + nF*a]
        double *sATb = sATa + MAXF * K2B_MS;   // [nF] adTarget[i + nF*b]
        double *sAHb = sATb + MAXF * K2B_MS;   // [nF] adHost[b + nF*k]
        double *sD1 = sAHb + MAXF * K2B_MS;    // [nF] D_i[a,b]
        double *sD2 = sD1 + MAXF * K2B_MS;     // [nF] D_b[a,k]
        double *sD3 = sD2 + MAXF * K2B_MS;     // [nF] D_a[j,b]
        double *sD4 = sD3 + MAXF * K2B_MS;     // [nF*nF] D_a[j,k]  (a == b only)
        double *sM = sD4 + MAXF * MAXF * K2B_MS;   // [2*nF] top blocks
        double *sZ = sM + 2 * MAXF * K2B_MS;   // [nF]  AT_ia * D_i[a,b]
        double *sX = sZ + MAXF * K2B_MS;       // [nF]  sum_j AH_aj * D_a[j,k]
        double *sT = sX + MAXF * K2B_MS;       // [2*nF] L_q * M_q
        double *sY2 = sT + 2 * MAXF * K2B_MS;  // sum_k D_b[a,k] * AH_bk^T
        double *sY3 = sY2 + K2B_MS;            // sum_j AH_aj * D_a[j,b]
        double *sP = sY3 + K2B_MS;             // [2][MAXF][64] per-frame partial products of Y2 / Y3
        // (K2B_NSLOT * 128 more doubles follow: the allocation also has to hold the select CTA's K2B_SELCAP keys)
        const int a = blockIdx.x % nF, b = blockIdx.x / nF;
        const bool diag = (a == b);
        // the marginalisation-prior element this thread will add in the epilogue: issue the load now
        double hm_pre = 0.0;
        if (do_assemble && tid < 64) hm_pre = sb.HM[(size_t) (CPARS + 8 * b + (tid & 7)) * n + CPARS + 8 * a + (tid >> 3)];
        PROF_ONLY(if (blockIdx.x == 0 && tid == 0) d.dbg[8] = clock64();)
        // -------- stage
        for (int o = tid; o < nF * 64; o += K2B_THREADS) {      // adjoints: constant for the window, staged before pdl_wait
            const int q = o >> 6, e = o & 63, m = K2B_M(q, e >> 3, e & 7);
            sAHa[m] = ws->adHost[a + nF * q][e];
            sATa[m] = ws->adTarget[q + nF * a][e];
            sATb[m] = ws->adTarget[q + nF * b][e];
            sAHb[m] = ws->adHost[b + nF * q][e];
        }
        pdl_wait();
        if (tid == 0) dbg_span(&ws->dbg[18], false);
        for (int o = tid; o < nF * 64; o += K2B_THREADS) {
            const int q = o >> 6, e = o & 63, m = K2B_M(q, e >> 3, e & 7);
            sD1[m] = red[q * PART_USED + PART_D + (a * MAXF + b) * 64 + e];
            sD2[m] = red[b * PART_USED + PART_D + (a * MAXF + q) * 64 + e];
            sD3[m] = red[a * PART_USED + PART_D + (q * MAXF + b) * 64 + e];
        }
        if (diag) {
            for (int o = tid; o < nF * nF * 64; o += K2B_THREADS) {
                const int jk = o >> 6, e = o & 63, j = jk % nF, k = jk / nF;
                sD4[K2B_M(jk, e >> 3, e & 7)] = red[a * PART_USED + PART_D + (j * MAXF + k) * 64 + e];
            }
            for (int o = tid; o < 2 * nF * 64; o += K2B_THREADS) {
                const int q = o >> 6, e = o & 63, i = e >> 3, c = e & 7;
                sM[K2B_M(q, i, c)] = (q < nF) ? top_elem(red, a, q, 4 + i, 4 + c) : top_elem(red, q - nF, a, 4 + i, 4 + c);
            }
        } else {
            for (int o = tid; o < 2 * 64; o += K2B_THREADS) {
                const int q = o >> 6, e = o & 63, i = e >> 3, c = e & 7;
                sM[K2B_M(q, i, c)] = (q == 0) ? top_elem(red, a, b, 4 + i, 4 + c) : top_elem(red, b, a, 4 + i, 4 + c);
            }
        }
        __syncthreads();
        PROF_ONLY(if (blockIdx.x == 0 && tid == 0) d.dbg[9] = clock64();)
        // -------- stage A: left products. Every thread runs short (8-term) chains only; sums over frames are kept as
        // independent partial chains and folded in a fixed order.
        // On a diagonal block the 64-term X_k products dominate (32 k of the 53 k FMAs) and, one output per thread, they are bound by
        // shared-memory load issue (2 loads per FMA): warps 0-3 compute them in 1x4 register tiles (3 loads -- one of them 16 bytes --
        // per 4 FMAs, same summation order as before), the other 12 warps do the short products meanwhile.
        const int lt0 = diag ? tid - 128 : tid, ltn = diag ? K2B_THREADS - 128 : K2B_THREADS;      // thread index / count for the short products
        if (diag && tid < 128) {                                   // X_k = sum_j AH_aj * D_a[j,k]
            const int k = tid >> 4, r = (tid >> 1) & 7, c0 = (tid & 1) * 4;
            if (k < nF) {
                double acc[4] = {0.0, 0.0, 0.0, 0.0};
                for (int j = 0; j < nF; j++) {
                    double sj[4] = {0.0, 0.0, 0.0, 0.0};
                    const double *Ar = sAHa + K2B_M(j, r, 0), *Dm = sD4 + K2B_M(j + nF * k, 0, c0);
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const double av = Ar[i];
                        const double2 d01 = *(const double2 *) (Dm + i * K2B_RS), d23 = *(const double2 *) (Dm + i * K2B_RS + 2);
                        sj[0] += av * d01.x; sj[1] += av * d01.y; sj[2] += av * d23.x; sj[3] += av * d23.y;
                    }
                    if (j == 0) { acc[0] = sj[0]; acc[1] = sj[1]; acc[2] = sj[2]; acc[3] = sj[3]; }
                    else { acc[0] += sj[0]; acc[1] += sj[1]; acc[2] += sj[2]; acc[3] += sj[3]; }
                }
                double *Xo = sX + K2B_M(k, r, c0);
                *(double2 *) Xo = make_double2(acc[0], acc[1]);
                *(double2 *) (Xo + 2) = make_double2(acc[2], acc[3]);
            }
        }
        if (lt0 >= 0) {
            // the 8-term products as 1x4 tiles: tile u <-> (matrix q, row r, column half): [0,128) Z, [128,384) the per-frame terms of
            // Y2 / Y3, then T (2 nF matrices on a diagonal block, 2 otherwise)
            const int nTile = 3 * MAXF * 16 + (diag ? 2 * nF : 2) * 16;
            for (int u = lt0; u < nTile; u += ltn) {
                const int q = u >> 4, r = (u >> 1) & 7, c0 = (u & 1) * 4;
                double o4[4];
                if (q < MAXF) {                                          // Z_q = AT_qa * D_q[a,b]
                    if (q < nF) {
                        k2b_tile_AD(sATa + K2B_M(q, r, 0), sD1 + K2B_M(q, 0, c0), o4);
                        k2b_store4(sZ + K2B_M(q, r, c0), o4);
                    }
                } else if (q < 3 * MAXF) {
                    const int which = (q - MAXF) / MAXF, k = (q - MAXF) & (MAXF - 1);
                    o4[0] = o4[1] = o4[2] = o4[3] = 0.0;
                    if (k < nF) {
                        if (which == 0) k2b_tile_ABt(sD2 + K2B_M(k, r, 0), sAHb + K2B_M(k, c0, 0), o4);      // D_b[a,k] * AH_bk^T
                        else k2b_tile_AD(sAHa + K2B_M(k, r, 0), sD3 + K2B_M(k, 0, c0), o4);                   // AH_ak * D_a[k,b]
                    }
                    k2b_store4(sP + which * MAXF * 64 + k * 64 + r * 8 + c0, o4);
                } else {
                    const int t = q - 3 * MAXF;
                    const double *Lm;
                    if (diag) Lm = (t < nF) ? (sAHa + t * K2B_MS) : (sATa + (t - nF) * K2B_MS);               // T_t = L_t * M_t
                    else Lm = (t == 0) ? (sAHa + b * K2B_MS) : (sAHb + a * K2B_MS);                           // AH_ab*M_ab, AH_ba*M_ba
                    k2b_tile_AD(Lm + r * K2B_RS, sM + K2B_M(t, 0, c0), o4);
                    k2b_store4(sT + K2B_M(t, r, c0), o4);
                }
            }
        }
        __syncthreads();
        if (tid < 128) {                                             // fold the per-frame terms of Y2 / Y3
            const int which = tid >> 6, e = tid & 63;
            double s = sP[which * MAXF * 64 + e];
#pragma unroll
            for (int k = 1; k < MAXF; k++) s += sP[which * MAXF * 64 + k * 64 + e];
            (which ? sY3 : sY2)[K2B_M(0, e >> 3, e & 7)] = s;
        }
        __syncthreads();
        PROF_ONLY(if (blockIdx.x == 0 && tid == 0) d.dbg[10] = clock64();)
        // -------- stage B: right products as 1x4 tiles, 32 groups of 16 threads, one term of the sum per group (two for groups 16, 17):
        //   H_sc terms s: [0,8) Z_s AT_sb^T | 8: AT_ba Y2 | 9: Y3 AT_ab^T | [10,18) X_(s-10) AH_a(s-10)^T (diagonal blocks)      -> group s
        //   H_A  terms t: diagonal block: [0,8) T_t AH_at^T, [8,16) T_(nF+t-8) AT_(t-8)a^T; else 0: T_0 AT_ab^T, 1: (T_1 AT_ba^T)^T -> group 16+t
        // The partial 8x8 outputs go to the (now dead) D_a[j,k] staging area; invalid terms store zeros.
        double *sOS = sD4, *sOA = sD4 + 18 * 64;
        {
            const int g = tid >> 4, u = tid & 15, r = u >> 1, c0 = (u & 1) * 4;
            double o4[4];
            if (g < 18) {
                o4[0] = o4[1] = o4[2] = o4[3] = 0.0;
                if (g < MAXF) { if (g < nF) k2b_tile_ABt(sZ + K2B_M(g, r, 0), sATb + K2B_M(g, c0, 0), o4); }
                else if (g == MAXF) k2b_tile_AD(sATa + K2B_M(b, r, 0), sY2 + K2B_M(0, 0, c0), o4);
                else if (g == MAXF + 1) k2b_tile_ABt(sY3 + K2B_M(0, r, 0), sATb + K2B_M(a, c0, 0), o4);
                else if (diag && g - (MAXF + 2) < nF) k2b_tile_ABt(sX + K2B_M(g - (MAXF + 2), r, 0), sAHa + K2B_M(g - (MAXF + 2), c0, 0), o4);
                k2b_store4(sOS + g * 64 + r * 8 + c0, o4);
            }
            if (g >= 16) {
                const int t = g - 16;
                o4[0] = o4[1] = o4[2] = o4[3] = 0.0;
                if (diag) {
                    if ((t & (MAXF - 1)) < nF) {
                        const int q = (t < MAXF) ? t : nF + (t - MAXF);
                        const double *Rm = (t < MAXF) ? (sAHa + t * K2B_MS) : (sATa + (t - MAXF) * K2B_MS);
                        k2b_tile_ABt(sT + K2B_M(q, r, 0), Rm + c0 * K2B_RS, o4);
                    }
                } else if (t == 0) k2b_tile_ABt(sT + K2B_M(0, r, 0), sATb + K2B_M(a, c0, 0), o4);
                else if (t == 1) k2b_tile_ABt(sATa + K2B_M(b, r, 0), sT + K2B_M(1, c0, 0), o4);
                k2b_store4(sOA + t * 64 + r * 8 + c0, o4);
            }
        }
        __syncthreads();
        if (tid < 64) {
            const int e = tid, r = e >> 3, c = e & 7;
            double vA = 0.0, vS = 0.0;
#pragma unroll
            for (int q = 0; q < 18; q++) vS += sOS[q * 64 + e];
#pragma unroll
            for (int q = 0; q < 16; q++) vA += sOA[q * 64 + e];
            const int row = CPARS + 8 * a + r, col = CPARS + 8 * b + c;
            sb.H_A[(size_t) col * n + row] = vA;
            sb.H_sc[(size_t) col * n + row] = vS;
            if (do_assemble) {       // HFinal_top = HL + HM + HA, lastHS, damping, Schur part (EnergyFunctional.cc:283-291)
                double v = vA + hm_pre;
                if (row == col) v += ws->fr[a].prior[r];
                sb.HSg[(size_t) col * n + row] = v - vS;
                if (row == col) v *= (1.0 + K2B_LAMBDA);
                const double a0 = v - vS * (1.0 / (1.0 + K2B_LAMBDA));
                sb.A0g[(size_t) col * n + row] = a0;
                if (row == col) sb.dg[row] = a0;
            }
        }
        PROF_ONLY(if (blockIdx.x == 0 && tid == 0) d.dbg[11] = clock64();)
        { if (tid == 0) dbg_span(&ws->dbg[18], true); return; }
    }
    if ((int) blockIdx.x < nBlocks + nF) {
        if (!do_stitch) return;
        // ---- calibration rows of frame a and its b segments: 80 outputs, 8 lanes per output (lane <-> other frame),
        // every lane issues its 32 independent loads at once, then a 3-step shuffle fold.
        const int a = blockIdx.x - nBlocks;
        __shared__ double s_cal[80];
        pdl_wait();
        if (tid == 0) dbg_span(&ws->dbg[18], false);
        for (int o8 = tid; o8 < 80 * 8; o8 += K2B_THREADS) {
            const int o = o8 >> 3, t = o8 & 7;
            double s = 0.0;
            if (t < nF && t != a) {
                const double *AH = ws->adHost[a + nF * t], *AT = ws->adTarget[t + nF * a];
                if (o < 32) {                 // H_A[a, c]
                    const int r = o >> 2, c = o & 3;
                    for (int i = 0; i < 8; i++) s += AH[r * 8 + i] * top_elem(red, a, t, 4 + i, c) + AT[r * 8 + i] * top_elem(red, t, a, 4 + i, c);
                } else if (o < 40) {          // b_A[a]
                    const int r = o - 32;
                    for (int i = 0; i < 8; i++) s += AH[r * 8 + i] * top_elem(red, a, t, 4 + i, 12) + AT[r * 8 + i] * top_elem(red, t, a, 4 + i, 12);
                } else if (o < 72) {          // H_sc[a, c]
                    const int r = (o - 40) >> 2, c = (o - 40) & 3;
                    const double *Eat = red + a * PART_USED + PART_E + t * 32, *Eta = red + t * PART_USED + PART_E + a * 32;
                    for (int i = 0; i < 8; i++) s += AH[r * 8 + i] * Eat[i * 4 + c] + AT[r * 8 + i] * Eta[i * 4 + c];
                } else {                      // b_sc[a]
                    const int r = o - 72;
                    const double *Bat = red + a * PART_USED + PART_EB + t * 8, *Bta = red + t * PART_USED + PART_EB + a * 8;
                    for (int i = 0; i < 8; i++) s += AH[r * 8 + i] * Bat[i] + AT[r * 8 + i] * Bta[i];
                }
            }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            if (t == 0) {
                s_cal[o] = s;
                if (o < 32) {
                    const int r = o >> 2, c = o & 3;
                    sb.H_A[(size_t) c * n + (CPARS + 8 * a + r)] = s;
                    sb.H_A[(size_t) (CPARS + 8 * a + r) * n + c] = s;
                } else if (o < 40) sb.b_A[CPARS + 8 * a + (o - 32)] = s;
                else if (o < 72) {
                    const int r = (o - 40) >> 2, c = (o - 40) & 3;
                    sb.H_sc[(size_t) c * n + (CPARS + 8 * a + r)] = s;
                    sb.H_sc[(size_t) (CPARS + 8 * a + r) * n + c] = s;
                } else sb.b_sc[CPARS + 8 * a + (o - 72)] = s;
            }
        }
        if (do_assemble) {
            __syncthreads();
            if (tid < 32) {                    // the two mirrored elements (R,c) and (c,R): no diagonal here
                const int r = tid >> 2, c = tid & 3, R = CPARS + 8 * a + r;
                const double sA = s_cal[tid], sS = s_cal[40 + tid];
                const double v1 = sA + sb.HM[(size_t) c * n + R], v2 = sA + sb.HM[(size_t) R * n + c];
                sb.HSg[(size_t) c * n + R] = v1 - sS;
                sb.HSg[(size_t) R * n + c] = v2 - sS;
                sb.A0g[(size_t) c * n + R] = v1 - sS * (1.0 / (1.0 + K2B_LAMBDA));
                sb.A0g[(size_t) R * n + c] = v2 - sS * (1.0 / (1.0 + K2B_LAMBDA));
            } else if (tid >= 64 && tid < 128) {   // bFinal_top = bL + (bM + HM*delta) + bA - b_sc (:257,284), 8 lanes per row
                const int r = (tid - 64) >> 3, t = tid & 7, R = CPARS + 8 * a + r;
                double hd = 0.0;
                for (int c = t; c < n; c += 8) hd += sb.HM[(size_t) c * n + R] * k2b_delta(ws, c);
                hd += __shfl_xor_sync(0xffffffffu, hd, 1);
                hd += __shfl_xor_sync(0xffffffffu, hd, 2);
                hd += __shfl_xor_sync(0xffffffffu, hd, 4);
                if (t == 0) {
                    const FrameDev &f = ws->fr[a];
                    const double bl = f.prior[r] * f.delta_prior[r];
                    sb.bFg[R] = bl + (sb.bM[R] + hd) + s_cal[32 + r] - s_cal[72 + r];
                }
            }
        }
        { if (tid == 0) dbg_span(&ws->dbg[18], true); return; }
    }
    if ((int) blockIdx.x == nBlocks + nF) {
        if (!do_stitch) return;
        // ---- calibration corner: 20 outputs x 8 lanes (lane <-> host frame)
        pdl_wait();
        if (tid == 0) dbg_span(&ws->dbg[18], false);
        if (tid < 20 * 8) {
            const int o = tid >> 3, h = tid & 7;
            double sA = 0.0, sS = 0.0;
            if (h < nF) {
                if (o < 16) {
                    const int r = o >> 2, c = o & 3;
                    for (int t = 0; t < nF; t++) if (t != h) sA += top_elem(red, h, t, r, c);
                    sS = red[h * PART_USED + PART_HCC + r * 4 + c];
                } else {
                    const int r = o - 16;
                    for (int t = 0; t < nF; t++) if (t != h) sA += top_elem(red, h, t, r, 12);
                    sS = red[h * PART_USED + PART_BC + r];
                }
            }
            for (int m = 1; m < 8; m <<= 1) { sA += __shfl_xor_sync(0xffffffffu, sA, m); sS += __shfl_xor_sync(0xffffffffu, sS, m); }
            double hd = 0.0;
            if (do_assemble && o >= 16)      // (HM*delta)[r], the 8 lanes split the columns
                for (int c = h; c < n; c += 8) hd += sb.HM[(size_t) c * n + (o - 16)] * k2b_delta(ws, c);
            for (int m = 1; m < 8; m <<= 1) hd += __shfl_xor_sync(0xffffffffu, hd, m);
            if (h == 0) {
                if (o < 16) {
                    const int r = o >> 2, c = o & 3;
                    sb.H_A[(size_t) c * n + r] = sA;
                    sb.H_sc[(size_t) c * n + r] = sS;
                    if (do_assemble) {
                        double v = sA + sb.HM[(size_t) c * n + r];
                        if (r == c) v += ws->cPrior[r];
                        sb.HSg[(size_t) c * n + r] = v - sS;
                        if (r == c) v *= (1.0 + K2B_LAMBDA);
                        const double a0 = v - sS * (1.0 / (1.0 + K2B_LAMBDA));
                        sb.A0g[(size_t) c * n + r] = a0;
                        if (r == c) sb.dg[r] = a0;
                    }
                } else {
                    const int r = o - 16;
                    sb.b_A[r] = sA; sb.b_sc[r] = sS;
                    if (do_assemble) {
                        const double bl = ws->cPrior[r] * (double) ws->calib.cDeltaF[r];
                        sb.bFg[r] = bl + (sb.bM[r] + hd) + sA - sS;
                    }
                }
            }
        }
        { if (tid == 0) dbg_span(&ws->dbg[18], true); return; }
    }
    // ---- last CTA: exact k-th order statistic of the newest frame's residual energies (radix select)
    pdl_wait();
    if (tid == 0) dbg_span(&ws->dbg[18], false);
    if (tid == 0) {   // publish the (all-reduced) scalar statistics
        ws->energy = red[RED_STATS + 0];
        ws->resInA = (int) (red[RED_STATS + 1] + 0.5);
        ws->sumNID = (float) red[RED_STATS + 2];
        ws->numID = (float) red[RED_STATS + 3];
    }
    if (!do_select) return;
    {
        extern __shared__ __align__(16) double sk2[];
        k2_select_body(red, d.newest_total, ws, sk2, d.dbg);
    }
    if (tid == 0) dbg_span(&ws->dbg[18], true);
}

// ---------------------------------------------------------------------------------------------------------
// piecewise helpers
// PointFrameResidual::applyRes(true) on every active residual (Residuals.h:70-87)
__global__ void k_apply_res(DevWindow d) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.nR) return;
    if (d.res_lin[r]) return;
    if (d.res_state[r] == LDSO_B200_RES_OOB) return;
    const uint8_t ns = d.res_new_state[r];
    if (ns == LDSO_B200_RES_IN) {
        d.res_active[r] = 1;
        for (int i = 0; i < 8; i++) d.res_JpJdF[8 * r + i] = d.res_JpJdF_new[8 * r + i];
    } else d.res_active[r] = 0;
    d.res_state[r] = ns;
    d.res_energy[r] = d.res_new_energy[r];
}

// what: 1 = backupState (idepth_backup = idepth), 2 = resubstituteFPt (step only), 4 = apply step
__global__ void k_points(DevWindow d, const WinState *__restrict__ ws, int what) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= d.nP) return;
    const int nF = ws->nF;
    if (what & 1) d.pt_idepth_backup[p] = d.pt_idepth[p];
    if (what & 2) {
        const int host = d.pt_host[p];
        const int r0 = d.pt_res_begin[p], r1 = d.pt_res_begin[p + 1];
        int ngood = 0;
        float b = d.pt_bdSumF[p];
        {
            float s = 0.f;
            for (int i = 0; i < 4; i++) s += ws->cstep[i] * d.pt_Hcd[4 * p + i];
            b -= s;
        }
        for (int r = r0; r < r1; r++) {
            if (!d.res_active[r]) continue;
            ngood++;
            const float *xa = ws->xAd[host * nF + d.res_target[r]];
            float s = 0.f;
            for (int i = 0; i < 8; i++) s += xa[i] * d.res_JpJdF[8 * r + i];
            b -= s;
        }
        if (ngood == 0) d.pt_step[p] = 0.f;
        else if (isfinite(b)) d.pt_step[p] = -b * d.pt_HdiF[p];
    }
    if (what & 4) {
        const float nid = d.pt_idepth_backup[p] + d.pt_step[p];
        d.pt_idepth[p] = nid;
        d.pt_idepth_zero[p] = nid;
    }
}

// sum |idepth_backup| for canbreak in the piecewise do_step
__global__ void k_sum_nid(DevWindow d, WinState *ws) {
    __shared__ float sh[256];
    float s = 0.f;
    for (int p = threadIdx.x; p < d.nP; p += 256) s += fabsf(d.pt_idepth_backup[p]);
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) { ws->sumNID = sh[0]; ws->numID = (float) d.nP; }
}

// ---------------------------------------------------------------------------------------------------------
// marginalisation helpers (SURVEY §8f rank 3)
// PointFrameResidual::fixLinearizationF (Residuals.cc:216-242) on the active residuals of the selected points
__global__ void k_fix_linearization(DevWindow d, const WinState *__restrict__ ws, const uint8_t *__restrict__ pt_sel) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= d.nR) return;
    const int p = d.res_point[r];
    if (!pt_sel[p] || !d.res_active[r]) return;
    const int nF = ws->nF, h = d.pt_host[p], t = d.res_target[r];
    const float *dp = ws->adHTdeltaF[h + nF * t];
    const float *J = d.res_J + (size_t) 74 * r;
    const float deltaF = d.pt_idepth[p] - d.pt_idepth_zero[p];
    float a0 = 0.f, b0 = 0.f, a1 = 0.f, b1 = 0.f;
    for (int i = 0; i < 6; i++) { a0 += J[8 + i] * dp[i]; a1 += J[14 + i] * dp[i]; }
    for (int i = 0; i < 4; i++) { b0 += J[20 + i] * ws->calib.cDeltaF[i]; b1 += J[24 + i] * ws->calib.cDeltaF[i]; }
    const float dx = a0 + b0 + J[28] * deltaF, dy = a1 + b1 + J[29] * deltaF;
    for (int i = 0; i < 8; i++) {
        float rtz = J[i];
        rtz = rtz - J[30 + i] * dx;
        rtz = rtz - J[38 + i] * dy;
        rtz = rtz - J[46 + i] * dp[6];
        rtz = rtz - J[54 + i] * dp[7];
        d.res_toZero[8 * r + i] = rtz;
    }
    d.res_lin[r] = 1;
}
__global__ void k_scale_prior(DevWindow d, const uint8_t *__restrict__ pt_sel, float fac) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p < d.nP && pt_sel[p]) d.pt_priorF[p] *= fac;
}
// HM += w (M - Msc), bM += w (Mb - Mbsc)   (EnergyFunctional.cc:200-214)
__global__ void k_add_marg(SolveBufs sb, int n, double w) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n * n) sb.HM[e] += w * (sb.H_A[e] - sb.H_sc[e]);
    if (e < n) sb.bM[e] += w * (sb.b_A[e] - sb.b_sc[e]);
}

// ---------------------------------------------------------------------------------------------------------
// EnergyFunctional::marginalizeFrame, the prior algebra (EnergyFunctional.cc:72-129), on the device-resident HM, bM:
// move the frame's 8 rows/columns to the end (:81-99), add its own prior (:103-104), scale by (|diag|+10)^1/2 (:106-111),
// invert the 8x8 block (partial-pivot LU like Eigen's fixed-size inverse(), :114-117), Schur complement (:120-122),
// unscale (:125-126), symmetrise (:129). Output is written with the NEW leading dimension n-8. One CTA.
#define KMF_THREADS 256
__global__ void __launch_bounds__(KMF_THREADS) k_marginalize_frame(SolveBufs sb, const WinState *ws, int n, int fidx) {
    extern __shared__ double smf[];
    const int ndim = n - 8, io = CPARS + 8 * fidx, tid = threadIdx.x;
    double *H = smf;                 // [n*n] column-major, frame block moved to the end
    double *b = H + n * n;           // [n]
    double *SV = b + n;              // [n]
    double *bli = SV + n;            // [ndim][8]
    double *hp = bli + ndim * 8;     // [8][8] row-major inverse
    double *lu = hp + 64;            // [8][8] row-major LU
    __shared__ int piv[8];
    auto pold = [&](int i) { return (i < io) ? i : ((i < ndim) ? i + 8 : io + (i - ndim)); };
    for (int e = tid; e < n * n; e += KMF_THREADS) {
        const int j = e / n, i = e - j * n;
        H[e] = sb.HM[(size_t) pold(j) * n + pold(i)];
    }
    if (tid < n) b[tid] = sb.bM[pold(tid)];
    __syncthreads();
    if (tid < 8) {
        const FrameDev &f = ws->fr[fidx];
        H[(ndim + tid) * n + ndim + tid] += f.prior[tid];
        b[ndim + tid] += f.prior[tid] * f.delta_prior[tid];
    }
    __syncthreads();
    if (tid < n) SV[tid] = sqrt(fabs(H[tid * n + tid]) + 10.0);
    __syncthreads();
    for (int e = tid; e < n * n; e += KMF_THREADS) {
        const int j = e / n, i = e - j * n;
        H[e] = ((1.0 / SV[i]) * H[e]) * (1.0 / SV[j]);
    }
    __syncthreads();            // (b is scaled after the matrix: its entries feed nothing before the next barrier)
    if (tid < n) b[tid] = (1.0 / SV[tid]) * b[tid];
    if (tid < 64) { const int r = tid >> 3, c = tid & 7; lu[tid] = 0.5f * (H[(ndim + c) * n + ndim + r] + H[(ndim + c) * n + ndim + r]); }
    __syncthreads();
    if (tid == 0) {             // unblocked partial-pivot LU of the 8x8 block (a few hundred flops, serial)
        int p[8];
        for (int i = 0; i < 8; i++) p[i] = i;
        for (int k = 0; k < 8; k++) {
            int pv = k;
            double best = fabs(lu[k * 8 + k]);
            for (int i = k + 1; i < 8; i++) if (fabs(lu[i * 8 + k]) > best) { best = fabs(lu[i * 8 + k]); pv = i; }
            if (pv != k) {
                for (int j = 0; j < 8; j++) { const double t = lu[k * 8 + j]; lu[k * 8 + j] = lu[pv * 8 + j]; lu[pv * 8 + j] = t; }
                const int t = p[k]; p[k] = p[pv]; p[pv] = t;
            }
            if (lu[k * 8 + k] != 0.0) {
                const double dd = lu[k * 8 + k];
                for (int i = k + 1; i < 8; i++) lu[i * 8 + k] /= dd;
            }
            for (int j = k + 1; j < 8; j++)
                for (int i = k + 1; i < 8; i++) lu[i * 8 + j] -= lu[i * 8 + k] * lu[k * 8 + j];
        }
        for (int i = 0; i < 8; i++) piv[i] = p[i];
    }
    __syncthreads();
    if (tid < 8) {              // column tid of the inverse: solve L U x = P e_c
        double x[8];
        for (int i = 0; i < 8; i++) x[i] = (piv[i] == tid) ? 1.0 : 0.0;
        for (int i = 0; i < 8; i++) for (int j = 0; j < i; j++) x[i] -= lu[i * 8 + j] * x[j];
        for (int i = 7; i >= 0; i--) {
            for (int j = i + 1; j < 8; j++) x[i] -= lu[i * 8 + j] * x[j];
            x[i] /= lu[i * 8 + i];
        }
        for (int i = 0; i < 8; i++) hp[i * 8 + tid] = 0.5f * (x[i] + x[i]);
    }
    __syncthreads();
    for (int e = tid; e < ndim * 8; e += KMF_THREADS) {     // bli = bottomLeft^T * hpi
        const int i = e >> 3, k = e & 7;
        double s = 0.0;
        for (int m = 0; m < 8; m++) s += H[i * n + ndim + m] * hp[m * 8 + k];
        bli[e] = s;
    }
    __syncthreads();
    for (int e = tid; e < ndim * ndim; e += KMF_THREADS) {  // topLeft -= bli * bottomLeft (rows >= ndim are read-only here)
        const int j = e / ndim, i = e - j * ndim;
        double s = 0.0;
        for (int k = 0; k < 8; k++) s += bli[i * 8 + k] * H[j * n + ndim + k];
        H[j * n + i] -= s;
    }
    if (tid < ndim) {
        double s = 0.0;
        for (int k = 0; k < 8; k++) s += bli[tid * 8 + k] * b[ndim + k];
        b[tid] -= s;
    }
    __syncthreads();
    for (int e = tid; e < ndim * ndim; e += KMF_THREADS) {
        const int j = e / ndim, i = e - j * ndim;
        H[j * n + i] = (SV[i] * H[j * n + i]) * SV[j];
    }
    if (tid < ndim) b[tid] = SV[tid] * b[tid];
    __syncthreads();
    for (int e = tid; e < ndim * ndim; e += KMF_THREADS) {
        const int j = e / ndim, i = e - j * ndim;
        sb.HM[(size_t) j * ndim + i] = 0.5 * (H[j * n + i] + H[i * n + j]);
    }
    if (tid < ndim) sb.bM[tid] = b[tid];
}
#define KMF_SMEM_BYTES(n) ((size_t) ((n) * (n) + 2 * (n) + ((n) - 8) * 8 + 128) * sizeof(double))

// EnergyFunctional::insertFrame's resize of HM, bM (EnergyFunctional.cc:38-44): re-lay the (n-8)^2 prior out with the new
// leading dimension n and zero the new frame's rows/columns. src = copy of the old HM.
__global__ void k_grow_prior(SolveBufs sb, const double *src, int n) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x, od = n - 8;
    if (e < n * n) {
        const int j = e / n, i = e - j * n;
        sb.HM[e] = (i < od && j < od) ? src[(size_t) j * od + i] : 0.0;
    }
    if (e >= od && e < n) sb.bM[e] = 0.0;
}

// ---------------------------------------------------------------------------------------------------------
// EnergyFunctional::calcLEnergyF_MT (EnergyFunctional.cc:361-378) with calcLEnergyPt (:627-682) and calcMEnergyF (:353-359).
// One thread per point folds its linearised, active residuals (2 res_toZeroF + J delta) . (J delta) and deltaF^2 priorF; block sums
// are written per block and folded in block order by the last block to finish (deterministic), which also adds the frame / calibration
// priors and evaluates the marginalisation energy delta . (2 bM + HM delta). out[0] = L energy, out[1] = M energy.
#define KEN_THREADS 256
__global__ void __launch_bounds__(KEN_THREADS) k_calc_energies(DevWindow d, const WinState *__restrict__ ws, SolveBufs sb, double *part, unsigned *counter, double *out) {
    __shared__ double s_sum[KEN_THREADS / 32];
    __shared__ bool s_last;
    const int nF = ws->nF, n = ws->n, tid = threadIdx.x, p = blockIdx.x * KEN_THREADS + tid;
    double e = 0.0;
    if (p < d.nP) {
        const float dd = d.pt_idepth[p] - d.pt_idepth_zero[p];      // deltaF (EnergyFunctional.cc:424)
        const int h = d.pt_host[p];
        float ef = 0.f;
        for (int r = d.pt_res_begin[p]; r < d.pt_res_begin[p + 1]; r++) {
            if (!d.res_lin[r] || !d.res_active[r]) continue;
            const float *dp = ws->adHTdeltaF[h + nF * d.res_target[r]];
            const float *J = d.res_J + (size_t) 74 * r;
            float a = 0.f, b = 0.f;
            for (int k = 0; k < 6; k++) a += J[8 + k] * dp[k];
            for (int k = 0; k < 4; k++) b += J[20 + k] * ws->calib.cDeltaF[k];
            const float jx = a + b + J[28] * dd;
            a = 0.f; b = 0.f;
            for (int k = 0; k < 6; k++) a += J[14 + k] * dp[k];
            for (int k = 0; k < 4; k++) b += J[24 + k] * ws->calib.cDeltaF[k];
            const float jy = a + b + J[29] * dd;
            for (int k = 0; k < 8; k++) {
                float jd = J[30 + k] * jx;
                jd = jd + J[38 + k] * jy;
                jd = jd + J[46 + k] * dp[6];
                jd = jd + J[54 + k] * dp[7];
                float r0 = d.res_toZero[8 * r + k];
                r0 = r0 + r0;
                r0 = r0 + jd;
                ef += jd * r0;
            }
        }
        ef += dd * dd * d.pt_priorF[p];
        e = (double) ef;
    }
    for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
    if ((tid & 31) == 0) s_sum[tid >> 5] = e;
    __syncthreads();
    if (tid == 0) {
        double s = 0.0;
        for (int w = 0; w < KEN_THREADS / 32; w++) s += s_sum[w];
        part[blockIdx.x] = s;
        __threadfence();
        s_last = atomicAdd(counter, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!s_last) return;
    __shared__ double s_m[MAXN];
    if (tid < n) {       // calcMEnergyF: delta . (2 bM + HM delta), getStitchedDeltaF (EnergyFunctional.h:178-184)
        double hd = 0.0;
        for (int c = 0; c < n; c++) hd += sb.HM[(size_t) c * n + tid] * k2b_delta(ws, c);
        s_m[tid] = k2b_delta(ws, tid) * (2.0 * sb.bM[tid] + hd);
    }
    __syncthreads();
    if (tid == 0) {
        double EL = 0.0;
        for (int f = 0; f < nF; f++) for (int i = 0; i < 8; i++) EL += ws->fr[f].delta_prior[i] * ws->fr[f].prior[i] * ws->fr[f].delta_prior[i];
        float sc = 0.f;
        for (int i = 0; i < 4; i++) sc += ws->calib.cDeltaF[i] * (float) ws->cPrior[i] * ws->calib.cDeltaF[i];
        EL += (double) sc;
        for (unsigned b = 0; b < gridDim.x; b++) EL += ((volatile double *) part)[b];
        double EM = 0.0;
        for (int r = 0; r < n; r++) EM += s_m[r];
        out[0] = EL; out[1] = EM;
        *counter = 0u;
    }
}
