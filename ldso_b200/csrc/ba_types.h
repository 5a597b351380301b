// Plain structs the BA kernels (ba_k2.cuh, ba_k3.cuh) take as arguments and the host context keeps: includable by any unit
// without defining a kernel.
#pragma once
#include "common.cuh"

struct SolveBufs {
    double *H_A, *b_A, *H_sc, *b_sc;      // stitched pieces, column-major n x n / n
    double *HM, *bM;                      // marginalisation prior
    double *Pns;                          // null-space projector (n x n, col-major)
    double *lastHS, *lastbS, *lastX;
    // assembled system handed from K2b to K3 (EnergyFunctional.cc:257,283-291): HFinal_top (column-major) and its
    // diagonal, HFinal_top - H_sc (becomes lastHS once solved), bFinal_top (becomes lastbS)
    double *A0g, *dg, *HSg, *bFg;
};

// peer-memory all-reduce of the reduced buffer (k2r_peer_allreduce)
#define K2R_MAX_PEERS 8
struct PeerExchange {
    int rank, world, n_doubles, n_chunks;
    int two_hop;                          // reduce-scatter + all-gather (world > 2) instead of the one-shot push
    uint4 *inbox[K2R_MAX_PEERS];          // rank r's inbox (peer-mapped for r != rank): [2][K2R_MAX_PEERS][n_doubles] (reduce-scatter / one-shot) + [2][n_doubles] (all-gather)
    int *epoch;                           // local: number of exchanges completed
    unsigned *done;                       // local: CTAs finished in this launch
    int *error;                           // local: set when a peer's data never arrived (bounded spin)
    double *out;                          // local: the summed buffer
};
