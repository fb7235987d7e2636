// SURVEY 8(f) #3: Cycle-Edge Message Passing on the incidence the DESC build made
// (reference: Algorithms/CEMP.m:98-129 == CEMP_GCW.m:100-125; MPLS.m:219-233 uses the same
// reweighting with the LAA residuals in place of SVec).
//
//   SVec_0(l)    = mean_s S0(l,s)                                            CEMP.m:101
//   SVec_{t+1}(l) = sum_s w_s S0(l,s) / sum_s w_s,  w_s = exp(-beta_t (SVec_t(e_ki) + SVec_t(e_jk)))   :116-124
//   SVec(l) = 1 for edges without a 3-cycle                                  :102,125
//
// The reference normalises the weights first (WeightMat./weightsum, :121) and then sums
// WeightMat.*S0Mat (:122-124); the kernel forms sum(w S0)/sum(w) in one pass over the slots -- the same
// value up to rounding (|diff| <= a few ulp, parity bar 1e-10).
//
// Layout: as k_cycle -- a group of G lanes per edge, lanes stride over the edge's slots; per slot one
// packed partner word pair (8 B) + S0 (8 B) streamed, two 8-byte gathers from the length-m vector
// (40 MB at cfg 4: L2 resident).  Algorithmic bytes per reweighting: 16*m_cycle + 8*m (vector in)
// + 8*m (rowptr) + 8*m (vector out).  HBM-bound; no tensor cores.
#include "internal.cuh"

#include <algorithm>

// Edge distribution: every CTA takes one contiguous run of edges instead of a grid-stride.  Edges are (i,j)-sorted, so
// a CTA then works through whole vertex blocks, and the x[] entries of the edges (i,k), k>i -- two thirds of the "via i"
// gathers -- are the CTA's own few-KB range and stay in L1 instead of costing an L2 sector each (the kernel is bound by
// L2 sector throughput: 7.7e8 sectors = 10 TB/s at 2.4 ms, profiles/r01_cemp_ncu_summary.txt).
template <int G>
__global__ void __launch_bounds__(256)
k_cemp_reweight(const int64_t* __restrict__ rowptr, const uint32_t* __restrict__ pk_jk,
                const uint32_t* __restrict__ pk_ki, const double* __restrict__ S0,
                const double* __restrict__ x_cur, double* __restrict__ x_next, int64_t e0, int64_t e1,
                int64_t slot_base, double beta, double empty_value) {
    const int r = threadIdx.x & (G - 1);
    const int sub = (threadIdx.x & 31) / G;
    const int64_t per = (e1 - e0 + gridDim.x - 1) / gridDim.x;
    const int64_t first = e0 + blockIdx.x * per + (threadIdx.x >> 5) * (32 / G);   // first group of this warp
    const int64_t last = min(e1, e0 + (blockIdx.x + 1) * per);
    const int64_t step = blockDim.x / G;
    // the trip count is warp-uniform (shuffles below): every lane of a warp iterates from the warp's first group
    for (int64_t eb = first; eb < last; eb += step) {
        const int64_t e = eb + sub;
        const bool valid = e < last;
        const int64_t s0 = valid ? rowptr[e] - slot_base : 0;
        const int ns = valid ? (int)(rowptr[e + 1] - rowptr[e]) : 0;
        double wsum = 0.0, acc = 0.0;
        for (int idx = r; idx < ns; idx += G) {
            const int64_t s = s0 + idx;
            double w = 1.0;
            if (x_cur) {
                const double ski = x_cur[pk_ki[s] & PK_MASK];
                const double sjk = x_cur[pk_jk[s] & PK_MASK];
                w = exp(-beta * (ski + sjk));
            }
            wsum += w;
            acc += w * S0[s];
        }
        wsum = group_sum<G>(wsum);
        acc = group_sum<G>(acc);
        if (r == 0 && valid) x_next[e] = ns > 0 ? acc / wsum : empty_value;
    }
}

// x_next[local edges] = reweighting of x_cur (x_cur == nullptr: plain mean of S0); all-gathered over ranks
int desc_cemp_reweight(desc_b200_handle* h, const double* x_cur, double* x_next, double beta, double empty_value) {
    if (h->e_end > h->e_begin) {
        const int grid = DESC_SMS * 8;
        cudaStream_t st = h->stream;
#define CEMP_LAUNCH(G)                                                                                        \
    k_cemp_reweight<G><<<grid, 256, 0, st>>>(h->rowptr, h->pk_jk, h->pk_ki, h->S0, x_cur, x_next, h->e_begin, \
                                             h->e_end, h->slot_base, beta, empty_value)
        if (h->max_ns <= 8)
            CEMP_LAUNCH(8);
        else if (h->max_ns <= 16)
            CEMP_LAUNCH(16);
        else
            CEMP_LAUNCH(32);
#undef CEMP_LAUNCH
        KERNEL_CHECK(h);
    }
    if (h->world > 1) DESC_TRY(desc_allgather_ranges(h, x_next, sizeof(double), h->shard_edges));
    return DESC_B200_OK;
}

int desc_cemp_impl(desc_b200_handle* h, int max_iter, const double* beta, int n_beta) {
    if (!h->have_s0) {
        desc_set_error("cemp before cycle_inconsistency");
        return DESC_B200_ERR_STATE;
    }
    if (max_iter < 0 || (max_iter > 0 && (!beta || n_beta <= 0))) {
        desc_set_error("bad max_iter / reweighting (max_iter=%d, %d reweighting values)", max_iter, n_beta);
        return DESC_B200_ERR_ARG;
    }
    for (int b = 0; b < 2; b++)
        if (!h->cemp_S[b]) CUDA_TRY(cudaMalloc(&h->cemp_S[b], (size_t)std::max<int64_t>(h->m, 1) * sizeof(double)));
    DESC_TRY(desc_cemp_reweight(h, nullptr, h->cemp_S[0], 0.0, 1.0));           // CEMP.m:101-102
    for (int t = 0; t < max_iter; t++) {
        const double b = beta[std::min(t, n_beta - 1)];                          // CEMP.m:31-35
        DESC_TRY(desc_cemp_reweight(h, h->cemp_S[t & 1], h->cemp_S[(t + 1) & 1], b, 1.0));   // :106-126
    }
    h->cemp_final = max_iter & 1;
    h->have_cemp = true;
    return DESC_B200_OK;
}
