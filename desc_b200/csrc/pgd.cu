// A6-A12: projected gradient descent over the per-cycle weights (reference: DESC.m:148-261).
//
// Every iteration takes state t-1 to state t.  A group of G lanes owns one edge l=(i,j) and keeps
// its <= G*EPL slots in registers; it
//   * gathers S_{t-1}[e_jk], S_{t-1}[e_ki]                                   (DESC.m:193)
//   * adds the partner sums A_l, B_l gated by the slot's appears flags        (DESC.m:189-193)
//   * removes the edge's mean gradient ("Riemannian" projection)              (DESC.m:195-204)
//   * takes the step-rule step                                                (DESC.m:207)
//   * projects onto the probability simplex                                   (DESC.m:208-224)
//   * writes w_t, S_t[l] = w.S0                                               (DESC.m:229)
//   * scatters w_t into the partner-sum accumulators of state t (next iteration's A, B)
//   * accumulates objective(state t-1) = sum w (S[e_jk]+S[e_ki]) and |S_t - S_{t-1}|  (DESC.m:232-233)
//
// Partner sums in scatter form (SURVEY 8e / appendix A.4): the reference's
//   A_l = sum_{k: IKJ_appears} w(ik;j),  B_l = sum_{k: JKI_appears} w(jk;i)
// are per-edge scalars; slot (ij;k) is the reciprocal of (ik;j) via vertex i and of (jk;i) via
// vertex j, and the appears flags are symmetric, so slot c adds w_c to the "via shared vertex"
// accumulator of each partner edge whose flag is set.  This needs no IKJ/JKI index arrays
// (the partner edge ids are already streamed for the S gathers) and shards over GPUs with one
// all-reduce of the 2m accumulators per iteration.
//
// The objective of state t is only known while running iteration t+1 (it needs all of S_t), so
// the early-stop decision lags by one kernel; w and S are ping-ponged, and when the reference
// would have stopped at iteration u the buffers of state u are still intact (later launches see
// the `stopped` flag and return immediately).
//
// The simplex projection uses Michelot's active-set iteration: T <- (sum_{w>T} w - 1)/#{w>T}
// until the active set stops shrinking.  It converges to the same threshold as the reference's
// sort-and-scan (DESC.m:215-223) without sorting.
//
// Three implementations share the arithmetic above; desc_pgd_impl picks one per solve.
//
//  * streamed (default; k_pgd_stream in pgd_stream.cuh, k_pgd_passb in pgd_passb.cuh): two passes per
//    iteration over per-vertex shared-memory tables.  Edges are (i,j)-sorted, so the edges with the same
//    smaller endpoint i form one contiguous "vertex block".  For a slot (ij;k) the partner edge {i,k} is
//    incident to i and {j,k} to j, so every S lookup and partner-sum update is a table operation indexed
//    by the rank of k in that vertex's adjacency row (rk_i, rk_j: 14 bits + appears flags).  Pass 1 (one
//    CTA per vertex block, TMA-fed) updates the edges and scatters "via i"; pass 2 (one CTA per vertex v,
//    in-edges (u,v) with u < v) writes sjk = S_t[e_jk] for the next pass 1 and scatters "via j".  The
//    scatters are read-modify-writes in warp-private tables (apices within one edge are distinct, one
//    edge per warp instruction => no conflicts), flushed once per CTA.  No atomics: every partner-sum
//    entry is owned by exactly one CTA per kernel, so the result is bit-reproducible.  On one GPU both
//    passes keep their per-vertex data in adjacency order: pass 1 stores its partner sums into P1 and
//    S_t into the next S_adj buffer (both copies of every edge), and pass 2 adds its sums to P1 and
//    stores the finished (A, B) of every edge into acc_next.  Multi-GPU handles add both passes' sums
//    into acc_next (one reduce-to-owners) and refill S_adj from the all-gathered S (k_pgd_s_adj).
//  * blocked (k_pgd_block + k_pgd_scatter<false>): the same tables with direct loads and an L2 gather of
//    S[e_jk].  Taken on single-GPU handles of sparse graphs (m < 100 n, where the streamed kernel's
//    per-block prologue dominates), and when the streamed passes do not fit (slot lists longer than 256,
//    or tables too large for their shared memory).
//  * generic (k_pgd_iter): edge-range kernel with FP64 atomicAdd scatter.  Taken when a vertex degree
//    exceeds the shared-memory table (DESC_BLOCKED_MAXDEG).
//
// DESC_B200_PGD_PATH=stream|blocked|generic forces a path (tests); a forced stream still takes the
// blocked kernels when the graph does not fit the streamed ones.
#include "internal.cuh"

#include <algorithm>
#include <cmath>

struct PgdArgs {
    const int64_t* rowptr;
    const uint32_t *pk_jk, *pk_ki;
    const double* S0;
    const double* w_cur;
    double* w_next;
    const double* S_cur;
    double* S_next;
    const double* acc_cur;
    double* acc_next;  // 2m + [obj, change]
    double* adam_m;
    double* adam_v;
    const int* ctrl;   // [0] = stopped
    int64_t e0, e1, slot_base, m;
    double lr;         // effective step size of this iteration
    double beta1, beta2, corr1, corr2;  // Adam
};

template <int G, int EPL, int RULE>
__global__ void __launch_bounds__(256)
k_pgd_iter(PgdArgs a) {
    if (a.ctrl[0]) return;
    const int r = threadIdx.x & (G - 1);
    const int64_t grp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    const int64_t e = a.e0 + grp;
    const bool valid = e < a.e1;
    int64_t s0 = 0;
    int ns = 0;
    if (valid) {
        s0 = a.rowptr[e];
        ns = (int)(a.rowptr[e + 1] - s0);
        s0 -= a.slot_base;
    }
    double objp = 0.0, chgp = 0.0;
    double w[EPL], d[EPL];
    uint32_t pj[EPL], pi[EPL];
    double A = 0.0, B = 0.0;
    if (ns > 0) {
        A = a.acc_cur[2 * e];
        B = a.acc_cur[2 * e + 1];
    }
    double gsum = 0.0;
#pragma unroll
    for (int x = 0; x < EPL; x++) {
        const int idx = r + x * G;
        w[x] = 0.0;
        d[x] = 0.0;
        pj[x] = pi[x] = 0u;
        if (idx < ns) {
            const int64_t s = s0 + idx;
            w[x] = a.w_cur[s];
            d[x] = a.S0[s];
            pj[x] = a.pk_jk[s];
            pi[x] = a.pk_ki[s];
        }
    }
    double g[EPL];
#pragma unroll
    for (int x = 0; x < EPL; x++) {
        g[x] = 0.0;
        if (r + x * G < ns) {
            const double sg = a.S_cur[pj[x] & PK_MASK] + a.S_cur[pi[x] & PK_MASK];
            objp += w[x] * sg;
            const double part = ((pi[x] & PK_APP) ? A : 0.0) + ((pj[x] & PK_APP) ? B : 0.0);
            g[x] = sg + part * d[x];
            gsum += g[x];
        }
    }
    gsum = group_sum<G>(gsum);
    const double gmean = ns > 0 ? gsum / (double)ns : 0.0;
    // step
    double wsum = 0.0;
#pragma unroll
    for (int x = 0; x < EPL; x++) {
        if (r + x * G < ns) {
            const double gr = g[x] - gmean;
            double step;
            if (RULE == 0) {
                step = -a.lr * gr;
            } else {
                const int64_t s = s0 + r + x * G;
                const double mt = a.beta1 * a.adam_m[s] + (1.0 - a.beta1) * gr;
                const double vt = a.beta2 * a.adam_v[s] + (1.0 - a.beta2) * (gr * gr);
                a.adam_m[s] = mt;
                a.adam_v[s] = vt;
                step = -a.lr * (mt / a.corr1) / (sqrt(vt / a.corr2) + 1e-8);
            }
            w[x] = w[x] + step;
            wsum += w[x];
        }
    }
    // Michelot projection onto the simplex
    wsum = group_sum<G>(wsum);
    int cnt = ns;
    double T = ns > 0 ? (wsum - 1.0) / (double)ns : 0.0;
    for (int mit = 0; mit < G * EPL + 2; mit++) {  // the active set shrinks every pass: <= ns passes
        double s2 = 0.0;
        int c2 = 0;
#pragma unroll
        for (int x = 0; x < EPL; x++) {
            if (r + x * G < ns && w[x] > T) {
                s2 += w[x];
                c2++;
            }
        }
        s2 = group_sum<G>(s2);
        c2 = group_sum_int<G>(c2);
        const bool changed = (c2 != cnt) && (c2 > 0);
        if (changed) {
            T = (s2 - 1.0) / (double)c2;
            cnt = c2;
        }
        if (!__any_sync(0xffffffffu, changed)) break;
    }
    double snew = 0.0;
#pragma unroll
    for (int x = 0; x < EPL; x++) {
        if (r + x * G < ns) {
            const double wo = fmax(w[x] - T, 0.0);
            w[x] = wo;
            snew += wo * d[x];
            a.w_next[s0 + r + x * G] = wo;
            if (pi[x] & PK_APP) atomicAdd(&a.acc_next[2 * (int64_t)(pi[x] & PK_MASK) + ((pi[x] & PK_SEL) ? 0 : 1)], wo);
            if (pj[x] & PK_APP) atomicAdd(&a.acc_next[2 * (int64_t)(pj[x] & PK_MASK) + ((pj[x] & PK_SEL) ? 0 : 1)], wo);
        }
    }
    snew = group_sum<G>(snew);
    if (ns > 0 && r == 0) {
        a.S_next[e] = snew;
        chgp = fabs(snew - a.S_cur[e]);
    }
    // block reduction of the two scalars -> one atomic pair per block
    objp = group_sum<32>(objp);
    chgp = group_sum<32>(chgp);
    __shared__ double sh[2][8];
    const int wid = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        sh[0][wid] = objp;
        sh[1][wid] = chgp;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double o = 0.0, c = 0.0;
        for (int x = 0; x < (int)(blockDim.x >> 5); x++) {
            o += sh[0][x];
            c += sh[1][x];
        }
        atomicAdd(&a.acc_next[2 * a.m], o);
        atomicAdd(&a.acc_next[2 * a.m + 1], c);
    }
}

// state 0: uniform weights, S = mean of the edge's S0, accumulators of state 0 (DESC.m:148-157)
template <int G>
__global__ void __launch_bounds__(256)
k_pgd_init(PgdArgs a) {
    const int r = threadIdx.x & (G - 1);
    const int64_t grp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    const int64_t ngrp = ((int64_t)gridDim.x * blockDim.x) / G;
    const int64_t grp0 = grp - ((threadIdx.x & 31) / G);  // first group of this warp: warp-uniform trip count
    for (int64_t eb = a.e0 + grp0; eb < a.e1; eb += ngrp) {
        const int64_t e = eb + ((threadIdx.x & 31) / G);
        const bool valid = e < a.e1;
        const int64_t s0 = valid ? a.rowptr[e] - a.slot_base : 0;
        const int ns = valid ? (int)(a.rowptr[e + 1] - a.rowptr[e]) : 0;
        const double w0 = ns > 0 ? 1.0 / (double)ns : 0.0;
        double sn = 0.0;
        for (int idx = r; idx < ns; idx += G) {
            const int64_t s = s0 + idx;
            a.w_next[s] = w0;
            sn += w0 * a.S0[s];
            const uint32_t pi = a.pk_ki[s], pj = a.pk_jk[s];
            if (a.acc_next) {   // generic path only; the vertex-blocked path scatters in k_pgd_scatter
                if (pi & PK_APP) atomicAdd(&a.acc_next[2 * (int64_t)(pi & PK_MASK) + ((pi & PK_SEL) ? 0 : 1)], w0);
                if (pj & PK_APP) atomicAdd(&a.acc_next[2 * (int64_t)(pj & PK_MASK) + ((pj & PK_SEL) ? 0 : 1)], w0);
            }
        }
        sn = group_sum<G>(sn);
        if (r == 0 && ns > 0) a.S_next[e] = sn;
    }
}

// objective of the final state when the loop ran out of iterations (no later kernel computes it)
template <int G>
__global__ void __launch_bounds__(256)
k_pgd_obj(PgdArgs a, double* __restrict__ partial) {
    if (a.ctrl[0]) return;
    const int r = threadIdx.x & (G - 1);
    const int64_t grp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) / G;
    const int64_t ngrp = ((int64_t)gridDim.x * blockDim.x) / G;
    double objp = 0.0;
    for (int64_t e = a.e0 + grp; e < a.e1; e += ngrp) {
        const int64_t s0 = a.rowptr[e] - a.slot_base;
        const int ns = (int)(a.rowptr[e + 1] - a.rowptr[e]);
        for (int idx = r; idx < ns; idx += G) {
            const int64_t s = s0 + idx;
            objp += a.w_cur[s] * (a.S_cur[a.pk_jk[s] & PK_MASK] + a.S_cur[a.pk_ki[s] & PK_MASK]);
        }
    }
    objp = group_sum<32>(objp);
    __shared__ double sh[8];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = objp;
    __syncthreads();
    if (threadIdx.x == 0) {
        double o = 0.0;
        for (int x = 0; x < (int)(blockDim.x >> 5); x++) o += sh[x];
        if (partial) {   // fixed-order reduction by k_pgd_partials: bit-reproducible
            partial[2 * blockIdx.x] = o;
            partial[2 * blockIdx.x + 1] = 0.0;
        } else {
            atomicAdd(&a.acc_next[2 * a.m], o);
        }
    }
}

__global__ void k_fill_double(double* p, int64_t n, double v) {
    int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

// Bookkeeping after iteration t (DESC.m:232-257), one thread.
//   red = acc_next tail of kernel t: red[0] = objective(state t-1), red[1] = sum|S_t - S_{t-1}|
//   ctrl: [0]=stopped [1]=final_iter [2]=misses ; ctrlf[0] = objective(state t-2)
// last==1: red[0] is objective(state t) from k_pgd_obj (no change term).
__global__ void k_pgd_finalize(const double* __restrict__ red, int t, int last, int64_t m,
                               double tol, int patience, double* __restrict__ hist,
                               int* __restrict__ ctrl, double* __restrict__ ctrlf) {
    if (ctrl[0]) return;
    if (last) {
        hist[2 * (t - 1) + 1] = red[0];
        ctrl[1] = t;
        return;
    }
    hist[2 * (t - 1)] = red[1] / (double)m;
    if (t >= 2) {
        const int u = t - 1;  // iteration whose objective just became known
        const double obj = red[0];
        hist[2 * (u - 1) + 1] = obj;
        if (u > 1 && ctrlf[0] - obj < tol) {
            ctrl[2] += 1;
            if (ctrl[2] >= patience) {
                ctrl[0] = 1;
                ctrl[1] = u;
            }
        } else {
            ctrl[2] = 0;
        }
        ctrlf[0] = obj;
    }
}


// ------------------------------------------------------------------------------------------
// vertex-blocked path
// ------------------------------------------------------------------------------------------
#define BLK_TB 128
#define BLK_WARPS (BLK_TB / 32)

struct BlkArgs {
    PgdArgs p;
    const uint16_t *rk_i, *rk_j;
    const int *rowstart, *adj_nbr, *adj_eid, *estart;
    const uint32_t* bm;
    const int* bmprefix;
    int nwords;
    int v0, v1;        // local vertex range
    int tstride;       // padded max degree (table stride)
    double* partial;   // 2 per CTA of k_pgd_block
    // streamed path only
    const double* S_adj;   // S of the current state in adjacency order
    // one GPU only (all three null on multi-GPU handles, whose pass 2 adds to acc_next and whose S_adj is refilled
    // by k_pgd_s_adj after the all-gather):
    double* P1;            // 2m: pass 1's partner sums in adjacency order; pass 2 adds its own and stores acc_next
    double* S_adj_next;    // S of the state pass 1 builds, in adjacency order (pass 1 stores both copies of S[e])
    const int* adj_mirror; // m: adjacency position of i in row j, for edge (i,j)
};

// shared tables: T_S[tstride] | T_acc[BLK_WARPS][tstride]
// p1 non-null: the sums go to p1[rs + r] (adjacency order, plain stores); else added to the (edge, side) entries
__device__ __forceinline__ void blk_flush(const BlkArgs& a, int v, int deg, int rs, const double* T_acc,
                                          double* __restrict__ acc_out, double* __restrict__ p1 = nullptr) {
    for (int r = threadIdx.x; r < deg; r += BLK_TB) {
        double x = 0.0;
#pragma unroll
        for (int q = 0; q < BLK_WARPS; q++) x += T_acc[q * a.tstride + r];
        if (p1) {
            p1[rs + r] = x;
            continue;
        }
        const int e2 = a.adj_eid[rs + r];
        const int k = a.adj_nbr[rs + r];
        acc_out[2 * (int64_t)e2 + (v < k ? 0 : 1)] += x;   // owned by this CTA within this kernel
    }
}

template <int G, int EPL, int RULE>
__global__ void __launch_bounds__(BLK_TB)
k_pgd_block(BlkArgs a) {
    if (a.p.ctrl[0]) return;
    extern __shared__ double sh[];
    double* T_S = sh;
    double* T_acc = sh + a.tstride;
    const int v = a.v0 + blockIdx.x;
    const int rs = a.rowstart[v];
    const int deg = a.rowstart[v + 1] - rs;
    for (int r = threadIdx.x; r < deg; r += BLK_TB) {
        T_S[r] = a.p.S_cur[a.adj_eid[rs + r]];
#pragma unroll
        for (int q = 0; q < BLK_WARPS; q++) T_acc[q * a.tstride + r] = 0.0;
    }
    __syncthreads();
    double* Tw = T_acc + (threadIdx.x >> 5) * a.tstride;
    const int r = threadIdx.x & (G - 1);
    const int gw = (threadIdx.x & 31) / G;       // group within the warp
    constexpr int GPW = 32 / G;
    const int e_lo = a.estart[v], e_hi = a.estart[v + 1];
    double objp = 0.0, chgp = 0.0;
    for (int eb = e_lo; eb < e_hi; eb += BLK_TB / G) {
        const int e = eb + threadIdx.x / G;
        const bool valid = e < e_hi;
        int64_t s0 = 0;
        int ns = 0;
        double A = 0.0, B = 0.0;
        if (valid) {
            s0 = a.p.rowptr[e];
            ns = (int)(a.p.rowptr[e + 1] - s0);
            s0 -= a.p.slot_base;
            if (ns > 0) {
                A = a.p.acc_cur[2 * (int64_t)e];
                B = a.p.acc_cur[2 * (int64_t)e + 1];
            }
        }
        double w[EPL], d[EPL];
        uint32_t pj[EPL];
        uint32_t rk[EPL];
#pragma unroll
        for (int x = 0; x < EPL; x++) {
            const int idx = r + x * G;
            w[x] = 0.0;
            d[x] = 0.0;
            pj[x] = 0u;
            rk[x] = 0u;
            if (idx < ns) {
                const int64_t s = s0 + idx;
                w[x] = __ldcs(a.p.w_cur + s);
                d[x] = __ldcs(a.p.S0 + s);
                pj[x] = __ldcs(a.p.pk_jk + s);
                rk[x] = __ldcs(a.rk_i + s);
            }
        }
        double g[EPL];
        double gsum = 0.0;
#pragma unroll
        for (int x = 0; x < EPL; x++) {
            g[x] = 0.0;
            if (r + x * G < ns) {
                const double sg = a.p.S_cur[pj[x] & PK_MASK] + T_S[rk[x] & RK_MASK];
                objp += w[x] * sg;
                const double part = ((rk[x] & RK_APP) ? A : 0.0) + ((pj[x] & PK_APP) ? B : 0.0);
                g[x] = sg + part * d[x];
                gsum += g[x];
            }
        }
        gsum = group_sum<G>(gsum);
        const double gmean = ns > 0 ? gsum / (double)ns : 0.0;
        double wsum = 0.0;
#pragma unroll
        for (int x = 0; x < EPL; x++) {
            if (r + x * G < ns) {
                const double gr = g[x] - gmean;
                double step;
                if (RULE == 0) {
                    step = -a.p.lr * gr;
                } else {
                    const int64_t s = s0 + r + x * G;
                    const double mt = a.p.beta1 * a.p.adam_m[s] + (1.0 - a.p.beta1) * gr;
                    const double vt = a.p.beta2 * a.p.adam_v[s] + (1.0 - a.p.beta2) * (gr * gr);
                    a.p.adam_m[s] = mt;
                    a.p.adam_v[s] = vt;
                    step = -a.p.lr * (mt / a.p.corr1) / (sqrt(vt / a.p.corr2) + 1e-8);
                }
                w[x] = w[x] + step;
                wsum += w[x];
            }
        }
        wsum = group_sum<G>(wsum);
        int cnt = ns;
        double T = ns > 0 ? (wsum - 1.0) / (double)ns : 0.0;
        for (int mit = 0; mit < G * EPL + 2; mit++) {
            double s2 = 0.0;
            int c2 = 0;
#pragma unroll
            for (int x = 0; x < EPL; x++) {
                if (r + x * G < ns && w[x] > T) {
                    s2 += w[x];
                    c2++;
                }
            }
            s2 = group_sum<G>(s2);
            c2 = group_sum_int<G>(c2);
            const bool changed = (c2 != cnt) && (c2 > 0);
            if (changed) {
                T = (s2 - 1.0) / (double)c2;
                cnt = c2;
            }
            if (!__any_sync(0xffffffffu, changed)) break;
        }
        double snew = 0.0;
#pragma unroll
        for (int x = 0; x < EPL; x++) {
            if (r + x * G < ns) {
                const double wo = fmax(w[x] - T, 0.0);
                w[x] = wo;
                snew += wo * d[x];
                __stcs(a.p.w_next + s0 + r + x * G, wo);
            }
        }
        snew = group_sum<G>(snew);
        if (ns > 0 && r == 0) {
            a.p.S_next[e] = snew;
            chgp += fabs(snew - a.p.S_cur[e]);
        }
        // scatter "via i" into the warp-private table: one edge (group) at a time so that the
        // ranks touched by one instruction are distinct
#pragma unroll
        for (int q = 0; q < GPW; q++) {
            __syncwarp();
            if (gw == q) {
#pragma unroll
                for (int x = 0; x < EPL; x++)
                    if (r + x * G < ns && (rk[x] & RK_APP)) Tw[rk[x] & RK_MASK] += w[x];
            }
        }
        __syncwarp();
    }
    __syncthreads();
    blk_flush(a, v, deg, rs, T_acc, a.p.acc_next);
    objp = group_sum<32>(objp);
    chgp = group_sum<32>(chgp);
    __shared__ double red[2][BLK_WARPS];
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = objp;
        red[1][threadIdx.x >> 5] = chgp;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double o = 0.0, c = 0.0;
#pragma unroll
        for (int q = 0; q < BLK_WARPS; q++) {
            o += red[0][q];
            c += red[1][q];
        }
        a.partial[2 * blockIdx.x] = o;
        a.partial[2 * blockIdx.x + 1] = c;
    }
}

// Vertex-centric scatter of w (state being built) into acc_next.
//   OUT = true : own edges (v,*) of the local range, ranks rk_i          (used for state 0 only; with P1 set,
//                into P1 in adjacency order, the layout of the streamed pass 1, for pass 2 to finish)
//   OUT = false: edges (u,v) with u < v, u in the local vertex range, ranks rk_j ("via j")
// One warp handles one edge at a time (distinct ranks per instruction), four edges in flight.
template <bool OUT>
__global__ void __launch_bounds__(BLK_TB)
k_pgd_scatter(BlkArgs a, const double* __restrict__ w) {
    if (a.p.ctrl[0]) return;
    extern __shared__ double sh[];
    double* T_acc = sh;
    const int v = blockIdx.x;
    const int rs = a.rowstart[v];
    const int deg = a.rowstart[v + 1] - rs;
    int lo, hi;   // OUT: edge ids; IN: adjacency positions
    if (OUT) {
        if (v < a.v0 || v >= a.v1) return;
        lo = a.estart[v];
        hi = a.estart[v + 1];
    } else {
        const int ub = min(a.v1, v);   // neighbours u with v0 <= u < ub
        if (ub <= a.v0) return;
        lo = rs + (a.v0 > 0 ? desc_rank(a.bm, a.bmprefix, a.nwords, v, a.v0) : 0);
        hi = rs + desc_rank(a.bm, a.bmprefix, a.nwords, v, ub);
    }
    if (hi <= lo) {
        if (OUT && a.P1)   // P1 holds every row: no own edges, no "via i" sums
            for (int r = threadIdx.x; r < deg; r += BLK_TB) a.P1[rs + r] = 0.0;
        return;
    }
    for (int r = threadIdx.x; r < deg; r += BLK_TB) {
#pragma unroll
        for (int q = 0; q < BLK_WARPS; q++) T_acc[q * a.tstride + r] = 0.0;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* Tw = T_acc + warp * a.tstride;
    const uint16_t* __restrict__ RK = OUT ? a.rk_i : a.rk_j;
    constexpr int U = 4;
    for (int base = lo + warp * U; base < hi; base += BLK_WARPS * U) {
        int64_t s0[U];
        int ns[U];
#pragma unroll
        for (int q = 0; q < U; q++) {
            ns[q] = 0;
            s0[q] = 0;
            if (base + q < hi) {
                const int e = OUT ? base + q : a.adj_eid[base + q];
                s0[q] = a.p.rowptr[e];
                ns[q] = (int)(a.p.rowptr[e + 1] - s0[q]);
                s0[q] -= a.p.slot_base;
            }
        }
        double wv[U];
        uint32_t rk[U];
#pragma unroll
        for (int q = 0; q < U; q++) {
            wv[q] = 0.0;
            rk[q] = 0u;
            if (lane < ns[q]) {
                wv[q] = w[s0[q] + lane];
                rk[q] = __ldcs(RK + s0[q] + lane);
            }
        }
#pragma unroll
        for (int q = 0; q < U; q++) {
            if (rk[q] & RK_APP) Tw[rk[q] & RK_MASK] += wv[q];
            __syncwarp();
            for (int t = lane + 32; t < ns[q]; t += 32) {   // slot lists longer than a warp; the ranks
                const uint32_t rr = RK[s0[q] + t];           // of one edge are distinct: no ordering needed
                if (rr & RK_APP) Tw[rr & RK_MASK] += w[s0[q] + t];
            }
            __syncwarp();
        }
    }
    __syncthreads();
    blk_flush(a, v, deg, rs, T_acc, a.p.acc_next, OUT ? a.P1 : nullptr);
}

// S in adjacency order, S_adj[p] = S[adj_eid[p]]: the table prologues of both streamed passes then read
// a vertex's row contiguously instead of gathering it (one 2m-entry L2 gather per state, here)
__global__ void __launch_bounds__(256)
k_pgd_s_adj(const int* __restrict__ adj_eid, const double* __restrict__ S, int64_t n2m, const int* __restrict__ ctrl,
            double* __restrict__ S_adj) {
    if (ctrl[0]) return;
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p < n2m) S_adj[p] = S[adj_eid[p]];
}

// fixed-order reduction of the per-CTA partials into red[0] (objective) and red[1] (change)
#define PGD_PART_TB 1024
__global__ void __launch_bounds__(PGD_PART_TB)
k_pgd_partials(const double* __restrict__ partial, int nblocks, const int* __restrict__ ctrl,
               double* __restrict__ red) {
    if (ctrl[0]) return;
    __shared__ double sh[2][PGD_PART_TB];
    double o = 0.0, c = 0.0;
    for (int b = threadIdx.x; b < nblocks; b += PGD_PART_TB) {
        const double2 v = reinterpret_cast<const double2*>(partial)[b];
        o += v.x;
        c += v.y;
    }
    sh[0][threadIdx.x] = o;
    sh[1][threadIdx.x] = c;
    __syncthreads();
    for (int off = PGD_PART_TB / 2; off > 0; off >>= 1) {
        if (threadIdx.x < off) {
            sh[0][threadIdx.x] += sh[0][threadIdx.x + off];
            sh[1][threadIdx.x] += sh[1][threadIdx.x + off];
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        red[0] += sh[0][0];
        red[1] += sh[1][0];
    }
}

#include "pgd_stream.cuh"
#include "pgd_passb.cuh"

template <int G, int EPL, int NCW, int NSW>
static int launch_stream(desc_b200_handle* h, const BlkArgs& a, int rule_kind, bool dry) {
    const int nv = a.v1 - a.v0;
    if (nv <= 0) return DESC_B200_OK;
    constexpr int TE = NCW * 32 / G;
    StreamArgs sa;
    sa.b = a;
    sa.max_ns = h->max_ns;
    sa.tsc = (TE * h->max_ns + G * EPL + 16 + 7) & ~7;
    const size_t fixed = st_fixed_bytes(a.tstride, h->max_ns, NSW), stage = st_stage_bytes(sa.tsc, TE) + st_hdr_bytes(TE);
    // up to four CTAs per SM: one CTA's table prologue / flush overlaps the others' streaming.
    // 228 KB of shared memory per SM, 1 KB reserved per CTA.
    int nst = 0;
    for (int ctas = 4; ctas >= 1 && !nst; ctas--) {
        const size_t budget = (size_t)(228 * 1024) / ctas - 1024 - 256;
        for (int c = ST_MAXSTAGES; c >= 2 && !nst; c--)
            if (fixed + c * stage <= budget) nst = c;
    }
    if (!nst) return DESC_B200_ERR_LIMIT;   // caller falls back to the blocked kernel
    if (dry) return DESC_B200_OK;
    sa.nstages = nst;
    sa.sjk = h->sjk;
    sa.S_adj = a.S_adj;
    const size_t smem = fixed + nst * stage;
    constexpr int NT = (NCW + NSW + 1) * 32;
    if (rule_kind == 0) {
        CUDA_TRY(cudaFuncSetAttribute(k_pgd_stream<G, EPL, NCW, NSW, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_pgd_stream<G, EPL, NCW, NSW, 0><<<nv, NT, smem, h->stream>>>(sa);
    } else {
        CUDA_TRY(cudaFuncSetAttribute(k_pgd_stream<G, EPL, NCW, NSW, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_pgd_stream<G, EPL, NCW, NSW, 1><<<nv, NT, smem, h->stream>>>(sa);
    }
    KERNEL_CHECK(h);
    return DESC_B200_OK;
}

// DESC_B200_ERR_LIMIT = this graph does not fit the streamed kernel (use the blocked one).
// Launch shape: 8 slots per lane, 16-edge tiles of 2 compute + 2 scatter warps, up to four CTAs per SM -- the best of
// the shapes measured at cfg 4 (profiles/README.md): smaller CTAs overlap each other's per-vertex prologue / drain
// (round 2: 1.29 -> 1.24 ms).  Lanes per edge follow max_ns.
static int launch_stream_any(desc_b200_handle* h, const BlkArgs& a, int rule_kind, bool dry = false) {
    const int ns = h->max_ns;
    if (ns <= 32) return launch_stream<4, 8, 2, 2>(h, a, rule_kind, dry);
    if (ns <= 64) return launch_stream<8, 8, 2, 2>(h, a, rule_kind, dry);
    if (ns <= 128) return launch_stream<16, 8, 2, 2>(h, a, rule_kind, dry);
    if (ns <= 256) return launch_stream<32, 8, 2, 2>(h, a, rule_kind, dry);
    return DESC_B200_ERR_LIMIT;
}

template <int G, int EPL>
static int launch_block(desc_b200_handle* h, const BlkArgs& a, int rule_kind, size_t smem) {
    const int nv = a.v1 - a.v0;
    if (nv <= 0) return DESC_B200_OK;
    if (rule_kind == 0) {
        CUDA_TRY(cudaFuncSetAttribute(k_pgd_block<G, EPL, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_pgd_block<G, EPL, 0><<<nv, BLK_TB, smem, h->stream>>>(a);
    } else {
        CUDA_TRY(cudaFuncSetAttribute(k_pgd_block<G, EPL, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_pgd_block<G, EPL, 1><<<nv, BLK_TB, smem, h->stream>>>(a);
    }
    KERNEL_CHECK(h);
    return DESC_B200_OK;
}

static int launch_block_any(desc_b200_handle* h, const BlkArgs& a, int rule_kind, size_t smem) {
    const int ns = h->max_ns;
    if (ns <= 32) return launch_block<8, 4>(h, a, rule_kind, smem);
    if (ns <= 64) return launch_block<16, 4>(h, a, rule_kind, smem);
    if (ns <= 128) return launch_block<32, 4>(h, a, rule_kind, smem);
    if (ns <= 256) return launch_block<32, 8>(h, a, rule_kind, smem);
    if (ns <= 512) return launch_block<32, 16>(h, a, rule_kind, smem);
    if (ns <= 1024) return launch_block<32, 32>(h, a, rule_kind, smem);
    desc_set_error("an edge has %d slots; the fused PGD kernel supports at most 1024 per edge "
                   "(lower n_sample)", ns);
    return DESC_B200_ERR_LIMIT;
}

template <bool OUT>
static int launch_scatter(desc_b200_handle* h, const BlkArgs& a, const double* w, size_t smem) {
    CUDA_TRY(cudaFuncSetAttribute(k_pgd_scatter<OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_pgd_scatter<OUT><<<h->n, BLK_TB, smem, h->stream>>>(a, w);
    KERNEL_CHECK(h);
    return DESC_B200_OK;
}

// pass over larger endpoints of the streamed path: sjk <- S_t[e_jk], partner sums "via j" of w_t
static int launch_passb(desc_b200_handle* h, const BlkArgs& a, const double* w_t) {
    // warps per CTA by the mean number of local in-edges per vertex (batches of PB_U edges per warp).  Fewer than 4
    // do not pay: measured on one rank's share of an 8-GPU solve, 4 warps beat 2 there (0.438 against 0.476 ms,
    // profiles/README.md round 2)
    const double per_cta = (double)(h->e_end - h->e_begin) / std::max(h->n, 1);
    const int nw = per_cta >= 256 ? 8 : 4;
    const size_t smem = (size_t)(2 + nw) * a.tstride * sizeof(double);   // T_S, nw private tables, header tile
#define PB_LAUNCH(NW)                                                                                              \
    {                                                                                                              \
        CUDA_TRY(cudaFuncSetAttribute(k_pgd_passb<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));       \
        k_pgd_passb<NW><<<h->n, NW * 32, smem, h->stream>>>(a, w_t, h->jhdr, h->sjk, (h->max_ns + 31) / 32);           \
    }
    if (nw == 8) PB_LAUNCH(8) else PB_LAUNCH(4)
#undef PB_LAUNCH
    KERNEL_CHECK(h);
    return DESC_B200_OK;
}

static int launch_s_adj(desc_b200_handle* h, const double* S) {
    const int64_t n2m = 2 * h->m;
    if (n2m == 0) return DESC_B200_OK;
    k_pgd_s_adj<<<(unsigned)((n2m + 255) / 256), 256, 0, h->stream>>>(h->adj_eid, S, n2m, h->d_ctrl, h->S_adj[0]);
    KERNEL_CHECK(h);
    return DESC_B200_OK;
}

template <int G, int EPL>
static int launch_iter(desc_b200_handle* h, const PgdArgs& a, int rule_kind) {
    const int64_t ne = h->e_end - h->e_begin;
    const int64_t threads = ne * G;
    const unsigned grid = (unsigned)((threads + 255) / 256);
    if (grid == 0) return DESC_B200_OK;
    if (rule_kind == 0)
        k_pgd_iter<G, EPL, 0><<<grid, 256, 0, h->stream>>>(a);
    else
        k_pgd_iter<G, EPL, 1><<<grid, 256, 0, h->stream>>>(a);
    KERNEL_CHECK(h);
    return DESC_B200_OK;
}

static int launch_iter_any(desc_b200_handle* h, const PgdArgs& a, int rule_kind) {
    const int ns = h->max_ns;
    if (ns <= 32) return launch_iter<8, 4>(h, a, rule_kind);
    if (ns <= 64) return launch_iter<16, 4>(h, a, rule_kind);
    if (ns <= 128) return launch_iter<32, 4>(h, a, rule_kind);
    if (ns <= 256) return launch_iter<32, 8>(h, a, rule_kind);
    if (ns <= 512) return launch_iter<32, 16>(h, a, rule_kind);
    if (ns <= 1024) return launch_iter<32, 32>(h, a, rule_kind);
    desc_set_error("an edge has %d slots; the fused PGD kernel supports at most 1024 per edge "
                   "(lower n_sample)", ns);
    return DESC_B200_ERR_LIMIT;
}

// step size of call number t (1-based count of GetStep calls on the rule object)
static double step_size(const desc_b200_step_rule* r, int64_t t) {
    switch (r->kind) {
        case 0: return r->lr;
        case 1: return r->lr / (std::trunc((double)t / r->decay_interval) + 1.0);
        default:
            if (r->strategy == 0) return r->lr;
            return 100.0 * (r->lr / (std::trunc((double)t / r->decay_interval) + 1.0));
    }
}

// a peer that died leaves the flag barrier of comm.cu with a timeout bit instead of a hang
static int check_peer_barrier(desc_b200_handle* h) {
    if (!h->sym) return DESC_B200_OK;
    int e = 0;
    CUDA_TRY(cudaMemcpy(&e, h->d_err, sizeof(int), cudaMemcpyDeviceToHost));
    if (e & 16) {
        CUDA_TRY(cudaMemset(h->d_err, 0, sizeof(int)));
        desc_set_error("multi-GPU exchange: a peer did not reach the barrier within the timeout");
        return DESC_B200_ERR_NCCL;
    }
    return DESC_B200_OK;
}

// the two exchanges of a multi-GPU iteration: peer stores + flag barrier when the communicator has a peer-mapped
// region (comm.cu), NCCL otherwise
static int exchange_S(desc_b200_handle* h, int which) {
    if (h->world <= 1) return DESC_B200_OK;
    if (h->sym && h->S_in_sym) return desc_sym_allgather_S(h, which, h->shard_edges);
    return desc_allgather_ranges(h, h->S[which], sizeof(double), h->shard_edges);
}
static int exchange_partner_sums(desc_b200_handle* h, int which) {
    if (h->world <= 1) return DESC_B200_OK;
    if (h->sym) return desc_sym_reduce_to_owners(h, h->acc[which], h->shard_edges);
    return desc_reduce_to_owners(h, h->acc[which], 2, h->shard_edges, 2);
}

int desc_pgd_impl(desc_b200_handle* h, int iters, desc_b200_step_rule* rule, int* iters_run) {
    if (!h->have_s0) {
        desc_set_error("pgd before cycle_inconsistency");
        return DESC_B200_ERR_STATE;
    }
    if (iters < 0 || !rule || rule->kind < 0 || rule->kind > 2) {
        desc_set_error("bad iters / step rule");
        return DESC_B200_ERR_ARG;
    }
    if (h->has_dup_apex) {
        desc_set_error("the explicit cycle lists repeat an apex within an edge (a CEMP-style with-replacement draw): DESC's "
                       "projected gradient needs distinct 3-cycles per edge (DESC.m:84 samples without replacement)");
        return DESC_B200_ERR_STATE;
    }
    cudaStream_t st = h->stream;
    const int64_t m = h->m;
    const int64_t nacc = 2 * m + 2;
    const bool adam = rule->kind == 2 && rule->strategy == 0;
    const bool blocked = h->blocked_ok && h->rk_i != nullptr;
    // DESC_B200_PGD_PATH = generic | blocked | stream (default: stream when the graph fits)
    bool stream = blocked;
    {
        const char* force = getenv("DESC_B200_PGD_PATH");
        if (force && strcmp(force, "blocked") == 0) stream = false;
        // sparse graphs (cfg 5's ring: 50 own edges per vertex) make tens of thousands of tiny vertex blocks, and the
        // streamed kernel pays ~31 ns of ring / table prologue and drain per block: measured 2.61 ms per iteration
        // against 2.12 ms of the direct-load blocked kernels there (single GPU; profiles/README.md round 2)
        if (!force && h->world == 1 && h->m < 100 * (int64_t)h->n) stream = false;
    }
    if (h->world > 1 && !h->sym && !h->S[0]) DESC_TRY(desc_sym_setup(h, m, h->shard_edges));
    for (int b = 0; b < 2; b++) {
        if (!h->S[b]) {
            if (h->sym) {   // multi-GPU: S lives in the peer-mapped region, the all-gather is peer stores (comm.cu)
                h->S[b] = desc_sym_S_buffer(h, b);
                h->S_in_sym = true;
            } else {
                CUDA_TRY(cudaMalloc(&h->S[b], (m + 4) * sizeof(double)));   // +4: 16-byte widened bulk copies
            }
        }
        if (!h->acc[b]) CUDA_TRY(cudaMalloc(&h->acc[b], nacc * sizeof(double)));
    }
    if (!h->d_ctrl) {
        CUDA_TRY(cudaMalloc(&h->d_ctrl, 4 * sizeof(int)));
        CUDA_TRY(cudaMalloc(&h->d_ctrl_f, 2 * sizeof(double)));
        CUDA_TRY(cudaMallocHost(&h->h_ctrl, 4 * sizeof(int)));
    }
    if (blocked && !h->pgd_partial)
        CUDA_TRY(cudaMalloc(&h->pgd_partial, (size_t)2 * (std::max(h->n, DESC_SMS * 8) + 1) * sizeof(double)));
    if (h->hist_cap < iters + 1) {
        cudaFree(h->d_hist);
        h->d_hist = nullptr;
        CUDA_TRY(cudaMalloc(&h->d_hist, (size_t)2 * (iters + 1) * sizeof(double)));
        h->hist_cap = iters + 1;
    }
    if (adam) {
        const size_t nb = (size_t)std::max<int64_t>(h->n_slots, 1) * sizeof(double);
        const bool fresh = !h->adam_m;
        if (!h->adam_m) CUDA_TRY(cudaMalloc(&h->adam_m, nb));
        if (!h->adam_v) CUDA_TRY(cudaMalloc(&h->adam_v, nb));
        if (rule->t > 0 && (fresh || !h->adam_valid)) {
            desc_set_error("HybridGradient rule with t=%lld > 0, but this handle holds no Adam moments that continue it "
                           "(new handle, rebuilt incidence, or a run that was stopped early): HybridGradient.m:24-27 "
                           "zeroes m_t / v_t only at t == 0", (long long)rule->t);
            return DESC_B200_ERR_STATE;
        }
        if (rule->t == 0) {  // HybridGradient.m:24-27: state is zeroed on the first call only
            CUDA_TRY(cudaMemsetAsync(h->adam_m, 0, nb, st));
            CUDA_TRY(cudaMemsetAsync(h->adam_v, 0, nb, st));
        }
        h->adam_valid = false;
    }
    CUDA_TRY(cudaMemsetAsync(h->d_ctrl, 0, 4 * sizeof(int), st));
    CUDA_TRY(cudaMemsetAsync(h->d_ctrl_f, 0, 2 * sizeof(double), st));
    CUDA_TRY(cudaMemsetAsync(h->d_hist, 0, (size_t)2 * (iters + 1) * sizeof(double), st));
    {
        const unsigned gb = (unsigned)((m + 255) / 256);
        k_fill_double<<<gb, 256, 0, st>>>(h->S[0], m, 1.0);  // S_vec = ones(1,m), DESC.m:148
        KERNEL_CHECK(h);
        k_fill_double<<<gb, 256, 0, st>>>(h->S[1], m, 1.0);
        KERNEL_CHECK(h);
        // S lives in peer-mapped memory on multi-GPU handles: no rank may push its first S slice into this rank's
        // buffers before the fills above have run (a faster peer's slice would be overwritten with ones)
        if (h->S_in_sym) DESC_TRY(desc_sym_barrier(h));
    }
    PgdArgs a;
    a.rowptr = h->rowptr;
    a.pk_jk = h->pk_jk;
    a.pk_ki = h->pk_ki;
    a.S0 = h->S0;
    a.adam_m = h->adam_m;
    a.adam_v = h->adam_v;
    a.ctrl = h->d_ctrl;
    a.e0 = h->e_begin;
    a.e1 = h->e_end;
    a.slot_base = h->slot_base;
    a.m = m;
    a.beta1 = rule->beta_1;
    a.beta2 = rule->beta_2;
    a.corr1 = a.corr2 = 1.0;
    a.lr = 0.0;
    BlkArgs ba;
    ba.rk_i = h->rk_i;
    ba.rk_j = h->rk_j;
    ba.rowstart = h->rowstart;
    ba.adj_nbr = h->adj_nbr;
    ba.adj_eid = h->adj_eid;
    ba.estart = h->estart;
    ba.bm = h->bm;
    ba.bmprefix = h->bmprefix;
    ba.nwords = h->nwords;
    ba.v0 = h->v_begin;
    ba.v1 = h->v_end;
    ba.tstride = (h->maxdeg + 1 + 3) & ~3;   // >= maxdeg + 1: the last entry is a dummy slot for inactive lanes
    ba.partial = h->pgd_partial;
    ba.S_adj = nullptr;
    ba.P1 = nullptr;
    ba.S_adj_next = nullptr;
    ba.adj_mirror = h->adj_mirror;
    const size_t smem_blk = (size_t)(1 + BLK_WARPS) * ba.tstride * sizeof(double);
    const size_t smem_sc = (size_t)BLK_WARPS * ba.tstride * sizeof(double);
    const int launches0 = h->launches;
    if (stream) {   // does this graph fit the streamed kernel (and the table of the second pass)?
        ba.p = a;
        stream = h->sjk != nullptr && launch_stream_any(h, ba, adam ? 1 : 0, true) == DESC_B200_OK &&
                 (size_t)(2 + 8) * ba.tstride * sizeof(double) <= 226 * 1024;
    }
    // one GPU: pass 1 stores its partner sums in adjacency order (P1) and S_t in adjacency order (S_adj ping-pong);
    // pass 2 adds its partner sums to P1 and stores the finished (A, B) of every edge.  Multi-GPU handles add both
    // passes' sums into acc_next, reduce them to the owners, and refill one S_adj from the all-gathered S.
    const bool use_p1 = stream && h->world == 1;
    if (stream) {
        for (int b = 0; b < (use_p1 ? 2 : 1); b++)   // +4: 16-byte widened bulk copies
            if (!h->S_adj[b]) CUDA_TRY(cudaMalloc(&h->S_adj[b], (2 * m + 4) * sizeof(double)));
        if (use_p1 && !h->P1) CUDA_TRY(cudaMalloc(&h->P1, std::max<int64_t>(2 * m, 1) * sizeof(double)));
        ba.S_adj = h->S_adj[0];
        ba.P1 = use_p1 ? h->P1 : nullptr;
    }
    const int G = h->max_ns <= 32 ? 8 : (h->max_ns <= 64 ? 16 : 32);
    const int aux_grid = DESC_SMS * 8;

    // ---- state 0: uniform weights, S = mean S0 (DESC.m:148-157), partner sums of state 0
    CUDA_TRY(cudaMemsetAsync(h->acc[0], 0, nacc * sizeof(double), st));
    a.w_cur = nullptr;
    a.w_next = h->w[0];
    a.S_cur = nullptr;
    a.S_next = h->S[0];
    a.acc_cur = nullptr;
    a.acc_next = blocked ? nullptr : h->acc[0];   // blocked path: no atomics in k_pgd_init
    if (h->n_slots > 0) {
        if (G == 8)
            k_pgd_init<8><<<aux_grid, 256, 0, st>>>(a);
        else if (G == 16)
            k_pgd_init<16><<<aux_grid, 256, 0, st>>>(a);
        else
            k_pgd_init<32><<<aux_grid, 256, 0, st>>>(a);
        KERNEL_CHECK(h);
        if (blocked) {
            a.acc_next = h->acc[0];
            ba.p = a;
            DESC_TRY(launch_scatter<true>(h, ba, h->w[0], smem_sc));
            if (!stream) DESC_TRY(launch_scatter<false>(h, ba, h->w[0], smem_sc));
        }
    }
    DESC_TRY(exchange_S(h, 0));
    if (stream) DESC_TRY(launch_s_adj(h, h->S[0]));   // needs every rank's S_0
    if (stream && h->n_slots > 0) DESC_TRY(launch_passb(h, ba, h->w[0]));
    DESC_TRY(exchange_partner_sums(h, 0));

    // per-iteration kernel timing: events around the iteration kernels only
    std::vector<cudaEvent_t>& evs = h->iter_events;
    while ((int)evs.size() < 5 * std::min(iters, 512)) {
        cudaEvent_t e;
        CUDA_TRY(cudaEventCreate(&e));
        evs.push_back(e);
    }
    int t_done = 0;
    bool stopped = false;
    const int check_every = h->diag_on ? 1 : 8;   // diagnostics run a GCW per iteration: stop as soon as the rule says
    for (int t = 1; t <= iters && !stopped; t++) {
        const int cur = (t - 1) & 1, nxt = t & 1;
        // the streamed kernel stores every partner-sum entry of its vertex range (no zero-fill needed
        // on one GPU); the all-reduce over ranks and the other kernels accumulate into zeros
        if (stream && h->world == 1)
            CUDA_TRY(cudaMemsetAsync(h->acc[nxt] + 2 * m, 0, 2 * sizeof(double), st));
        else
            CUDA_TRY(cudaMemsetAsync(h->acc[nxt], 0, nacc * sizeof(double), st));
        a.w_cur = h->w[cur];
        a.w_next = h->w[nxt];
        a.S_cur = h->S[cur];
        a.S_next = h->S[nxt];
        a.acc_cur = h->acc[cur];
        a.acc_next = h->acc[nxt];
        const int64_t tcall = rule->t + t;
        a.lr = step_size(rule, tcall);
        if (adam) {
            a.corr1 = 1.0 - std::pow(rule->beta_1, (double)tcall);
            a.corr2 = 1.0 - std::pow(rule->beta_2, (double)tcall);
        }
        const bool timed = t <= 512;
        if (timed) CUDA_TRY(cudaEventRecord(evs[5 * (t - 1)], st));
        if (stream) {
            // pass 1 (smaller endpoints): update; pass 2 (larger endpoints) needs all of S_t.  S_t in adjacency
            // order serves pass 2 of iteration t and pass 1 of iteration t+1 (stream order): on one GPU pass 1
            // stores it into the other S_adj buffer, on multi-GPU handles k_pgd_s_adj refills the one buffer after
            // the all-gather.  It is no output: once the lagged stop flag is set every later kernel returns, and
            // the results are read from the ping-ponged S / w.
            ba.p = a;
            ba.S_adj = h->S_adj[use_p1 ? cur : 0];
            ba.S_adj_next = use_p1 ? h->S_adj[nxt] : nullptr;
            DESC_TRY(launch_stream_any(h, ba, adam ? 1 : 0));
            if (timed) CUDA_TRY(cudaEventRecord(evs[5 * (t - 1) + 1], st));
            DESC_TRY(exchange_S(h, nxt));
            if (timed) CUDA_TRY(cudaEventRecord(evs[5 * (t - 1) + 2], st));
            if (use_p1)
                ba.S_adj = h->S_adj[nxt];
            else
                DESC_TRY(launch_s_adj(h, h->S[nxt]));   // timed with pass 2
            DESC_TRY(launch_passb(h, ba, h->w[nxt]));
            k_pgd_partials<<<1, PGD_PART_TB, 0, st>>>(h->pgd_partial, h->v_end - h->v_begin, h->d_ctrl, h->acc[nxt] + 2 * m);
            KERNEL_CHECK(h);
        } else if (blocked) {
            ba.p = a;
            DESC_TRY(launch_block_any(h, ba, adam ? 1 : 0, smem_blk));
            DESC_TRY(launch_scatter<false>(h, ba, h->w[nxt], smem_sc));
            k_pgd_partials<<<1, PGD_PART_TB, 0, st>>>(h->pgd_partial, h->v_end - h->v_begin, h->d_ctrl, h->acc[nxt] + 2 * m);
            KERNEL_CHECK(h);
        } else {
            DESC_TRY(launch_iter_any(h, a, adam ? 1 : 0));
        }
        if (timed) {
            if (!stream) {   // single-phase paths: no events inside
                CUDA_TRY(cudaEventRecord(evs[5 * (t - 1) + 1], st));
                CUDA_TRY(cudaEventRecord(evs[5 * (t - 1) + 2], st));
            }
            CUDA_TRY(cudaEventRecord(evs[5 * (t - 1) + 3], st));
        }
        if (h->world > 1) {
            // a rank reads only the partner sums of its own edges: deliver each range's sum to its owner
            DESC_TRY(exchange_partner_sums(h, nxt));
            if (!stream) DESC_TRY(exchange_S(h, nxt));
        }
        if (timed) CUDA_TRY(cudaEventRecord(evs[5 * (t - 1) + 4], st));
        if (h->diag_on) DESC_TRY(desc_diag_record(h, t, h->S[nxt]));   // make_plots branch, DESC.m:235-239
        k_pgd_finalize<<<1, 1, 0, st>>>(h->acc[nxt] + 2 * m, t, 0, m, 1e-5, 30, h->d_hist, h->d_ctrl, h->d_ctrl_f);
        KERNEL_CHECK(h);
        t_done = t;
        if (t % check_every == 0 || t == iters) {
            CUDA_TRY(cudaMemcpyAsync(h->h_ctrl, h->d_ctrl, 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            stopped = h->h_ctrl[0] != 0;
        }
    }
    int final_iter = 0;
    if (stopped) {
        final_iter = h->h_ctrl[1];
    } else if (iters > 0) {
        // objective of the last state
        const int cur = iters & 1, nxt = (iters + 1) & 1;
        CUDA_TRY(cudaMemsetAsync(h->acc[nxt] + 2 * m, 0, 2 * sizeof(double), st));
        a.w_cur = h->w[cur];
        a.S_cur = h->S[cur];
        a.acc_next = h->acc[nxt];
        if (h->n_slots > 0) {
            double* part = blocked ? h->pgd_partial : nullptr;
            if (G == 8)
                k_pgd_obj<8><<<aux_grid, 256, 0, st>>>(a, part);
            else if (G == 16)
                k_pgd_obj<16><<<aux_grid, 256, 0, st>>>(a, part);
            else
                k_pgd_obj<32><<<aux_grid, 256, 0, st>>>(a, part);
            KERNEL_CHECK(h);
            if (blocked) {
                k_pgd_partials<<<1, PGD_PART_TB, 0, st>>>(h->pgd_partial, aux_grid, h->d_ctrl, h->acc[nxt] + 2 * m);
                KERNEL_CHECK(h);
            }
        }
        if (h->world > 1) DESC_TRY(desc_allreduce_sum(h, h->acc[nxt] + 2 * m, 2));
        k_pgd_finalize<<<1, 1, 0, st>>>(h->acc[nxt] + 2 * m, iters, 1, m, 1e-5, 30, h->d_hist, h->d_ctrl, h->d_ctrl_f);
        KERNEL_CHECK(h);
        final_iter = iters;
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    h->final_buf = final_iter & 1;
    h->have_pgd = true;
    *iters_run = final_iter;
    rule->t += final_iter;
    if (adam) h->adam_valid = !stopped;   // a stopped run has advanced the moments one launch past the reported state
    // mean durations over the iterations that did real work: kernels of pass 1 / pass 2, collectives
    double s1 = 0.0, s2 = 0.0, sc = 0.0;
    int cnt = 0;
    for (int t = 1; t <= std::min(std::min(t_done, 512), std::max(final_iter, 1)); t++) {
        float a1 = 0.f, ag = 0.f, a2 = 0.f, ar = 0.f;
        cudaEvent_t* e = &evs[5 * (t - 1)];
        if (cudaEventElapsedTime(&a1, e[0], e[1]) == cudaSuccess && cudaEventElapsedTime(&ag, e[1], e[2]) == cudaSuccess &&
            cudaEventElapsedTime(&a2, e[2], e[3]) == cudaSuccess && cudaEventElapsedTime(&ar, e[3], e[4]) == cudaSuccess) {
            s1 += a1;
            s2 += a2;
            sc += ag + ar;
            cnt++;
        }
    }
    DESC_TRY(check_peer_barrier(h));
    h->tm.pgd_pass1_ms = cnt > 0 ? s1 / cnt : 0.0;
    h->tm.pgd_pass2_ms = cnt > 0 ? s2 / cnt : 0.0;
    h->tm.pgd_comm_ms = cnt > 0 ? sc / cnt : 0.0;
    h->tm.pgd_iter_ms = cnt > 0 ? (s1 + s2) / cnt : 0.0;
    h->tm.pgd_launches = h->launches - launches0;
    return DESC_B200_OK;
}
