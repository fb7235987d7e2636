// Pass over LARGER endpoints (included by pgd.cu after BlkArgs): the second half of a PGD iteration.
//
// One CTA per vertex v walks the slot lists of the edges (u,v), u < v, whose smaller endpoint lies in
// the local vertex range.  For a slot (uv;k) the partner edge {v,k} is incident to v, so with the
// rank of k in v's adjacency row (rk_j, 14 bits + JKI_appears) both
//   * S_t[{v,k}]          -> sjk[slot]      (read by the streamed kernel of iteration t+1 instead of
//                                            a random gather: DESC.m:193, first term) and
//   * w_t[slot] (if JKI_appears) -> partner sum "via v" of edge {v,k}      (DESC.m:185-191)
// are shared-memory table operations.  Every warp owns a private partner-sum table (the ranks inside
// one edge are distinct, so one edge per instruction is a conflict-free read-modify-write) and keeps
// the (w, rank) loads of the next two batches of edges and the headers of the third in flight in
// registers while it works on the current batch.
// No atomics: every partner-sum entry (edge, side v) is owned by vertex v's CTA.
// The S table is a contiguous read of S_adj (S in adjacency order).  On one GPU the flush finishes the
// partner sums: it adds the table to pass 1's share of the same row, P1[rs + r], and stores the sum into
// acc_next, every entry of the vertex's row in every launch (also when the vertex has no local
// in-edges).  Positions r >= low (the upper neighbours) are the vertex's own edges estart[v] + r - low in
// order, side A: contiguous stores.  Positions r < low are in-edges, side B: one adj_eid load and one
// scattered store each.  Multi-GPU handles (P1 null) add the table to acc_next instead, so that one
// exchange reduces the whole sum to the owners.
#ifndef PB_U
#define PB_U 4
#endif
#ifndef PB_PF
#define PB_PF 6                         // L2 prefetch distance in batches
#endif

// partner-sum entry (edge, side v) of adjacency position rs + r of vertex v
__device__ __forceinline__ int64_t pb_acc_pos(const BlkArgs& a, int v, int rs, int r) {
    return 2 * (int64_t)a.adj_eid[rs + r] + (v < a.adj_nbr[rs + r] ? 0 : 1);
}
// One GPU: acc_next of v's row = P1 (pass 1's share) + the sum of the NQ tables T_acc (this pass's share, zero
// when T_acc is null), by a CTA of NQ warps, KU entries per thread at a time so that the loads overlap
template <int NQ, int KU>
__device__ __forceinline__ void pb_finish_row(const BlkArgs& a, int v, int rs, int deg, const double* T_acc) {
    const int eb = a.estart[v];
    const int low = deg - (a.estart[v + 1] - eb);   // in-edges (u, v), u < v, come first in the row
    constexpr int NT = NQ * 32;
    for (int rb = threadIdx.x; rb < deg; rb += NT * KU) {
        double p1[KU];
        int e[KU];
#pragma unroll
        for (int k = 0; k < KU; k++) {
            const int r = rb + k * NT;
            p1[k] = r < deg ? a.P1[rs + r] : 0.0;
            e[k] = r < low ? a.adj_eid[rs + r] : eb + r - low;
        }
#pragma unroll
        for (int k = 0; k < KU; k++) {
            const int r = rb + k * NT;
            if (r < deg) {
                double x = 0.0;
                if (T_acc) {
#pragma unroll
                    for (int q = 0; q < NQ; q++) x += T_acc[q * a.tstride + r];
                }
                a.p.acc_next[2 * (int64_t)e[k] + (r < low ? 1 : 0)] = p1[k] + x;   // x1 + x2, as multi-GPU forms it
            }
        }
    }
}

// PB_WARPS warps (= private tables) per CTA: 8 when a vertex has hundreds of local in-edges, else 4
// (smaller CTAs, more of them per SM), so that the O(degree) table prologue / flush of one CTA
// overlaps the others'.
template <int PB_WARPS>
__global__ void __launch_bounds__(PB_WARPS * 32)
k_pgd_passb(BlkArgs a, const double* __restrict__ w, const int2* __restrict__ jhdr, double* __restrict__ sjk,
            int cpe) {
    // cpe = ceil(longest slot list / 32): an in-edge is walked as `cpe` pieces of <= 32 slots ("virtual
    // edges": ranks inside one edge are distinct, so its pieces never conflict with each other)
    if (a.p.ctrl[0]) return;
    constexpr int PB_TB = PB_WARPS * 32;
    extern __shared__ double sh[];
    double* T_S = sh;
    double* T_acc = sh + a.tstride;
    const int v = (int)gridDim.x - 1 - (int)blockIdx.x;   // long in-edge lists first
    const int rs = a.rowstart[v];
    const int deg = a.rowstart[v + 1] - rs;
    // (KU grows as the CTA shrinks: both shapes cover 1280 entries per trip)
    constexpr int KU = 40 / PB_WARPS;
    const int ub = min(a.v1, v);                           // neighbours u with v0 <= u < ub
    if (ub <= a.v0) {
        if (a.P1) pb_finish_row<PB_WARPS, KU>(a, v, rs, deg, nullptr);
        return;
    }
    const int lo = rs + (a.v0 > 0 ? desc_rank(a.bm, a.bmprefix, a.nwords, v, a.v0) : 0);
    const int hi = rs + desc_rank(a.bm, a.bmprefix, a.nwords, v, ub);
    if (hi <= lo) {
        if (a.P1) pb_finish_row<PB_WARPS, KU>(a, v, rs, deg, nullptr);
        return;
    }
    int2* shdr = reinterpret_cast<int2*>(T_acc + (size_t)PB_WARPS * a.tstride);   // headers of the in-edges [lo, hi)
    // table prologue, KU entries per thread at a time: all loads in flight together
    for (int rb = threadIdx.x; rb < deg; rb += PB_TB * KU) {
        double sv[KU];
        int2 hv[KU];
#pragma unroll
        for (int k = 0; k < KU; k++) {
            const int r = rb + k * PB_TB;
            sv[k] = r < deg ? a.S_adj[rs + r] : 0.0;
            hv[k] = lo + r < hi ? __ldg(jhdr + lo + r) : make_int2(0, 0);
        }
#pragma unroll
        for (int k = 0; k < KU; k++) {
            const int r = rb + k * PB_TB;
            if (r < deg) {
                T_S[r] = sv[k];
                shdr[r] = hv[k];
#pragma unroll
                for (int q = 0; q < PB_WARPS; q++) T_acc[q * a.tstride + r] = 0.0;
            }
        }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* TA = T_acc + (size_t)warp * a.tstride;
    const uint16_t* __restrict__ RK = a.rk_j;
    const uint32_t dummy = (uint32_t)a.tstride - 1u;
    constexpr int U = PB_U;
    // Register pipeline: three buffers of U edges; while one is worked on, the (w, rank) loads of the
    // next two are in flight.  The loop is unrolled over the three buffers so that no register holding
    // an in-flight load is ever copied (a rotation `cur = next` would wait for the loads).  Headers
    // come from shared memory, so a buffer's loads can be issued as soon as it is free.
    struct Buf {
        int2 h[U];
        double w[U];
        uint32_t r[U];
    };
    const int nv = (hi - lo) * cpe;          // virtual edges of this vertex
    auto header = [&](int vi) {              // (first slot, slot count <= 32) of virtual edge vi
        int2 hh = make_int2(0, 0);
        if (vi < nv) {
            if (cpe == 1) {
                hh = shdr[vi];
            } else {
                const int r = vi / cpe, j = vi - r * cpe;
                const int2 e = shdr[r];
                hh = make_int2(e.x + 32 * j, max(0, min(32, e.y - 32 * j)));
            }
        }
        return hh;
    };
    auto load = [&](Buf& B, int bb) {
#pragma unroll
        for (int u = 0; u < U; u++) {
            B.h[u] = header(bb + u);
            B.w[u] = 0.0;
            B.r[u] = 0u;
            if (lane < B.h[u].y) {
                B.w[u] = __ldcs(w + B.h[u].x + lane);
                B.r[u] = __ldcs(RK + B.h[u].x + lane);
            }
        }
    };
    // L2 prefetch of the chunks PB_PF batches ahead (headers are in shared memory, so the addresses
    // are known long before the loads are issued): lanes 4u..4u+3 touch the three 128-byte lines of
    // edge u's weights and the line of its ranks.  Takes the DRAM latency off the register pipeline.
    auto prefetch = [&](int bb) {
        const int u = lane >> 2, part = lane & 3;
        if (u < U) {
            const int2 hh = header(bb + u);
            if (part * 16 < hh.y) {
                const void* ptr = part < 3 ? (const void*)(w + hh.x + part * 16) : (const void*)(RK + hh.x);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(ptr));
            }
        }
    };
    auto work = [&](const Buf& B) {
        // branch-free: inactive lanes (past the list end / flag off) use the dummy table entry
        double ts[U];
#pragma unroll
        for (int u = 0; u < U; u++) ts[u] = T_S[lane < B.h[u].y ? (B.r[u] & RK_MASK) : dummy];
#pragma unroll
        for (int u = 0; u < U; u++) {
            if (lane < B.h[u].y) __stcs(sjk + B.h[u].x + lane, ts[u]);
            const bool f = (B.r[u] & RK_APP) != 0u;
            const uint32_t ia = f ? (B.r[u] & RK_MASK) : dummy;
            const double t = TA[ia];
            TA[ia] = t + (f ? B.w[u] : 0.0);
            __syncwarp();
        }
    };
    const int stride = PB_WARPS * U;
    int base = warp * U;
    const int hi_v = nv;
    Buf X, Y, Z;
    load(X, base);
    load(Y, base + stride);
    load(Z, base + 2 * stride);
#pragma unroll
    for (int k = 3; k < 3 + PB_PF; k++) prefetch(base + k * stride);
    while (base < hi_v) {
        work(X);
        load(X, base + 3 * stride);
        prefetch(base + (3 + PB_PF) * stride);
        if (base + stride >= hi_v) break;
        work(Y);
        load(Y, base + 4 * stride);
        prefetch(base + (4 + PB_PF) * stride);
        if (base + 2 * stride >= hi_v) break;
        work(Z);
        load(Z, base + 5 * stride);
        prefetch(base + (5 + PB_PF) * stride);
        base += 3 * stride;
    }
    __syncthreads();
    // flush (every entry (edge, side v) is owned by this CTA within this kernel)
    if (a.P1) {
        pb_finish_row<PB_WARPS, KU>(a, v, rs, deg, T_acc);
        return;
    }
    // multi-GPU: KU entries per thread at a time so that the index loads and read-modify-writes overlap
    for (int rb = threadIdx.x; rb < deg; rb += PB_TB * KU) {
        int64_t pos[KU];
        double old[KU];
#pragma unroll
        for (int k = 0; k < KU; k++) {
            const int r = rb + k * PB_TB;
            pos[k] = r < deg ? pb_acc_pos(a, v, rs, r) : -1;
        }
#pragma unroll
        for (int k = 0; k < KU; k++) old[k] = pos[k] >= 0 ? a.p.acc_next[pos[k]] : 0.0;
#pragma unroll
        for (int k = 0; k < KU; k++) {
            const int r = rb + k * PB_TB;
            if (r < deg) {
                double x = 0.0;
#pragma unroll
                for (int q = 0; q < PB_WARPS; q++) x += T_acc[q * a.tstride + r];
                a.p.acc_next[pos[k]] = old[k] + x;
            }
        }
    }
}

