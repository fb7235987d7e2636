// Streamed vertex-blocked PGD iteration (included by pgd.cu after PgdArgs / BlkArgs).
//
// Same arithmetic and the same ownership rules as k_pgd_block (one CTA per vertex block, S and
// partner-sum tables in shared memory, no atomics), re-organised around the Blackwell async-copy
// machinery so that the HBM stream never waits for the arithmetic:
//
//   * one PRODUCER warp: lane 0 issues cp.async.bulk (TMA, 1-D) copies of the next tile's slot
//     arrays (w, S0, sjk, rk_i: contiguous because the edges of a vertex block and their slot
//     lists are contiguous) and per-edge arrays (rowptr, partner sums, S) into a ring of shared-
//     memory stages; completion is signalled on an mbarrier (complete_tx::bytes).  L2 policy
//     evict_first for the slot streams: they must not evict S.  Before the first tile it copies the
//     vertex's S table, S_adj[rowstart[v] .. rowstart[v+1]) (S in adjacency order), with one more
//     bulk copy on its own mbarrier: no index-dependent gather in the prologue.
//   * One GPU: the compute warps store both adjacency-order copies of S_t[e] into the next S_adj
//     buffer (the upper end of row i, contiguous, and adj_mirror[e] in row j, copied with the tile),
//     and the flush stores the partner-sum table into P1 in adjacency order; pass 2 finishes the sums.
//     Multi-GPU handles store the table into acc_next's (edge, side) entries and refill S_adj after
//     the all-gather (k_pgd_s_adj).
//   * COMPUTE warps: G lanes own one edge and keep EPL slots each in registers.  They read the
//     stage, compute gradient / step / projection, write w_t in place into the stage, publish
//     (slot offset, count) of their edges and arrive on the stage's `done` mbarrier.  There is NO
//     global gather in this kernel: S[e_ki] comes from the vertex block's shared-memory S table and
//     S[e_jk] arrives as the streamed array sjk, which the pass over larger endpoints
//     (pgd_passb.cuh) wrote from ITS shared-memory table.  (A divergent 8-byte gather costs the
//     SM's load/store pipe ~2 cycles per lane - measured: it, not HBM, bounded the first versions.)
//   * the SCATTER warp owns the private partner-sum table: it stores the finished w_t tile to
//     global memory with one bulk copy (TMA store), re-reads (w_t, rank) of the stage with one
//     lane per slot (distinct ranks within an edge => conflict-free read-modify-write), and
//     releases the stage to the producer through the `empty` mbarrier once the bulk store has
//     read it.
//
// Bulk copies need 16-byte aligned addresses and sizes: a tile's slot range [sA, sB) is widened to
// [sA & ~7, (sB + 7) & ~7) (8 slots = 16 B of the 2-byte rank array); arrays are allocated with
// spare elements (build.cu, pgd.cu) so the widened reads stay inside the allocations.  The w_t store
// covers the 16-byte aligned interior of [sA, sB); a ragged first / last element is stored directly.

#define ST_MAXSTAGES 4
#ifndef ST_PFT
#define ST_PFT 2                       // L2 prefetch distance of the producer, in tiles (2: 1.29 ms, 3: 1.30, 5: 1.32, 8: 1.37)
#endif

__device__ __forceinline__ uint32_t st_smem(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(st_smem(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(st_smem(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(st_smem(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(st_smem(bar)),
        "r"(parity), "r"(20000u)   // suspend-time hint (ns): sleep in hardware instead of spinning
        : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void bulk_g2s_plain(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     st_smem(dst)),
                 "l"(src), "r"(bytes), "r"(st_smem(bar))
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar, uint64_t pol) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
            st_smem(dst)),
        "l"(src), "r"(bytes), "r"(st_smem(bar)), "l"(pol)
        : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* dst, const void* src, uint32_t bytes, uint64_t pol) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group.L2::cache_hint [%0], [%1], %2, %3;" ::"l"(dst),
                 "r"(st_smem(src)), "r"(bytes), "l"(pol)
                 : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

struct StreamArgs {
    BlkArgs b;
    int nstages;
    int tsc;          // slot capacity of one stage (multiple of 8)
    int max_ns;       // longest slot list (size of the reciprocal table)
    const double* sjk;  // S[e_jk] per slot for the current state (pgd_passb.cuh)
    const double* S_adj;    // S_cur in adjacency order (2m + 4: 16-byte widened bulk copy)
};

// shared-memory carve-up: barriers | edge headers[nstages][TE] | 1/c table | T_S[tstride+2] | T_acc[NSW] | stages.
// One stage: w[tsc] f64 | S0[tsc] f64 | sjk[tsc] f64 | rk_i[tsc] u16 | rowptr[TE+2] i64 |
//            acc_cur[2*TE] f64 | S_cur[TE+2] f64 | adj_mirror[st_mir_cap] i32   (every offset a multiple of 16 bytes)
// The edge headers of a stage (st_hdr_bytes) sit apart from its ring slot, so only the stages in use take room.
// adj_mirror is copied from a multiple of 4 edges: TE + 3 + 3 entries at most, rounded up to 4.
__host__ __device__ __forceinline__ int st_mir_cap(int te) { return (te + 9) & ~3; }
__host__ __device__ __forceinline__ size_t st_stage_bytes(int tsc, int te) {
    return (size_t)tsc * (8 + 8 + 8 + 2) + (size_t)(te + 2) * 8 + (size_t)te * 16 + (size_t)(te + 2) * 8 +
           (size_t)st_mir_cap(te) * 4;
}
__host__ __device__ __forceinline__ size_t st_hdr_bytes(int te) { return (size_t)te * sizeof(int2); }
__host__ __device__ __forceinline__ size_t st_rcp_bytes(int max_ns) { return ((size_t)(max_ns + 1) * 8 + 15) & ~(size_t)15; }
__host__ __device__ __forceinline__ size_t st_fixed_bytes(int tstride, int max_ns, int nsw) {
    return 128 + st_rcp_bytes(max_ns) +
           (size_t)(1 + nsw) * tstride * sizeof(double) + 16;   // T_S (+2: widened copy) + the scatter warps' private tables
}

// G lanes per edge with EPL slots each, NCW compute warps, ST_NSW scatter warps (private tables),
// RULE 0 = constant/piecewise/decayed-SGD step, 1 = Adam
template <int G, int EPL, int NCW, int ST_NSW, int RULE>
__global__ void __launch_bounds__((NCW + ST_NSW + 1) * 32)
k_pgd_stream(StreamArgs sa) {
    const BlkArgs& a = sa.b;
    if (a.p.ctrl[0]) return;
    constexpr int TE = NCW * 32 / G;   // edges per tile
    constexpr int NTHREADS = (NCW + ST_NSW + 1) * 32;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw);
    uint64_t* full = bars;
    uint64_t* done = bars + ST_MAXSTAGES;
    uint64_t* empty = bars + 2 * ST_MAXSTAGES;
    uint64_t* tbar = bars + 3 * ST_MAXSTAGES;   // the S table
    int2* hdr = reinterpret_cast<int2*>(smem_raw + 128);
    double* rcp = reinterpret_cast<double*>(smem_raw + 128 + (size_t)sa.nstages * st_hdr_bytes(TE));
    double* T_S0 = reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(rcp) + st_rcp_bytes(sa.max_ns));
    double* T_acc = T_S0 + a.tstride + 2;
    unsigned char* stage0 = reinterpret_cast<unsigned char*>(T_acc + (size_t)ST_NSW * a.tstride);
    const int tsc = sa.tsc;
    const size_t stage_bytes = st_stage_bytes(tsc, TE);
    const size_t off_d = (size_t)tsc * 8, off_sj = (size_t)tsc * 16, off_rk = (size_t)tsc * 24;
    const size_t off_rp = (size_t)tsc * 26, off_acc = off_rp + (size_t)(TE + 2) * 8;
    const size_t off_so = off_acc + (size_t)TE * 16, off_mi = off_so + (size_t)(TE + 2) * 8;
    const int NST = sa.nstages;

    const int v = a.v0 + blockIdx.x;
    const int rs = a.rowstart[v];
    const int deg = a.rowstart[v + 1] - rs;
    const int e_lo = a.estart[v], e_hi = a.estart[v + 1];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (e_hi <= e_lo) {   // no own edges: nothing to update; its partner-sum entries start at zero
        for (int r = threadIdx.x; r < deg; r += NTHREADS) {
            if (a.P1) {
                a.P1[rs + r] = 0.0;
                continue;
            }
            const int e2 = a.adj_eid[rs + r];
            const int k = a.adj_nbr[rs + r];
            a.p.acc_next[2 * (int64_t)e2 + (v < k ? 0 : 1)] = 0.0;
        }
        if (threadIdx.x == 0) {
            a.partial[2 * blockIdx.x] = 0.0;
            a.partial[2 * blockIdx.x + 1] = 0.0;
        }
        return;
    }
    const int ntiles = (e_hi - e_lo + TE - 1) / TE;
    const int eoff = e_lo & 1;   // the per-edge arrays are copied from an even edge index (16-byte alignment)
    const double* T_S = T_S0 + (rs & 1);   // the same for the S table: copied from an even adjacency position
    if (threadIdx.x == 0) {
        for (int s = 0; s < NST; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&done[s], NCW);
            mbar_init(&empty[s], ST_NSW);
        }
        mbar_init(tbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    double objp = 0.0, chgp = 0.0;
    if (warp == NCW + ST_NSW) {
        // ------------------------------------------------------------------ producer
        // lanes prefetch the slot boundaries of 32 tiles at a time; lane 0 issues the bulk copies
        const uint64_t pol = l2_evict_first_policy();
        if (lane == 0) {   // the S table first: its latency overlaps the ring fill
            const int p0 = rs & ~1, cnt = ((rs + deg + 1) & ~1) - p0;
            mbar_expect_tx(tbar, (uint32_t)(cnt * 8));
            bulk_g2s_plain(T_S0, sa.S_adj + p0, (uint32_t)(cnt * 8), tbar);
        }
        int s = 0;
        uint32_t ph = 0;
        for (int tb = 0; tb < ntiles; tb += 32) {
            const int tl = min(tb + lane, ntiles - 1);
            const int le0 = e_lo + tl * TE, le1 = min(le0 + TE, e_hi);
            const int64_t lA = a.p.rowptr[le0] - a.p.slot_base;
            const int64_t lB = a.p.rowptr[le1] - a.p.slot_base;
            const int nu = min(32, ntiles - tb);
            for (int u = 0; u < nu; u++) {
                const int64_t sA = __shfl_sync(0xffffffffu, lA, u);
                const int64_t sB = __shfl_sync(0xffffffffu, lB, u);
                // L2 prefetch of a tile that no stage is free for yet: its bulk copies will then be L2 hits
                // (the ring is too short - shared memory - to cover the DRAM latency of ~3000 cycles)
                const int up = min(u + ST_PFT, 31);
                const int64_t pA = __shfl_sync(0xffffffffu, lA, up) & ~(int64_t)7;
                const int64_t pB = (__shfl_sync(0xffffffffu, lB, up) + 7) & ~(int64_t)7;
                if (lane == 0 && u + ST_PFT < nu && pB > pA) {
                    const uint32_t c = (uint32_t)(pB - pA);
                    bulk_prefetch_l2(a.p.w_cur + pA, c * 8);
                    bulk_prefetch_l2(a.p.S0 + pA, c * 8);
                    bulk_prefetch_l2(sa.sjk + pA, c * 8);
                    bulk_prefetch_l2(a.rk_i + pA, c * 2);
                }
                if (lane == 0) {
                    const int t = tb + u;
                    const int e0 = e_lo + t * TE, e1 = min(e0 + TE, e_hi);
                    const int e0a = e0 - eoff;
                    const int rp_cnt = (e1 + 1 - e0a + 1) & ~1;
                    const int so_cnt = (e1 - e0a + 1) & ~1;
                    const int e0m = e0 & ~3;   // adj_mirror (4-byte entries): from a multiple of 4 edges
                    const int mi_cnt = a.S_adj_next ? (e1 - e0m + 3) & ~3 : 0;
                    const int64_t base = sA & ~(int64_t)7;
                    const int64_t cnt = ((sB + 7) & ~(int64_t)7) - base;
                    unsigned char* st = stage0 + (size_t)s * stage_bytes;
                    mbar_wait(&empty[s], ph ^ 1u);
                    mbar_expect_tx(&full[s], (uint32_t)(cnt * 26 + rp_cnt * 8 + (e1 - e0) * 16 + so_cnt * 8 + mi_cnt * 4));
                    bulk_g2s_plain(st + off_rp, a.p.rowptr + e0a, (uint32_t)(rp_cnt * 8), &full[s]);
                    bulk_g2s_plain(st + off_acc, a.p.acc_cur + 2 * (int64_t)e0, (uint32_t)((e1 - e0) * 16), &full[s]);
                    bulk_g2s_plain(st + off_so, a.p.S_cur + e0a, (uint32_t)(so_cnt * 8), &full[s]);
                    if (mi_cnt > 0) bulk_g2s_plain(st + off_mi, a.adj_mirror + e0m, (uint32_t)(mi_cnt * 4), &full[s]);
                    if (cnt > 0) {
                        bulk_g2s(st, a.p.w_cur + base, (uint32_t)(cnt * 8), &full[s], pol);
                        bulk_g2s(st + off_d, a.p.S0 + base, (uint32_t)(cnt * 8), &full[s], pol);
                        bulk_g2s(st + off_sj, sa.sjk + base, (uint32_t)(cnt * 8), &full[s], pol);
                        bulk_g2s(st + off_rk, a.rk_i + base, (uint32_t)(cnt * 2), &full[s], pol);
                    }
                }
                if (++s == NST) {
                    s = 0;
                    ph ^= 1u;
                }
                __syncwarp();
            }
        }
    } else {
        // ------------------------------------------------------------------ tables (compute + scatter warps)
        constexpr int NT = (NCW + ST_NSW) * 32;
        for (int c = threadIdx.x; c <= sa.max_ns; c += NT) rcp[c] = c > 0 ? 1.0 / (double)c : 0.0;
        for (int r = threadIdx.x; r < deg; r += NT) {
#pragma unroll
            for (int q = 0; q < ST_NSW; q++) T_acc[q * a.tstride + r] = 0.0;
        }
        asm volatile("bar.sync 1, %0;" ::"n"(NT) : "memory");
        if (warp < NCW) {
            mbar_wait(tbar, 0);   // the S table has arrived
            // -------------------------------------------------------------- compute
            // Branch-free inner loop: a lane's EPL slots are idx = r + x*G; lanes past the end of the
            // slot list read harmless stage bytes and are neutralised with selects.
            const int r = threadIdx.x & (G - 1);
            // edge within the tile.  The groups of a warp take the warp's edges in the order even edges
            // (first half-warp), odd edges (second half-warp): consecutive slot lists are ~max_ns doubles
            // apart, so neighbouring edges in one half-warp collide in the shared-memory banks (for
            // 30-slot lists: 2-way on every 64-bit stage access), edges two apart do not.
            constexpr int GPW = 32 / G;              // groups (= edges) per warp
            const int g = (threadIdx.x & 31) / G;
            const int q = (threadIdx.x >> 5) * GPW + (GPW >= 4 ? 2 * (g % (GPW / 2)) + g / (GPW / 2) : g);
            const double nlr = -a.p.lr;
            const int up = rs + deg - e_hi;   // S_adj position of own edge e: up + e (the upper end of the row)
            int s = 0;
            uint32_t ph = 0;
            unsigned char* st = stage0;
            int e = e_lo + q;
            for (int t = 0; t < ntiles; t++, e += TE) {
                const int64_t* rp = reinterpret_cast<const int64_t*>(st + off_rp) + eoff;
                mbar_wait(&full[s], ph);
                int sl = 0, ns = 0;
                int64_t s0 = 0;
                double A = 0.0, B = 0.0, Sold = 0.0;
                if (e < e_hi) {
                    const int64_t rq = rp[q];
                    s0 = rq - a.p.slot_base;
                    ns = (int)(rp[q + 1] - rq);
                    sl = (int)(s0 - ((rp[0] - a.p.slot_base) & ~(int64_t)7));
                    const double2 ab = reinterpret_cast<const double2*>(st + off_acc)[q];
                    A = ab.x;
                    B = ab.y;
                    Sold = (reinterpret_cast<const double*>(st + off_so) + eoff)[q];
                }
                const int nx = (ns - r + G - 1) / G;   // this lane owns slots x < nx  (G is a power of two)
                double* pw = reinterpret_cast<double*>(st) + sl + r;
                const double* pd = reinterpret_cast<const double*>(st + off_d) + sl + r;
                const double* psj = reinterpret_cast<const double*>(st + off_sj) + sl + r;
                const uint16_t* prk = reinterpret_cast<const uint16_t*>(st + off_rk) + sl + r;
                double u[EPL], d[EPL];
                double gsum = 0.0, wsum = 0.0;
#pragma unroll
                for (int x = 0; x < EPL; x++) {
                    const bool ok = x < nx;
                    const uint32_t rk = prk[x * G];
                    const double sj = ok ? psj[x * G] : 0.0;
                    const double ts = T_S[ok ? (rk & RK_MASK) : 0u];
                    const double w = ok ? pw[x * G] : 0.0;
                    d[x] = ok ? pd[x * G] : 0.0;
                    const double sg = sj + ts;
                    objp = fma(w, sg, objp);
                    const double part = ((rk & RK_APP) ? A : 0.0) + ((rk & RK_APP2) ? B : 0.0);
                    const double g = ok ? fma(part, d[x], sg) : 0.0;
                    gsum += g;
                    wsum += w;
                    u[x] = RULE == 0 ? fma(nlr, g, w) : g;   // w - lr g  (the mean is added back below)
                }
#pragma unroll
                for (int o = G / 2; o > 0; o >>= 1) {
                    gsum += __shfl_xor_sync(0xffffffffu, gsum, o);
                    wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
                }
                const double fns = (double)ns;
                const double rns = rcp[ns];          // 1/ns (0 when the edge has no slots)
                const double gmean = gsum * rns;
                if (RULE == 0) {
                    // sum(w + step) = sum(w) - lr (sum(g) - ns mean(g))
                    wsum = fma(nlr, gsum - fns * gmean, wsum);
                    const double c = a.p.lr * gmean;
#pragma unroll
                    for (int x = 0; x < EPL; x++) u[x] = x < nx ? u[x] + c : -1e300;
                } else {
                    wsum = 0.0;
#pragma unroll
                    for (int x = 0; x < EPL; x++) {
                        if (x < nx) {
                            const double gr = u[x] - gmean;
                            const int64_t sg = s0 + r + x * G;
                            const double mt = a.p.beta1 * a.p.adam_m[sg] + (1.0 - a.p.beta1) * gr;
                            const double vt = a.p.beta2 * a.p.adam_v[sg] + (1.0 - a.p.beta2) * (gr * gr);
                            a.p.adam_m[sg] = mt;
                            a.p.adam_v[sg] = vt;
                            u[x] = pw[x * G] + -a.p.lr * (mt / a.p.corr1) / (sqrt(vt / a.p.corr2) + 1e-8);
                            wsum += u[x];
                        } else {
                            u[x] = -1e300;
                        }
                    }
                    wsum = group_sum<G>(wsum);
                }
                // Michelot: T <- (sum_{w>T} w - 1)/#{w>T} until the active set stops shrinking
                int cnt = ns;
                double T = (wsum - 1.0) * rns;
                for (int mit = 0; mit < G * EPL + 2; mit++) {
                    double s2 = 0.0;
                    int c2 = 0;
#pragma unroll
                    for (int x = 0; x < EPL; x++) {
                        const bool in = u[x] > T;
                        s2 += in ? u[x] : 0.0;
                        c2 += in ? 1 : 0;
                    }
#pragma unroll
                    for (int o = G / 2; o > 0; o >>= 1) {
                        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
                        c2 += __shfl_xor_sync(0xffffffffu, c2, o);
                    }
                    const bool changed = (c2 != cnt) && (c2 > 0);
                    if (changed) {
                        T = (s2 - 1.0) * rcp[c2];
                        cnt = c2;
                    }
                    if (!__any_sync(0xffffffffu, changed)) break;
                }
                double snew = 0.0;
#pragma unroll
                for (int x = 0; x < EPL; x++) {
                    const double wo = fmax(u[x] - T, 0.0);
                    snew = fma(wo, d[x], snew);
                    if (x < nx) pw[x * G] = wo;
                }
                snew = group_sum<G>(snew);
                if (r == 0) {
                    hdr[s * TE + q] = make_int2(sl, ns);
                    if (ns > 0) {
                        a.p.S_next[e] = snew;
                        chgp += fabs(snew - Sold);
                    }
                    if (a.S_adj_next && e < e_hi) {
                        // S_t in adjacency order, both copies: (i, j) in row i (contiguous: the own edges are
                        // the upper end of the row) and (j, i) in row j.  An edge without slots keeps its S.
                        const double sv = ns > 0 ? snew : Sold;
                        a.S_adj_next[up + e] = sv;
                        a.S_adj_next[(reinterpret_cast<const int*>(st + off_mi) + ((e - q) & 3))[q]] = sv;
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // w_t tile: generic writes -> bulk store
                __syncwarp();
                if (lane == 0) mbar_arrive(&done[s]);
                st += stage_bytes;
                if (++s == NST) {
                    s = 0;
                    ph ^= 1u;
                    st = stage0;
                }
            }
        } else {
            // -------------------------------------------------------------- scatter
            const int swi = warp - NCW;
            double* Tw = T_acc + (size_t)swi * a.tstride;
            const uint32_t dummy = (uint32_t)a.tstride - 1u;
            const uint64_t pol = l2_evict_first_policy();
            int s = 0;
            uint32_t ph = 0;
            unsigned char* st = stage0;
            for (int t = 0; t < ntiles; t++) {
                const double* sw = reinterpret_cast<const double*>(st);
                const uint16_t* srk = reinterpret_cast<const uint16_t*>(st + off_rk);
                const int64_t* rp = reinterpret_cast<const int64_t*>(st + off_rp) + eoff;
                mbar_wait(&done[s], ph);
                if (swi == 0 && lane < 3) {
                    // w_t tile -> global: 16-byte aligned interior as one bulk store, ragged ends directly
                    const int e0 = e_lo + t * TE, e1 = min(e0 + TE, e_hi);
                    const int64_t sA = rp[0] - a.p.slot_base, sB = rp[e1 - e0] - a.p.slot_base;
                    const int64_t base = sA & ~(int64_t)7;
                    const int64_t iA = (sA + 1) & ~(int64_t)1, iB = sB & ~(int64_t)1;
                    if (lane == 0) {
                        if (iB > iA) bulk_s2g(a.p.w_next + iA, sw + (iA - base), (uint32_t)((iB - iA) * 8), pol);
                        bulk_commit();
                    } else if (lane == 1) {
                        if (iA > sA && sB > sA) a.p.w_next[sA] = sw[sA - base];
                    } else {
                        if (iB < sB && sB - 1 >= iA) a.p.w_next[sB - 1] = sw[sB - 1 - base];
                    }
                }
                // This warp's edges q = swi, swi + NSW, ... in batches of U, one edge after the other into the
                // warp's private table; the (w, rank) loads of the next batch are issued before the current
                // batch's read-modify-writes.
                constexpr int U = 4;
                constexpr int NK = (TE + ST_NSW - 1) / ST_NSW;      // edges per scatter warp and tile
                constexpr int NB = (NK + U - 1) / U;
                int nsu[U], nsn[U], offn[U];
                double wv[U], wn[U];
                uint32_t rk[U], rn[U];
                auto load_batch = [&](int b, int (&ns_)[U], int (&off_)[U], double (&w_)[U], uint32_t (&r_)[U]) {
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        const int q = swi + (b * U + u) * ST_NSW;
                        const int2 h2 = q < TE ? hdr[s * TE + q] : make_int2(0, 0);
                        ns_[u] = h2.y;
                        off_[u] = h2.x;
                        w_[u] = 0.0;
                        r_[u] = 0u;
                        if (lane < h2.y) {
                            w_[u] = sw[h2.x + lane];
                            r_[u] = srk[h2.x + lane];
                        }
                    }
                };
                int offu[U];
                load_batch(0, nsu, offu, wv, rk);
                for (int b = 0; b < NB; b++) {
                    if (b + 1 < NB) load_batch(b + 1, nsn, offn, wn, rn);
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        // branch-free: lanes without the flag update the dummy entry with 0
                        const bool f = (rk[u] & RK_APP) != 0u;
                        const uint32_t ia = f ? (rk[u] & RK_MASK) : dummy;
                        const double x = Tw[ia];
                        Tw[ia] = x + (f ? wv[u] : 0.0);
                        __syncwarp();
                    }
                    // slot lists longer than a warp (ranks of one edge are distinct: no ordering needed inside)
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        if (nsu[u] > 32) {
                            for (int i2 = lane + 32; i2 < nsu[u]; i2 += 32) {
                                const uint32_t rr = srk[offu[u] + i2];
                                if (rr & RK_APP) Tw[rr & RK_MASK] += sw[offu[u] + i2];
                            }
                            __syncwarp();
                        }
                    }
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        nsu[u] = nsn[u];
                        offu[u] = offn[u];
                        wv[u] = wn[u];
                        rk[u] = rn[u];
                    }
                }
                if (swi == 0 && lane == 0) bulk_wait_read0();   // the bulk store has read the stage
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
                st += stage_bytes;
                if (++s == NST) {
                    s = 0;
                    ph ^= 1u;
                    st = stage0;
                }
            }
            if (swi == 0 && lane == 0) bulk_wait0();
        }
    }
    __syncthreads();
    // flush the private tables: every (edge, side) entry belongs to exactly one vertex block.  One GPU: into
    // P1 in adjacency order, contiguous (pass 2 adds its share and stores the finished sums into acc_next).
    // Multi-GPU: this kernel is the first writer of acc_next in an iteration => plain stores (pass 2 adds
    // its share to them).
    if (a.P1) {
        for (int r = threadIdx.x; r < deg; r += NTHREADS) {
            double x = 0.0;
#pragma unroll
            for (int q = 0; q < ST_NSW; q++) x += T_acc[q * a.tstride + r];
            a.P1[rs + r] = x;
        }
    } else {
        constexpr int KU = 4;
        for (int rb = threadIdx.x; rb < deg; rb += NTHREADS * KU) {
            int64_t pos[KU];
#pragma unroll
            for (int k = 0; k < KU; k++) {
                const int r = rb + k * NTHREADS;
                pos[k] = -1;
                if (r < deg) pos[k] = 2 * (int64_t)a.adj_eid[rs + r] + (v < a.adj_nbr[rs + r] ? 0 : 1);
            }
#pragma unroll
            for (int k = 0; k < KU; k++) {
                const int r = rb + k * NTHREADS;
                if (r < deg) {
                    double x = 0.0;
#pragma unroll
                    for (int q = 0; q < ST_NSW; q++) x += T_acc[q * a.tstride + r];
                    a.p.acc_next[pos[k]] = x;
                }
            }
        }
    }
    objp = group_sum<32>(objp);
    chgp = group_sum<32>(chgp);
    __shared__ double red[2 * NCW];
    if (lane == 0 && warp < NCW) {
        red[2 * warp] = objp;
        red[2 * warp + 1] = chgp;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double o = 0.0, c = 0.0;
#pragma unroll
        for (int q = 0; q < NCW; q++) {
            o += red[2 * q];
            c += red[2 * q + 1];
        }
        a.partial[2 * blockIdx.x] = o;
        a.partial[2 * blockIdx.x + 1] = c;
    }
}
