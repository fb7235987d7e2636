// Graph setup and CSR edge->3-cycle incidence build on device (reference: DESC.m:19-127).
//
// Data structures (all in HBM, built once):
//   * adjacency bitmap  bm[n][nwords]  + per-word prefix popcounts bmprefix[n][nwords]
//     -> "is k a common neighbour of i and j" is one AND, and the CSR position of (row, v) is
//        bmprefix + popc, so the symmetric CSR (adj_nbr/adj_eid) is filled without any sort.
//     replaces AdjMat (DESC.m:23-24), IndMat (DESC.m:67-68) and the dense DGEMM co-degree
//     (DESC.m:29).
//   * rowptr[m+1] (int64) / apex[m_cycle]: the CSR incidence = cum_ind / IJK (DESC.m:49,93),
//     kept over ALL edges (edges without triangles have empty rows).
//   * pk_jk / pk_ki: Ind_jk / Ind_ki (DESC.m:87-88) packed with the orientation bit and the
//     IKJ_appears / JKI_appears flag (DESC.m:113,124).
#include "internal.cuh"

#include <stdlib.h>

#include <algorithm>
#include <cmath>

// error bits written by kernels into h->d_err[0]
#define ERRB_RANGE 1
#define ERRB_ORDER 2
#define ERRB_NOTINT 4
#define ERRB_APEX 8

// ------------------------------------------------------------------------------------------
// A1: Ind (m x 2 doubles, 1-based) -> ei/ej int32 0-based, with validation (SURVEY H9)
// ------------------------------------------------------------------------------------------
__global__ void k_convert_ind(const double* __restrict__ Ind, int64_t m, int* __restrict__ ei,
                              int* __restrict__ ej, int* __restrict__ err, int* __restrict__ nmax) {
    int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    double di = Ind[e], dj = Ind[m + e];
    int bad = 0;
    if (!(di >= 1.0) || !(dj > di) || !(dj <= 2147483647.0)) bad |= ERRB_RANGE;
    if (di != floor(di) || dj != floor(dj)) bad |= ERRB_NOTINT;
    if (!bad && e > 0) {
        double pi = Ind[e - 1], pj = Ind[m + e - 1];
        if (!(pi < di || (pi == di && pj < dj))) bad |= ERRB_ORDER;
    }
    if (bad) {
        atomicOr(err, bad);
        return;
    }
    ei[e] = (int)di - 1;
    ej[e] = (int)dj - 1;
    atomicMax(nmax, (int)dj);
}

__global__ void k_set_bits(const int* __restrict__ ei, const int* __restrict__ ej, int64_t m,
                           uint32_t* __restrict__ bm, int nwords) {
    int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    int i = ei[e], j = ej[e];
    atomicOr(&bm[(size_t)i * nwords + (j >> 5)], 1u << (j & 31));
    atomicOr(&bm[(size_t)j * nwords + (i >> 5)], 1u << (i & 31));
}

// one warp per row: exclusive prefix of popcounts over the row's words, row degree
__global__ void k_row_prefix(const uint32_t* __restrict__ bm, int* __restrict__ bmprefix,
                             int* __restrict__ deg, int n, int nwords) {
    int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (row >= n) return;
    int run = 0;
    for (int base = 0; base < nwords; base += 32) {
        int w = base + lane;
        int c = (w < nwords) ? __popc(bm[(size_t)row * nwords + w]) : 0;
        int inc = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (w < nwords) bmprefix[(size_t)row * nwords + w] = run + inc - c;
        run += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) deg[row] = run;
}

// single-block exclusive scan of n ints into n+1 ints (n is the node count: small)
__global__ void k_scan_nodes(const int* __restrict__ deg, int* __restrict__ rowstart, int n,
                             int* __restrict__ err_isolated) {
    __shared__ int sh[1024];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += 1024) {
        int idx = base + threadIdx.x;
        int v = idx < n ? deg[idx] : 0;
        if (idx < n && v == 0) atomicOr(err_isolated, 1);
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            int t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += t;
            __syncthreads();
        }
        if (idx < n) rowstart[idx] = carry + sh[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry += sh[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) rowstart[n] = carry;
}

__global__ void k_fill_adj(const int* __restrict__ ei, const int* __restrict__ ej, int64_t m,
                           const uint32_t* __restrict__ bm, const int* __restrict__ bmprefix,
                           int nwords, const int* __restrict__ rowstart, int* __restrict__ adj_nbr,
                           int* __restrict__ adj_eid, int* __restrict__ adj_mirror) {
    int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    int i = ei[e], j = ej[e];
    int pi = rowstart[i] + desc_rank(bm, bmprefix, nwords, i, j);
    int pj = rowstart[j] + desc_rank(bm, bmprefix, nwords, j, i);
    adj_nbr[pi] = j;
    adj_eid[pi] = (int)e;
    adj_nbr[pj] = i;
    adj_eid[pj] = (int)e;
    adj_mirror[e] = pj;   // where the streamed PGD pass 1 stores the second copy of S[e] in adjacency order
}

// estart[v] = first edge whose smaller endpoint is >= v (edges sorted by (i,j)); estart[n] = m
__global__ void k_estart(const int* __restrict__ ei, int64_t m, int n, int* __restrict__ estart) {
    int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v > n) return;
    int64_t lo = 0, hi = m;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (ei[mid] < v)
            lo = mid + 1;
        else
            hi = mid;
    }
    estart[v] = (int)lo;
}

int desc_graph_setup(desc_b200_handle* h, const double* d_Ind) {
    const int64_t m = h->m;
    cudaStream_t st = h->stream;
    CUDA_TRY(cudaMalloc(&h->d_err, 8 * sizeof(int)));
    CUDA_TRY(cudaMemsetAsync(h->d_err, 0, 8 * sizeof(int), st));
    CUDA_TRY(cudaMalloc(&h->ei, std::max<int64_t>(m, 1) * sizeof(int)));
    CUDA_TRY(cudaMalloc(&h->ej, std::max<int64_t>(m, 1) * sizeof(int)));
    const int TB = 256;
    const unsigned gb = (unsigned)((m + TB - 1) / TB);
    if (m > 0) {
        k_convert_ind<<<gb, TB, 0, st>>>(d_Ind, m, h->ei, h->ej, h->d_err, h->d_err + 1);
        KERNEL_CHECK(h);
    }
    int herr[2];
    CUDA_TRY(cudaMemcpyAsync(herr, h->d_err, sizeof(herr), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (herr[0]) {
        desc_set_error("Ind violates the layout contract (%s%s%s): rows must be 1-based integers "
                       "with i<j, strictly sorted by (i,j) [DESC.m:31-37 matches edges to tril(:) "
                       "order by position]",
                       (herr[0] & ERRB_RANGE) ? "range " : "", (herr[0] & ERRB_ORDER) ? "order " : "",
                       (herr[0] & ERRB_NOTINT) ? "non-integer" : "");
        return DESC_B200_ERR_ARG;
    }
    int nmax = herr[1];
    if (h->n <= 0) h->n = nmax;
    if (nmax > h->n) {
        desc_set_error("Ind references node %d but n=%d", nmax, h->n);
        return DESC_B200_ERR_ARG;
    }
    if (h->n <= 0 || m <= 0) {
        desc_set_error("empty graph (n=%d, m=%lld)", h->n, (long long)m);
        return DESC_B200_ERR_ARG;
    }
    const int n = h->n;
    h->nwords = (((n + 31) / 32) + 3) & ~3;  // rows are 16-byte aligned for uint4 loads
    const size_t bmsz = (size_t)n * h->nwords;
    if (bmsz * 8 > (size_t)24 << 30) {
        desc_set_error("n=%d needs a %.1f GB adjacency bitmap; the sorted-list build path for very "
                       "large sparse graphs is not implemented",
                       n, bmsz * 8 / 1e9);
        return DESC_B200_ERR_LIMIT;
    }
    CUDA_TRY(cudaMalloc(&h->bm, bmsz * sizeof(uint32_t)));
    CUDA_TRY(cudaMalloc(&h->bmprefix, bmsz * sizeof(int)));
    CUDA_TRY(cudaMalloc(&h->rowstart, (size_t)(n + 1) * sizeof(int)));
    CUDA_TRY(cudaMalloc(&h->adj_nbr, 2 * m * sizeof(int)));
    CUDA_TRY(cudaMalloc(&h->adj_eid, 2 * m * sizeof(int)));
    CUDA_TRY(cudaMalloc(&h->adj_mirror, (m + 4) * sizeof(int)));   // +4: 16-byte widened bulk copies
    int* d_deg = nullptr;
    CUDA_TRY(cudaMalloc(&d_deg, (size_t)n * sizeof(int)));
    CUDA_TRY(cudaMemsetAsync(h->bm, 0, bmsz * sizeof(uint32_t), st));
    k_set_bits<<<gb, TB, 0, st>>>(h->ei, h->ej, m, h->bm, h->nwords);
    KERNEL_CHECK(h);
    k_row_prefix<<<(n * 32 + TB - 1) / TB, TB, 0, st>>>(h->bm, h->bmprefix, d_deg, n, h->nwords);
    KERNEL_CHECK(h);
    k_scan_nodes<<<1, 1024, 0, st>>>(d_deg, h->rowstart, n, h->d_err + 2);
    KERNEL_CHECK(h);
    k_fill_adj<<<gb, TB, 0, st>>>(h->ei, h->ej, m, h->bm, h->bmprefix, h->nwords, h->rowstart,
                                  h->adj_nbr, h->adj_eid, h->adj_mirror);
    KERNEL_CHECK(h);
    CUDA_TRY(cudaMalloc(&h->estart, (size_t)(n + 1) * sizeof(int)));
    k_estart<<<(n + 1 + TB - 1) / TB, TB, 0, st>>>(h->ei, m, n, h->estart);
    KERNEL_CHECK(h);
    h->h_estart.resize(n + 1);
    {
        std::vector<int> rs(n + 1);
        CUDA_TRY(cudaMemcpyAsync(rs.data(), h->rowstart, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaMemcpyAsync(h->h_estart.data(), h->estart, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        h->maxdeg = 0;
        for (int v = 0; v < n; v++) h->maxdeg = std::max(h->maxdeg, rs[v + 1] - rs[v]);
    }
    h->blocked_ok = h->maxdeg <= DESC_BLOCKED_MAXDEG;
    {
        const char* force = getenv("DESC_B200_PGD_PATH");   // "generic" forces the atomic edge-range kernel (tests)
        if (force && strcmp(force, "generic") == 0) h->blocked_ok = false;
    }
    int iso = 0;
    CUDA_TRY(cudaMemcpyAsync(&iso, h->d_err + 2, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaFree(d_deg));
    if (iso) {
        desc_set_error("a node in 1..n has no edge: GCW.m:21 would divide by zero (SURVEY H9)");
        return DESC_B200_ERR_ARG;
    }
    return DESC_B200_OK;
}

// ------------------------------------------------------------------------------------------
// generic exclusive scan int32 -> int64 (three kernels)
// ------------------------------------------------------------------------------------------
#define SCAN_TB 256
#define SCAN_PER 8
#define SCAN_TILE (SCAN_TB * SCAN_PER)

__global__ void k_scan_tile_sums(const int* __restrict__ in, int64_t count, int64_t* __restrict__ sums) {
    __shared__ int64_t sh[SCAN_TB / 32];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE;
    int64_t s = 0;
    for (int x = 0; x < SCAN_PER; x++) {
        int64_t idx = base + x * SCAN_TB + threadIdx.x;
        if (idx < count) s += in[idx];
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int64_t t = 0;
        for (int x = 0; x < SCAN_TB / 32; x++) t += sh[x];
        sums[blockIdx.x] = t;
    }
}

__global__ void k_scan_sums(int64_t* __restrict__ sums, int64_t nt) {
    // single thread block, sequential over chunks; nt is small (count / 2048)
    __shared__ int64_t sh[1024];
    __shared__ int64_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int64_t base = 0; base < nt; base += 1024) {
        int64_t idx = base + threadIdx.x;
        int64_t v = idx < nt ? sums[idx] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            int64_t t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += t;
            __syncthreads();
        }
        if (idx < nt) sums[idx] = carry + sh[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry += sh[1023];
        __syncthreads();
    }
}

__global__ void k_scan_apply(const int* __restrict__ in, int64_t count,
                             const int64_t* __restrict__ sums, int64_t* __restrict__ out) {
    // thread t owns SCAN_PER consecutive elements of the tile
    __shared__ int64_t sh[SCAN_TB];
    int64_t base = (int64_t)blockIdx.x * SCAN_TILE + (int64_t)threadIdx.x * SCAN_PER;
    int v[SCAN_PER];
    int64_t s = 0;
#pragma unroll
    for (int x = 0; x < SCAN_PER; x++) {
        v[x] = (base + x < count) ? in[base + x] : 0;
        s += v[x];
    }
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < SCAN_TB; o <<= 1) {
        int64_t t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
        __syncthreads();
        sh[threadIdx.x] += t;
        __syncthreads();
    }
    int64_t run = sums[blockIdx.x] + sh[threadIdx.x] - s;
#pragma unroll
    for (int x = 0; x < SCAN_PER; x++) {
        if (base + x < count) out[base + x] = run;
        run += v[x];
    }
    if (base <= count - 1 && base + SCAN_PER > count - 1) out[count] = run;  // total
}

int desc_exclusive_scan_i64(desc_b200_handle* h, const int* in, int64_t* out, int64_t count) {
    // out has count+1 entries; out[count] = total
    if (count == 0) {
        CUDA_TRY(cudaMemsetAsync(out, 0, sizeof(int64_t), h->stream));
        return DESC_B200_OK;
    }
    int64_t nt = (count + SCAN_TILE - 1) / SCAN_TILE;
    int64_t* sums = nullptr;
    CUDA_TRY(cudaMalloc(&sums, nt * sizeof(int64_t)));
    k_scan_tile_sums<<<(unsigned)nt, SCAN_TB, 0, h->stream>>>(in, count, sums);
    KERNEL_CHECK(h);
    k_scan_sums<<<1, 1024, 0, h->stream>>>(sums, nt);
    KERNEL_CHECK(h);
    k_scan_apply<<<(unsigned)nt, SCAN_TB, 0, h->stream>>>(in, count, sums, out);
    KERNEL_CHECK(h);
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    CUDA_TRY(cudaFree(sums));
    return DESC_B200_OK;
}

// ------------------------------------------------------------------------------------------
// A2: co-degree of every edge = popc(bm[i] & bm[j])  (replaces (A*A).*A, DESC.m:29)
// one warp per edge, 128-bit loads; consecutive edges share row i, so it stays in L1
// ------------------------------------------------------------------------------------------
__global__ void k_codeg(const int* __restrict__ ei, const int* __restrict__ ej, int64_t e0,
                        int64_t e1, const uint32_t* __restrict__ bm, int nwords,
                        int* __restrict__ codeg) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const int nq = nwords >> 2;
    for (int64_t e = e0 + warp; e < e1; e += nwarps) {
        const uint4* ri = reinterpret_cast<const uint4*>(bm + (size_t)ei[e] * nwords);
        const uint4* rj = reinterpret_cast<const uint4*>(bm + (size_t)ej[e] * nwords);
        int c = 0;
        for (int q = lane; q < nq; q += 32) {
            uint4 a = ri[q], b = rj[q];
            c += __popc(a.x & b.x) + __popc(a.y & b.y) + __popc(a.z & b.z) + __popc(a.w & b.w);
        }
        c = group_sum_int<32>(c);
        if (lane == 0) codeg[e] = c;
    }
}

__global__ void k_hist(const int* __restrict__ codeg, int64_t m, int* __restrict__ hist) {
    int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    int c = codeg[e];
    // warp-aggregate equal values (co-degrees cluster tightly around n*p^2)
    unsigned peers = __match_any_sync(__activemask(), c);
    if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&hist[c], __popc(peers));
}

__global__ void k_ns(const int* __restrict__ codeg, int64_t m, int n_sample, int* __restrict__ ns) {
    int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e < m) ns[e] = min(codeg[e], n_sample);
}

__global__ void k_ns_from_ptr(const int64_t* __restrict__ ptr, int64_t m, int* __restrict__ ns) {
    int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e < m) ns[e] = (int)(ptr[e + 1] - ptr[e]);
}

// ------------------------------------------------------------------------------------------
// A3: fill the incidence.  One warp per edge: enumerate common neighbours in ascending order
// from the AND of the two bitmap rows; if the co-degree exceeds the budget keep the n_sample
// smallest sampler keys (rank counting in shared memory); emit apex + packed partner edges.
// ------------------------------------------------------------------------------------------
struct FillArgs {
    const int *ei, *ej;
    const uint32_t* bm;
    const int* bmprefix;
    int nwords;
    const int *rowstart, *adj_eid;
    const int* codeg;
    const int64_t* rowptr;
    int* apex;              // global slot index
    uint32_t *pk_jk, *pk_ki;  // local slot index (slot - slot_base), may be null (apex only)
    uint16_t *rk_i, *rk_j;    // ranks of the apex in rows i / j (null: not wanted)
    int64_t e0, e1;         // edges to process
    int64_t l0, l1;         // local edge range for pk_* output
    int64_t slot_base;
    int n_sample, maxc;
    uint64_t seed;
    uint64_t* thr_key;      // per-edge sampler threshold (largest selected key, its apex); may be null
    int* thr_k;
};

__global__ void k_fill_slots(FillArgs a) {
    extern __shared__ unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int wpb = blockDim.x >> 5;
    // per-warp scratch: keys (8B) | k (4B) | sel (1B)
    const size_t per_warp = ((size_t)a.maxc * 13 + 15) & ~(size_t)15;
    unsigned char* base = smem_raw + per_warp * wib;
    uint64_t* ckey = reinterpret_cast<uint64_t*>(base);
    int* ck = reinterpret_cast<int*>(base + (size_t)a.maxc * 8);
    unsigned char* csel = base + (size_t)a.maxc * 12;

    const int64_t warp = (int64_t)blockIdx.x * wpb + wib;
    const int64_t nwarps = (int64_t)gridDim.x * wpb;
    for (int64_t e = a.e0 + warp; e < a.e1; e += nwarps) {
        const int c = a.codeg[e];
        if (c == 0) continue;
        const int i = a.ei[e], j = a.ej[e];
        const uint32_t* ri = a.bm + (size_t)i * a.nwords;
        const uint32_t* rj = a.bm + (size_t)j * a.nwords;
        // enumerate candidates in ascending k
        int run = 0;
        for (int wb = 0; wb < a.nwords; wb += 32) {
            int w = wb + lane;
            uint32_t x = (w < a.nwords) ? (ri[w] & rj[w]) : 0u;
            int cnt = __popc(x);
            int inc = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            int pos = run + inc - cnt;
            while (x) {
                int b = __ffs(x) - 1;
                x &= x - 1;
                ck[pos++] = (w << 5) + b;
            }
            run += __shfl_sync(0xffffffffu, inc, 31);
        }
        __syncwarp();
        const bool sample = c > a.n_sample;  // len==n_sample keeps everything (DESC.m:83)
        uint64_t tkey = ~0ull;               // threshold of an unsampled list: everything is a member
        int tk = 0x7fffffff;
        if (sample) {
            // keep the n_sample smallest (key, apex) pairs: MSB-first radix selection over the 64-bit keys.
            // csel: 0 = rejected, 1 = selected, 2 = undecided.  ~log2(c)+4 rounds instead of c^2/32 compares.
            for (int q = lane; q < c; q += 32) {
                ckey[q] = desc_key(a.seed, (uint64_t)e, (uint64_t)ck[q]);
                csel[q] = 2;
            }
            __syncwarp();
            int need = a.n_sample, und = c;
            for (int bit = 63; bit >= 0 && need > 0 && und > need; bit--) {
                int cnt0 = 0;
                for (int q = lane; q < c; q += 32) cnt0 += (csel[q] == 2) && !((ckey[q] >> bit) & 1ull);
                cnt0 = __reduce_add_sync(0xffffffffu, cnt0);
                if (cnt0 <= need) {   // all undecided keys with a 0 bit are among the smallest
                    for (int q = lane; q < c; q += 32)
                        if (csel[q] == 2 && !((ckey[q] >> bit) & 1ull)) csel[q] = 1;
                    need -= cnt0;
                    und -= cnt0;
                } else {              // the n_sample-th smallest has a 0 bit: keys with a 1 bit are out
                    for (int q = lane; q < c; q += 32)
                        if (csel[q] == 2 && ((ckey[q] >> bit) & 1ull)) csel[q] = 0;
                    und = cnt0;
                }
                __syncwarp();
            }
            // the rest: exactly `need` undecided keys left, or equal keys (smallest apices first: the
            // candidates are in ascending apex order)
            int taken = 0;
            for (int qb = 0; qb < c; qb += 32) {
                const int q = qb + lane;
                const bool u = q < c && csel[q] == 2;
                const unsigned bal = __ballot_sync(0xffffffffu, u);
                if (u) csel[q] = (taken + __popc(bal & ((1u << lane) - 1u))) < need ? 1 : 0;
                taken += __popc(bal);
            }
            __syncwarp();
            // threshold = largest selected (key, apex)
            uint64_t mk = 0ull;
            int mv = -1;
            for (int q = lane; q < c; q += 32)
                if (csel[q] == 1 && (ckey[q] > mk || (ckey[q] == mk && ck[q] > mv))) {
                    mk = ckey[q];
                    mv = ck[q];
                }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const uint64_t ok = __shfl_xor_sync(0xffffffffu, mk, o);
                const int ov = __shfl_xor_sync(0xffffffffu, mv, o);
                if (ok > mk || (ok == mk && ov > mv)) {
                    mk = ok;
                    mv = ov;
                }
            }
            tkey = mk;
            tk = mv;
        }
        if (a.thr_key && lane == 0) {
            a.thr_key[e] = tkey;
            a.thr_k[e] = tk;
        }
        // compaction + output
        const int64_t r0 = a.rowptr[e];
        const bool local = (e >= a.l0 && e < a.l1) && a.pk_jk != nullptr;
        int outpos = 0;
        for (int qb = 0; qb < c; qb += 32) {
            int q = qb + lane;
            bool sel = q < c && (!sample || csel[q] == 1);
            unsigned bal = __ballot_sync(0xffffffffu, sel);
            if (sel) {
                int p = outpos + __popc(bal & ((1u << lane) - 1u));
                int k = ck[q];
                a.apex[r0 + p] = k;
                if (local) {
                    const int ri_k = desc_rank(a.bm, a.bmprefix, a.nwords, i, k);
                    const int rj_k = desc_rank(a.bm, a.bmprefix, a.nwords, j, k);
                    int eik = a.adj_eid[a.rowstart[i] + ri_k];
                    int ejk = a.adj_eid[a.rowstart[j] + rj_k];
                    a.pk_ki[r0 - a.slot_base + p] = (uint32_t)eik | (i < k ? PK_SEL : 0u);
                    a.pk_jk[r0 - a.slot_base + p] = (uint32_t)ejk | (j < k ? PK_SEL : 0u);
                    if (a.rk_i) {
                        a.rk_i[r0 - a.slot_base + p] = (uint16_t)ri_k;
                        a.rk_j[r0 - a.slot_base + p] = (uint16_t)rj_k;
                    }
                }
            }
            outpos += __popc(bal);
        }
        __syncwarp();
    }
}

// Register-resident version of k_fill_slots for co-degrees up to 32 T (cfg 4: T = 8, cfg 2: T = 16): candidate
// q = lane + 32 t lives in register t of its lane.  The MSB-first radix selection then costs one ballot + popc per
// register and bit (no shared-memory state, no second pass to update it), and the bitmap rows are ANDed with 128-bit
// loads.  Same selection rule and the same outputs as k_fill_slots (bit-exact; tests compare both with the oracle).
template <int T>
__global__ void __launch_bounds__(256)
k_fill_slots_reg(FillArgs a) {
    extern __shared__ unsigned char smem_raw[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int wpb = blockDim.x >> 5;
    int* ck = reinterpret_cast<int*>(smem_raw) + (size_t)wib * (32 * T);
    const unsigned lt = (1u << lane) - 1u;
    const int nq = a.nwords >> 2;
    const int64_t warp = (int64_t)blockIdx.x * wpb + wib;
    const int64_t nwarps = (int64_t)gridDim.x * wpb;
    for (int64_t e = a.e0 + warp; e < a.e1; e += nwarps) {
        const int c = a.codeg[e];
        if (c == 0) continue;
        const int i = a.ei[e], j = a.ej[e];
        const uint4* ri = reinterpret_cast<const uint4*>(a.bm + (size_t)i * a.nwords);
        const uint4* rj = reinterpret_cast<const uint4*>(a.bm + (size_t)j * a.nwords);
        // common neighbours in ascending order -> ck[0..c)
        int run = 0;
        for (int qb = 0; qb < nq; qb += 32) {
            const int q = qb + lane;
            uint4 x = make_uint4(0u, 0u, 0u, 0u);
            if (q < nq) {
                const uint4 u = ri[q], v = rj[q];
                x = make_uint4(u.x & v.x, u.y & v.y, u.z & v.z, u.w & v.w);
            }
            const int cnt = __popc(x.x) + __popc(x.y) + __popc(x.z) + __popc(x.w);
            int inc = cnt;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, inc, o);
                if (lane >= o) inc += t;
            }
            int pos = run + inc - cnt;
            const uint32_t xs[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int wi = 0; wi < 4; wi++) {
                uint32_t y = xs[wi];
                while (y) {
                    const int b = __ffs(y) - 1;
                    y &= y - 1;
                    ck[pos++] = ((4 * q + wi) << 5) + b;
                }
            }
            run += __shfl_sync(0xffffffffu, inc, 31);
        }
        __syncwarp();
        int kk[T];
#pragma unroll
        for (int t = 0; t < T; t++) kk[t] = lane + 32 * t < c ? ck[lane + 32 * t] : -1;
        __syncwarp();
        const bool sample = c > a.n_sample;   // len==n_sample keeps everything (DESC.m:83)
        const int tmax = (c + 31) >> 5;       // registers that hold candidates (warp-uniform): skip the empty ones
        uint32_t sel = 0u;                    // bit t: candidate of register t is in the slot list
#pragma unroll
        for (int t = 0; t < T; t++) sel |= (kk[t] >= 0 ? 1u : 0u) << t;
        uint64_t tkey = ~0ull;
        int tk = 0x7fffffff;
        if (sample) {
            uint64_t key[T];
#pragma unroll
            for (int t = 0; t < T; t++) key[t] = (t < tmax && kk[t] >= 0) ? desc_key(a.seed, (uint64_t)e, (uint64_t)kk[t]) : ~0ull;
            uint32_t und = sel;
            sel = 0u;
            int need = a.n_sample, undc = c;
            for (int bit = 63; bit >= 0 && need > 0 && undc > need; bit--) {
                uint32_t zero = 0u;
                int cnt0 = 0;
#pragma unroll
                for (int t = 0; t < T; t++) {
                    if (t < tmax) {
                        const bool p = ((und >> t) & 1u) && !((key[t] >> bit) & 1ull);
                        cnt0 += __popc(__ballot_sync(0xffffffffu, p));
                        zero |= (p ? 1u : 0u) << t;
                    }
                }
                if (cnt0 <= need) {   // all undecided keys with a 0 bit are among the smallest
                    sel |= zero;
                    und &= ~zero;
                    need -= cnt0;
                    undc -= cnt0;
                } else {              // the n_sample-th smallest has a 0 bit: keys with a 1 bit are out
                    und = zero;
                    undc = cnt0;
                }
            }
            // the rest: exactly `need` undecided keys left, or equal keys (smallest apices first: candidates are in
            // ascending apex order, q = lane + 32 t)
            int taken = 0;
#pragma unroll
            for (int t = 0; t < T; t++) {
                if (t < tmax) {
                    const bool u = (und >> t) & 1u;
                    const unsigned bal = __ballot_sync(0xffffffffu, u);
                    if (u && taken + __popc(bal & lt) < need) sel |= 1u << t;
                    taken += __popc(bal);
                }
            }
            // threshold = largest selected (key, apex)
            uint64_t mk = 0ull;
            int mv = -1;
#pragma unroll
            for (int t = 0; t < T; t++)
                if (t < tmax && ((sel >> t) & 1u) && (key[t] > mk || (key[t] == mk && kk[t] > mv))) {
                    mk = key[t];
                    mv = kk[t];
                }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const uint64_t ok = __shfl_xor_sync(0xffffffffu, mk, o);
                const int ov = __shfl_xor_sync(0xffffffffu, mv, o);
                if (ok > mk || (ok == mk && ov > mv)) {
                    mk = ok;
                    mv = ov;
                }
            }
            tkey = mk;
            tk = mv;
        }
        if (a.thr_key && lane == 0) {
            a.thr_key[e] = tkey;
            a.thr_k[e] = tk;
        }
        const int64_t r0 = a.rowptr[e];
        const bool local = (e >= a.l0 && e < a.l1) && a.pk_jk != nullptr;
        const int rsi = a.rowstart[i], rsj = a.rowstart[j];
        int outpos = 0;
#pragma unroll
        for (int t = 0; t < T; t++) {
            if (32 * t >= c) break;
            const bool s1 = (sel >> t) & 1u;
            const unsigned bal = __ballot_sync(0xffffffffu, s1);
            if (s1) {
                const int p = outpos + __popc(bal & lt);
                const int k = kk[t];
                a.apex[r0 + p] = k;
                if (local) {
                    const int ri_k = desc_rank(a.bm, a.bmprefix, a.nwords, i, k);
                    const int rj_k = desc_rank(a.bm, a.bmprefix, a.nwords, j, k);
                    const int eik = a.adj_eid[rsi + ri_k];
                    const int ejk = a.adj_eid[rsj + rj_k];
                    a.pk_ki[r0 - a.slot_base + p] = (uint32_t)eik | (i < k ? PK_SEL : 0u);
                    a.pk_jk[r0 - a.slot_base + p] = (uint32_t)ejk | (j < k ? PK_SEL : 0u);
                    if (a.rk_i) {
                        a.rk_i[r0 - a.slot_base + p] = (uint16_t)ri_k;
                        a.rk_j[r0 - a.slot_base + p] = (uint16_t)rj_k;
                    }
                }
            }
            outpos += __popc(bal);
        }
    }
}

template <int T>
static int launch_fill_reg(desc_b200_handle* h, const FillArgs& fa) {
    const size_t smem = (size_t)8 * 32 * T * sizeof(int);
    CUDA_TRY(cudaFuncSetAttribute(k_fill_slots_reg<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int ctas = T <= 8 ? 8 : 4;
    k_fill_slots_reg<T><<<DESC_SMS * ctas, 256, smem, h->stream>>>(fa);
    KERNEL_CHECK(h);
    return DESC_B200_OK;
}

// explicit cycle lists: apex is given; compute packed partner edges and validate
__global__ void k_fill_explicit(FillArgs a, int* __restrict__ err) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t e = a.l0 + warp; e < a.l1; e += nwarps) {
        const int i = a.ei[e], j = a.ej[e];
        const int64_t r0 = a.rowptr[e], r1 = a.rowptr[e + 1];
        for (int64_t s = r0 + lane; s < r1; s += 32) {
            int k = a.apex[s];
            bool ok = k >= 0 && (k >> 5) < a.nwords;
            if (ok) {
                uint32_t bit = 1u << (k & 31);
                ok = (a.bm[(size_t)i * a.nwords + (k >> 5)] & bit) &&
                     (a.bm[(size_t)j * a.nwords + (k >> 5)] & bit);
            }
            if (!ok) {
                atomicOr(err, ERRB_APEX);
                continue;
            }
            const int ri_k = desc_rank(a.bm, a.bmprefix, a.nwords, i, k);
            const int rj_k = desc_rank(a.bm, a.bmprefix, a.nwords, j, k);
            int eik = a.adj_eid[a.rowstart[i] + ri_k];
            int ejk = a.adj_eid[a.rowstart[j] + rj_k];
            a.pk_ki[s - a.slot_base] = (uint32_t)eik | (i < k ? PK_SEL : 0u);
            a.pk_jk[s - a.slot_base] = (uint32_t)ejk | (j < k ? PK_SEL : 0u);
            if (a.rk_i) {
                a.rk_i[s - a.slot_base] = (uint16_t)ri_k;
                a.rk_j[s - a.slot_base] = (uint16_t)rj_k;
            }
            // a repeated apex within one edge (CEMP's with-replacement draw, CEMP.m:63) is legal for CEMP but not
            // for the PGD kernels (their table updates assume distinct apices per edge): record it in err[3]
            for (int64_t q = r0; q < s; q++)
                if (a.apex[q] == k) {
                    atomicOr(err + 3, 1);
                    break;
                }
        }
    }
}

// ------------------------------------------------------------------------------------------
// A4: reciprocal-slot flags.  Slot (ij;k): IKJ_appears <=> j is in the apex list of edge {i,k};
// JKI_appears <=> i is in the apex list of edge {j,k}  (DESC.m:111-125).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ bool apex_lsearch(const int* __restrict__ apex, int64_t lo, int64_t hi,
                                             int v) {
    for (int64_t s = lo; s < hi; s++)
        if (apex[s] == v) return true;
    return false;
}

// explicit cycle lists (in any order): a linear search of the partner edges' apex lists
__global__ void k_recip_flags(const int* __restrict__ ei, const int* __restrict__ ej,
                              const int64_t* __restrict__ rowptr, const int* __restrict__ apex,
                              uint32_t* __restrict__ pk_jk, uint32_t* __restrict__ pk_ki,
                              uint16_t* __restrict__ rk_i, uint16_t* __restrict__ rk_j, int64_t l0,
                              int64_t l1, int64_t slot_base) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t e = l0 + warp; e < l1; e += nwarps) {
        const int i = ei[e], j = ej[e];
        const int64_t r0 = rowptr[e], r1 = rowptr[e + 1];
        for (int64_t s = r0 + lane; s < r1; s += 32) {
            uint32_t pki = pk_ki[s - slot_base], pjk = pk_jk[s - slot_base];
            int64_t eik = pki & PK_MASK, ejk = pjk & PK_MASK;
            bool fa = apex_lsearch(apex, rowptr[eik], rowptr[eik + 1], j);
            bool fb = apex_lsearch(apex, rowptr[ejk], rowptr[ejk + 1], i);
            pk_ki[s - slot_base] = (pki & ~PK_APP) | (fa ? PK_APP : 0u);
            pk_jk[s - slot_base] = (pjk & ~PK_APP) | (fb ? PK_APP : 0u);
            if (rk_i) {
                rk_i[s - slot_base] = (uint16_t)((rk_i[s - slot_base] & RK_MASK) | (fa ? RK_APP : 0u) | (fb ? RK_APP2 : 0u));
                rk_j[s - slot_base] = (uint16_t)((rk_j[s - slot_base] & RK_MASK) | (fb ? RK_APP : 0u));
            }
        }
    }
}

// Reciprocal-slot flags for the hash sampler (DESC.m:98-127): apex j is in the sampled list of edge
// {i,k} iff (key(seed, e_ik, j), j) <= that edge's threshold pair: two table lookups per slot instead
// of two searches in the partner edges' apex lists.
__global__ void k_recip_flags_thr(const int* __restrict__ ei, const int* __restrict__ ej,
                                  const int64_t* __restrict__ rowptr, uint32_t* __restrict__ pk_jk,
                                  uint32_t* __restrict__ pk_ki, uint16_t* __restrict__ rk_i,
                                  uint16_t* __restrict__ rk_j, const uint64_t* __restrict__ thr_key,
                                  const int* __restrict__ thr_k, uint64_t seed, int64_t l0, int64_t l1,
                                  int64_t slot_base) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t e = l0 + warp; e < l1; e += nwarps) {
        const int i = ei[e], j = ej[e];
        const int64_t r0 = rowptr[e], r1 = rowptr[e + 1];
        for (int64_t s = r0 + lane; s < r1; s += 32) {
            const uint32_t pki = pk_ki[s - slot_base], pjk = pk_jk[s - slot_base];
            const int64_t eik = pki & PK_MASK, ejk = pjk & PK_MASK;
            const uint64_t ka = desc_key(seed, (uint64_t)eik, (uint64_t)j), ta = thr_key[eik];
            const uint64_t kb = desc_key(seed, (uint64_t)ejk, (uint64_t)i), tb = thr_key[ejk];
            const bool fa = ka < ta || (ka == ta && j <= thr_k[eik]);
            const bool fb = kb < tb || (kb == tb && i <= thr_k[ejk]);
            pk_ki[s - slot_base] = (pki & ~PK_APP) | (fa ? PK_APP : 0u);
            pk_jk[s - slot_base] = (pjk & ~PK_APP) | (fb ? PK_APP : 0u);
            if (rk_i) {
                rk_i[s - slot_base] = (uint16_t)((rk_i[s - slot_base] & RK_MASK) | (fa ? RK_APP : 0u) | (fb ? RK_APP2 : 0u));
                rk_j[s - slot_base] = (uint16_t)((rk_j[s - slot_base] & RK_MASK) | (fb ? RK_APP : 0u));
            }
        }
    }
}

// header of every adjacency position: (first local slot, slot count) of its edge; (0,0) for edges of
// other shards.  Lets the pass over larger endpoints find an in-edge's slot list with one load.
__global__ void k_jhdr(const int* __restrict__ adj_eid, const int64_t* __restrict__ rowptr, int64_t n2m,
                       int64_t e0, int64_t e1, int64_t slot_base, int2* __restrict__ jhdr) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n2m) return;
    const int64_t e = adj_eid[p];
    int2 h = make_int2(0, 0);
    if (e >= e0 && e < e1) h = make_int2((int)(rowptr[e] - slot_base), (int)(rowptr[e + 1] - rowptr[e]));
    jhdr[p] = h;
}

// slot-balanced contiguous edge ranges (SURVEY 8e): boundary r = first edge whose rowptr >= r*m_cycle/world
__global__ void k_shard_bounds(const int64_t* __restrict__ rowptr, int64_t m, int64_t m_cycle,
                               int world, int64_t* __restrict__ bounds) {
    int r = threadIdx.x;
    if (r > world) return;
    if (r == 0) {
        bounds[0] = 0;
        return;
    }
    if (r == world) {
        bounds[world] = m;
        return;
    }
    int64_t target = (m_cycle * r) / world;
    int64_t lo = 0, hi = m;
    while (lo < hi) {
        int64_t mid = (lo + hi) >> 1;
        if (rowptr[mid] < target)
            lo = mid + 1;
        else
            hi = mid;
    }
    bounds[r] = lo;
}

// rowptr at the first edge of every vertex block (cumulative slots per vertex), n+1 values
__global__ void k_vertex_slots(const int64_t* __restrict__ rowptr, const int* __restrict__ estart, int n,
                               int64_t* __restrict__ out) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v <= n) out[v] = rowptr[estart[v]];
}

// Vertex-aligned shard boundaries from a cost model instead of equal slot counts (round 2).  Per-rank times fitted
// on 2 and 8 B200 at cfg 4 (profiles/README.md): pass 1 costs its slots plus ~4.5 slot-equivalents per adjacency
// entry of every LOCAL vertex block (table prologue / flush of the CTA), pass 2 costs its slots (x1.2) plus ~3.9
// slot-equivalents per adjacency entry of every vertex ABOVE the rank's first vertex (each of them gets a CTA with
// a full table).  The passes are separated by the exchange of S, so the iteration takes max(pass 1) + max(pass 2):
// coordinate descent on the N-1 boundaries from the slot-balanced start.  cs[v] = cumulative slots before vertex
// block v, ca[v] = cumulative adjacency entries (rowstart).
static void cost_model_bounds(const std::vector<int64_t>& cs, const std::vector<int>& ca, int n, int W,
                              std::vector<int>& vb) {
    const double k1 = 4.5, k2 = 3.9, b2 = 1.2;
    auto objective = [&](const std::vector<int>& b) {
        double m1 = 0.0, m2 = 0.0;
        for (int r = 0; r < W; r++) {
            const double slots = (double)(cs[b[r + 1]] - cs[b[r]]);
            m1 = std::max(m1, slots + k1 * (double)(ca[b[r + 1]] - ca[b[r]]));
            m2 = std::max(m2, slots > 0.0 ? b2 * slots + k2 * (double)(ca[n] - ca[b[r]]) : 0.0);
        }
        return m1 + m2;
    };
    double best = objective(vb);
    for (int step = std::max(1, n / 16); step >= 1; step /= 2) {
        bool moved = true;
        for (int sweep = 0; sweep < 64 && moved; sweep++) {
            moved = false;
            for (int r = 1; r < W; r++) {
                for (int dir = -1; dir <= 1; dir += 2) {
                    std::vector<int> t = vb;
                    t[r] = std::min(std::max(t[r] + dir * step, t[r - 1]), t[r + 1]);
                    if (t[r] == vb[r]) continue;
                    const double o = objective(t);
                    if (o < best * (1.0 - 1e-9)) {
                        best = o;
                        vb = t;
                        moved = true;
                    }
                }
            }
        }
    }
}

// The shard plan as a host-only entry point (no device needed): CPU tests pin the rule, and a caller can ask where
// the boundaries of a world would fall.  cum_slots[v] = slots of the vertex blocks before v (n+1 values),
// cum_adj[v] = adjacency entries before v (n+1 values); v_bounds gets world+1 vertex boundaries: the slot-balanced
// start (the vertex block that contains the r/world point of the slots; the build finds it on the device with
// k_shard_bounds) followed by the same cost-model descent desc_b200_build_incidence runs on a multi-GPU handle.
extern "C" int desc_b200_plan_shards(int32_t n, int32_t world, const int64_t* cum_slots, const int32_t* cum_adj,
                                     int32_t slots_only, int32_t* v_bounds) {
    if (n <= 0 || world < 1 || world > 64 || !cum_slots || !cum_adj || !v_bounds) {
        desc_set_error("plan_shards: bad arguments");
        return DESC_B200_ERR_ARG;
    }
    std::vector<int64_t> cs(cum_slots, cum_slots + n + 1);
    std::vector<int> ca(cum_adj, cum_adj + n + 1);
    std::vector<int> vb(world + 1, 0);
    vb[world] = n;
    for (int r = 1; r < world; r++) {   // first vertex block starting at or after r/world of the slots (k_shard_bounds + alignment)
        const int64_t target = (cs[n] * r) / world;
        int v = (int)(std::lower_bound(cs.begin(), cs.end(), target) - cs.begin());
        // k_shard_bounds picks the first EDGE whose rowptr >= target and the shard starts at that edge's vertex block
        if (v > 0 && cs[v] > target) v -= 1;
        vb[r] = std::min(std::max(v, vb[r - 1]), n);
    }
    if (!slots_only && world > 1) cost_model_bounds(cs, ca, n, world, vb);
    for (int r = 0; r <= world; r++) v_bounds[r] = vb[r];
    return DESC_B200_OK;
}

static void free_incidence(desc_b200_handle* h) {
    cudaFree(h->rowptr);
    cudaFree(h->apex);
    cudaFree(h->pk_jk);
    cudaFree(h->pk_ki);
    cudaFree(h->S0);
    cudaFree(h->rk_i);
    cudaFree(h->rk_j);
    cudaFree(h->jhdr);
    cudaFree(h->sjk);
    h->rk_i = h->rk_j = nullptr;
    h->jhdr = nullptr;
    h->sjk = nullptr;
    h->adam_valid = false;
    h->has_dup_apex = false;
    for (int b = 0; b < 2; b++) {
        cudaFree(h->w[b]);
        h->w[b] = nullptr;
    }
    cudaFree(h->adam_m);
    cudaFree(h->adam_v);
    h->rowptr = nullptr;
    h->apex = nullptr;
    h->pk_jk = h->pk_ki = nullptr;
    h->S0 = nullptr;
    h->adam_m = h->adam_v = nullptr;
    h->built = h->have_s0 = h->have_pgd = h->have_cemp = false;
}

int desc_build_incidence_impl(desc_b200_handle* h, int n_sample_req, uint64_t seed,
                              const int64_t* cyc_ptr, const int32_t* cyc_apex) {
    const int64_t m = h->m;
    const int n = h->n;
    cudaStream_t st = h->stream;
    const int TB = 256;
    const unsigned gb = (unsigned)((m + TB - 1) / TB);
    free_incidence(h);
    if (!h->codeg) CUDA_TRY(cudaMalloc(&h->codeg, m * sizeof(int)));
    const int warp_grid = DESC_SMS * 8;  // 8 CTAs of 8 warps per SM, grid-stride over edges

    // ---- co-degrees of all edges.  Multi-GPU: every rank counts an equal slice, then all-gather.
    {
        std::vector<int64_t> b(h->world + 1);
        for (int r = 0; r <= h->world; r++) b[r] = (m * r) / h->world;
        k_codeg<<<warp_grid, 256, 0, st>>>(h->ei, h->ej, b[h->rank], b[h->rank + 1], h->bm, h->nwords,
                                           h->codeg);
        KERNEL_CHECK(h);
        DESC_TRY(desc_allgather_ranges(h, h->codeg, sizeof(int), b));
    }
    // ---- histogram -> m_pos, max co-degree, sampling budget (DESC.m:36-43)
    DescTmp t_hist;
    CUDA_TRY(t_hist.alloc((size_t)(n + 1) * sizeof(int)));
    int* d_hist = t_hist.as<int>();
    CUDA_TRY(cudaMemsetAsync(d_hist, 0, (size_t)(n + 1) * sizeof(int), st));
    k_hist<<<gb, TB, 0, st>>>(h->codeg, m, d_hist);
    KERNEL_CHECK(h);
    std::vector<int> hist(n + 1);
    CUDA_TRY(cudaMemcpyAsync(hist.data(), d_hist, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    t_hist.release();
    int64_t m_pos = 0;
    int maxc = 0;
    for (int c = 1; c <= n; c++)
        if (hist[c]) {
            m_pos += hist[c];
            maxc = c;
        }
    h->m_pos = m_pos;
    h->max_codeg = maxc;

    DescTmp t_ns;   // (freed on the argument-error returns below as well)
    CUDA_TRY(t_ns.alloc(m * sizeof(int)));
    int* d_ns = t_ns.as<int>();
    CUDA_TRY(cudaMalloc(&h->rowptr, (m + 4) * sizeof(int64_t)));   // +3: 16-byte widened bulk copies (pgd_stream.cuh)
    const bool explicit_lists = cyc_ptr != nullptr;
    if (explicit_lists) {
        if (!cyc_apex) {
            desc_set_error("cyc_ptr given without cyc_apex");
            return DESC_B200_ERR_ARG;
        }
        if (cyc_ptr[0] != 0) {
            desc_set_error("cyc_ptr[0] must be 0");
            return DESC_B200_ERR_ARG;
        }
        int mx = 0;
        for (int64_t e = 0; e < m; e++) {
            int64_t d = cyc_ptr[e + 1] - cyc_ptr[e];
            if (d < 0 || d > n) {
                desc_set_error("cyc_ptr is not a valid row pointer at edge %lld", (long long)e);
                return DESC_B200_ERR_ARG;
            }
            mx = std::max<int>(mx, (int)d);
        }
        h->n_sample = mx;
        h->m_cycle = cyc_ptr[m];
        CUDA_TRY(cudaMemcpyAsync(h->rowptr, cyc_ptr, (m + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        k_ns_from_ptr<<<gb, TB, 0, st>>>(h->rowptr, m, d_ns);
        KERNEL_CHECK(h);
    } else {
        int ns;
        if (n_sample_req > 0)
            ns = n_sample_req;
        else if (n_sample_req < 0)
            ns = std::max(maxc, 1);
        else {
            // MATLAB median of the positive co-degrees from the histogram (DESC.m:43)
            double med = 0.0;
            if (m_pos > 0) {
                int64_t lo_idx = (m_pos - 1) / 2, hi_idx = m_pos / 2;  // 0-based order statistics
                int64_t cum = 0;
                int vlo = -1, vhi = -1;
                for (int c = 1; c <= n && vhi < 0; c++) {
                    cum += hist[c];
                    if (vlo < 0 && cum > lo_idx) vlo = c;
                    if (vhi < 0 && cum > hi_idx) vhi = c;
                }
                med = 0.5 * ((double)vlo + (double)vhi);
            }
            ns = std::max((int)std::ceil(med / 4.0), 30);
        }
        h->n_sample = ns;
        k_ns<<<gb, TB, 0, st>>>(h->codeg, m, ns, d_ns);
        KERNEL_CHECK(h);
        DESC_TRY(desc_exclusive_scan_i64(h, d_ns, h->rowptr, m));
        CUDA_TRY(cudaMemcpyAsync(&h->m_cycle, h->rowptr + m, sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
    }
    h->max_ns = std::min(h->n_sample, std::max(maxc, 1));
    if (explicit_lists) h->max_ns = h->n_sample;
    t_ns.release();

    // ---- shard: slot-balanced contiguous edge ranges
    h->shard_edges.assign(h->world + 1, 0);
    {
        int64_t* d_b = nullptr;
        CUDA_TRY(cudaMalloc(&d_b, (h->world + 1) * sizeof(int64_t)));
        k_shard_bounds<<<1, 64, 0, st>>>(h->rowptr, m, h->m_cycle, h->world, d_b);
        KERNEL_CHECK(h);
        CUDA_TRY(cudaMemcpyAsync(h->shard_edges.data(), d_b, (h->world + 1) * sizeof(int64_t),
                                 cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        CUDA_TRY(cudaFree(d_b));
    }
    // align shard boundaries to vertex blocks (all edges with the same smaller endpoint stay together)
    {
        std::vector<int> v_of(h->world + 1, 0);
        v_of[h->world] = n;
        for (int r = 1; r < h->world; r++) {
            if (h->shard_edges[r] >= m) {
                v_of[r] = n;
                h->shard_edges[r] = m;
            } else {
                CUDA_TRY(cudaMemcpy(&v_of[r], h->ei + h->shard_edges[r], sizeof(int), cudaMemcpyDeviceToHost));
                h->shard_edges[r] = h->h_estart[v_of[r]];
            }
        }
        // cost-model boundaries
        if (h->world > 1 && h->blocked_ok) {
            DescTmp t_cs;
            CUDA_TRY(t_cs.alloc((size_t)(n + 1) * sizeof(int64_t)));
            k_vertex_slots<<<(n + 1 + 255) / 256, 256, 0, st>>>(h->rowptr, h->estart, n, t_cs.as<int64_t>());
            KERNEL_CHECK(h);
            std::vector<int64_t> cs(n + 1);
            std::vector<int> ca(n + 1);
            CUDA_TRY(cudaMemcpyAsync(cs.data(), t_cs.p, (size_t)(n + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaMemcpyAsync(ca.data(), h->rowstart, (size_t)(n + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            cost_model_bounds(cs, ca, n, h->world, v_of);
            for (int r = 1; r < h->world; r++) h->shard_edges[r] = h->h_estart[v_of[r]];
        }
        h->v_begin = v_of[h->rank];
        h->v_end = v_of[h->rank + 1];
    }
    h->e_begin = h->shard_edges[h->rank];
    h->e_end = h->shard_edges[h->rank + 1];
    h->shard_slots.assign(h->world + 1, 0);
    for (int r = 0; r <= h->world; r++)
        CUDA_TRY(cudaMemcpyAsync(&h->shard_slots[r], h->rowptr + h->shard_edges[r], sizeof(int64_t),
                                 cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    h->slot_base = h->shard_slots[h->rank];
    h->n_slots = h->shard_slots[h->rank + 1] - h->slot_base;

    // + 16: the streamed PGD kernel widens its bulk copies to 16-byte boundaries (pgd_stream.cuh)
    const size_t ns_alloc = (size_t)std::max<int64_t>(h->n_slots, 1) + 16;
    CUDA_TRY(cudaMalloc(&h->apex, (size_t)std::max<int64_t>(h->m_cycle, 1) * sizeof(int)));
    CUDA_TRY(cudaMalloc(&h->pk_jk, ns_alloc * sizeof(uint32_t)));
    CUDA_TRY(cudaMalloc(&h->pk_ki, ns_alloc * sizeof(uint32_t)));
    CUDA_TRY(cudaMalloc(&h->S0, ns_alloc * sizeof(double)));
    if (h->blocked_ok && h->n_slots < (1ll << 31) - 64) {   // (jhdr holds 32-bit local slot offsets)
        CUDA_TRY(cudaMalloc(&h->rk_i, ns_alloc * sizeof(uint16_t)));
        CUDA_TRY(cudaMalloc(&h->rk_j, ns_alloc * sizeof(uint16_t)));
        CUDA_TRY(cudaMalloc(&h->sjk, ns_alloc * sizeof(double)));
        CUDA_TRY(cudaMalloc(&h->jhdr, (size_t)(2 * m + 32) * sizeof(int2)));
        k_jhdr<<<(unsigned)((2 * m + TB - 1) / TB), TB, 0, st>>>(h->adj_eid, h->rowptr, 2 * m, h->e_begin, h->e_end,
                                                               h->slot_base, h->jhdr);
        KERNEL_CHECK(h);
    }
    CUDA_TRY(cudaMalloc(&h->w[0], ns_alloc * sizeof(double)));
    CUDA_TRY(cudaMalloc(&h->w[1], ns_alloc * sizeof(double)));

    FillArgs fa;
    fa.ei = h->ei;
    fa.ej = h->ej;
    fa.bm = h->bm;
    fa.bmprefix = h->bmprefix;
    fa.nwords = h->nwords;
    fa.rowstart = h->rowstart;
    fa.adj_eid = h->adj_eid;
    fa.codeg = h->codeg;
    fa.rowptr = h->rowptr;
    fa.apex = h->apex;
    fa.pk_jk = h->pk_jk;
    fa.pk_ki = h->pk_ki;
    fa.rk_i = h->rk_i;
    fa.rk_j = h->rk_j;
    fa.e0 = h->e_begin;
    fa.e1 = h->e_end;
    fa.l0 = h->e_begin;
    fa.l1 = h->e_end;
    fa.slot_base = h->slot_base;
    fa.n_sample = h->n_sample;
    fa.maxc = std::max(maxc, 1);
    fa.seed = seed;
    fa.thr_key = nullptr;
    fa.thr_k = nullptr;
    if (h->m_cycle > 0) {
        if (explicit_lists) {
            CUDA_TRY(cudaMemcpyAsync(h->apex, cyc_apex, h->m_cycle * sizeof(int), cudaMemcpyHostToDevice, st));
            k_fill_explicit<<<warp_grid, 256, 0, st>>>(fa, h->d_err);
            KERNEL_CHECK(h);
            int herr4[4] = {0, 0, 0, 0};
            CUDA_TRY(cudaMemcpyAsync(herr4, h->d_err, sizeof(herr4), cudaMemcpyDeviceToHost, st));
            CUDA_TRY(cudaStreamSynchronize(st));
            const int herr = herr4[0];
            h->has_dup_apex = herr4[3] != 0;
            if (herr4[3]) CUDA_TRY(cudaMemsetAsync(h->d_err + 3, 0, sizeof(int), st));
            if (herr & ERRB_APEX) {
                CUDA_TRY(cudaMemsetAsync(h->d_err, 0, sizeof(int), st));
                desc_set_error("explicit cycle list contains an apex that is not a common neighbour");
                return DESC_B200_ERR_ARG;
            }
        } else {
            const size_t per_warp = ((size_t)fa.maxc * 13 + 15) & ~(size_t)15;
            int wpb = 8;
            while (wpb > 1 && per_warp * wpb > 200 * 1024) wpb >>= 1;
            if (per_warp * wpb > 220 * 1024) {
                desc_set_error("max co-degree %d exceeds the shared-memory sampler scratch", maxc);
                return DESC_B200_ERR_LIMIT;
            }
            const size_t smem = per_warp * wpb;
            CUDA_TRY(cudaFuncSetAttribute(k_fill_slots, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int ctas_per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / std::max<size_t>(smem, 1)));
            if (!h->thr_key) {
                CUDA_TRY(cudaMalloc(&h->thr_key, (size_t)m * sizeof(uint64_t)));
                CUDA_TRY(cudaMalloc(&h->thr_k, (size_t)m * sizeof(int)));
            }
            fa.thr_key = h->thr_key;
            fa.thr_k = h->thr_k;
            // register-resident selection for co-degrees up to 512.  Above, the shared-memory kernel: 32 candidate
            // registers per lane needed 242 registers per thread and took 43 ms against its 11.5 ms at cfg 3
            // (co-degrees ~500, profiles/README.md round 2)
            if (maxc <= 128) {
                DESC_TRY(launch_fill_reg<4>(h, fa));
            } else if (maxc <= 256) {
                DESC_TRY(launch_fill_reg<8>(h, fa));
            } else if (maxc <= 512) {
                DESC_TRY(launch_fill_reg<16>(h, fa));
            } else {
                k_fill_slots<<<DESC_SMS * ctas_per_sm, wpb * 32, smem, st>>>(fa);
                KERNEL_CHECK(h);
            }
            // every rank needs every edge's apex list (getters, explicit replays) and sampler threshold
            DESC_TRY(desc_allgather_ranges(h, h->apex, sizeof(int), h->shard_slots));
            DESC_TRY(desc_allgather_ranges(h, h->thr_key, sizeof(uint64_t), h->shard_edges));
            DESC_TRY(desc_allgather_ranges(h, h->thr_k, sizeof(int), h->shard_edges));
        }
        if (!explicit_lists) {
            k_recip_flags_thr<<<warp_grid, 256, 0, st>>>(h->ei, h->ej, h->rowptr, h->pk_jk, h->pk_ki, h->rk_i, h->rk_j,
                                                         h->thr_key, h->thr_k, seed, h->e_begin, h->e_end, h->slot_base);
        } else {
            k_recip_flags<<<warp_grid, 256, 0, st>>>(h->ei, h->ej, h->rowptr, h->apex, h->pk_jk, h->pk_ki, h->rk_i,
                                                     h->rk_j, h->e_begin, h->e_end, h->slot_base);
        }
        KERNEL_CHECK(h);
    }
    h->built = true;
    return DESC_B200_OK;
}
