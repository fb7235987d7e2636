// Internal declarations shared by the translation units of libdesc_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <vector>

#include "../../include/desc_b200.h"

#include <string.h>

// ---- pooled device memory (pool.cu): every cudaMalloc / cudaFree of the library goes through it
cudaError_t desc_pool_malloc(void** p, size_t bytes);
cudaError_t desc_pool_free(void* p);
cudaError_t desc_raw_malloc(void** p, size_t bytes);
cudaError_t desc_raw_free(void* p);
#define cudaMalloc(p, n) desc_pool_malloc((void**)(p), (n))
#define cudaFree(p) desc_pool_free((void*)(p))

// temporary device buffer that returns to the pool on every exit path (error returns included)
struct DescTmp {
    void* p = nullptr;
    DescTmp() = default;
    DescTmp(const DescTmp&) = delete;
    DescTmp& operator=(const DescTmp&) = delete;
    ~DescTmp() { release(); }
    cudaError_t alloc(size_t bytes) { return desc_pool_malloc(&p, bytes); }
    void release() {
        if (p) desc_pool_free(p);
        p = nullptr;
    }
    template <class T>
    T* as() const { return static_cast<T*>(p); }
};

// ---- error plumbing -----------------------------------------------------------------
void desc_set_error(const char* fmt, ...);

#define CUDA_TRY(expr)                                                                        \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            desc_set_error("CUDA error %s at %s:%d: %s", cudaGetErrorName(_e), __FILE__,      \
                           __LINE__, cudaGetErrorString(_e));                                 \
            return DESC_B200_ERR_CUDA;                                                        \
        }                                                                                     \
    } while (0)

#define DESC_TRY(expr)                                                                        \
    do {                                                                                      \
        int _r = (expr);                                                                      \
        if (_r != DESC_B200_OK) return _r;                                                    \
    } while (0)

#define KERNEL_CHECK(h)                                                                       \
    do {                                                                                      \
        (h)->launches++;                                                                      \
        CUDA_TRY(cudaGetLastError());                                                         \
    } while (0)

// ---- packed partner-edge words ------------------------------------------------------
// pk_ki = e_ki | (i<k ? SEL : 0) | (IKJ_appears ? APP : 0)
// pk_jk = e_jk | (j<k ? SEL : 0) | (JKI_appears ? APP : 0)
// SEL says the vertex shared with the partner edge is that edge's smaller endpoint; it selects
// the partner-sum accumulator (0 = via min endpoint, 1 = via max endpoint) and, for d_ijk, the
// orientation of the stored relative rotation.
#define PK_APP 0x80000000u
#define PK_SEL 0x40000000u
#define PK_MASK 0x3FFFFFFFu
// rank words (vertex-blocked / streamed PGD): rank of the apex in the adjacency row of i (rk_i) or
// j (rk_j) in 14 bits; bit 15 = IKJ_appears (rk_i) / JKI_appears (rk_j); bit 14 of rk_i = JKI_appears
#define RK_APP 0x8000u
#define RK_APP2 0x4000u
#define RK_MASK 0x3FFFu
// vertex-blocked PGD: shared memory per CTA = 8 B * (1 + warps) * padded max degree
#define DESC_BLOCKED_MAXDEG 5000   // (< 2^14: the rank field)
#define DESC_MAX_EDGES 0x3FFFFFFFll

static constexpr int DESC_SMS = 148;  // B200
static constexpr int DESC_GCW_MAXIT = 4000;

struct desc_b200_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int rank = 0, world = 1;
    void* comm = nullptr;       // ncclComm_t (comm.cu)
    void* comm_scratch = nullptr;   // receive buffer of desc_reduce_to_owners
    size_t comm_scratch_bytes = 0;
    int launches = 0;
    int collectives = 0;
    void* sym = nullptr;        // peer-mapped symmetric region of this rank's communicator (comm.cu), or null
    bool S_in_sym = false;      // S[0], S[1] live inside the symmetric region (not pool blocks)

    // graph ---------------------------------------------------------------------------
    int n = 0;
    int64_t m = 0;
    int* ei = nullptr;          // m, 0-based smaller endpoint
    int* ej = nullptr;          // m
    const double* Rij = nullptr;  // 9m, MATLAB layout
    double* Rij_owned = nullptr;
    int nwords = 0;             // 32-bit words per adjacency bitmap row
    uint32_t* bm = nullptr;     // n x nwords adjacency bitmap
    int* bmprefix = nullptr;    // n x nwords: set bits before each word of the row
    int* rowstart = nullptr;    // n+1: CSR offsets of the symmetric adjacency
    int* adj_nbr = nullptr;     // 2m: neighbours, ascending within a row
    int* adj_eid = nullptr;     // 2m: edge id of (row, neighbour)
    int* adj_mirror = nullptr;  // m+4: adjacency position of i in row j, for edge (i,j)

    // incidence -----------------------------------------------------------------------
    bool built = false, have_s0 = false, have_pgd = false;
    int* codeg = nullptr;       // m
    uint64_t* thr_key = nullptr;  // m: sampler threshold of every edge = largest selected (key, apex) pair;
    int* thr_k = nullptr;         //    membership of an apex in an edge's sampled list is then one comparison
    int n_sample = 0, max_codeg = 0, max_ns = 0;
    int64_t m_pos = 0, m_cycle = 0;
    int64_t* rowptr = nullptr;  // m+1 over ALL edges (empty rows for edges without triangles)
    int* apex = nullptr;        // m_cycle (global): k of every slot
    int64_t e_begin = 0, e_end = 0;   // local edge range (sharding); [0,m) when world==1
    int64_t slot_base = 0, n_slots = 0;  // local slots = [slot_base, slot_base+n_slots)
    std::vector<int64_t> shard_edges;  // world+1 edge boundaries
    std::vector<int64_t> shard_slots;  // world+1 slot boundaries (rowptr at shard_edges)
    uint32_t* pk_jk = nullptr;  // n_slots
    uint32_t* pk_ki = nullptr;  // n_slots
    // vertex-blocked PGD path (pgd.cu): rank of the apex k in the adjacency row of i (resp. j),
    // bit 15 = IKJ_appears (resp. JKI_appears).  Null when a degree exceeds the 15-bit/shared-memory limit.
    uint16_t* rk_i = nullptr;   // n_slots
    uint16_t* rk_j = nullptr;   // n_slots
    int2* jhdr = nullptr;       // 2m: per adjacency position (v, u<v): local first slot and slot count of edge (u,v)
    double* sjk = nullptr;      // n_slots: S[e_jk] of the current state, written by the pass over larger endpoints
    int* estart = nullptr;      // n+1: first edge whose smaller endpoint is >= v (edges are (i,j)-sorted)
    std::vector<int> h_estart;  // host copy
    int maxdeg = 0;
    int v_begin = 0, v_end = 0; // local vertex range (shards are aligned to vertex blocks)
    bool blocked_ok = false;    // the vertex-blocked path is usable for this graph
    double* pgd_partial = nullptr;  // 2 per CTA: objective / change partials (deterministic reduction)
    std::vector<cudaEvent_t> iter_events;  // per-iteration kernel timing
    double* S0 = nullptr;       // n_slots
    bool has_dup_apex = false;  // explicit cycle lists that repeat an apex within an edge (CEMP's with-replacement draw)

    // PGD state -------------------------------------------------------------------------
    double* w[2] = {nullptr, nullptr};     // n_slots each (ping-pong)
    double* S[2] = {nullptr, nullptr};     // m each
    double* acc[2] = {nullptr, nullptr};   // 2m+2 each: partner sums via min/max endpoint, + [obj, change]
    double* P1 = nullptr;                   // 2m (streamed path, one GPU): pass 1's partner sums in adjacency order
    double* S_adj[2] = {nullptr, nullptr};  // 2m+4 each (streamed path): S in adjacency order; [1] on one GPU only
    double* adam_m = nullptr;
    double* adam_v = nullptr;
    bool adam_valid = false;                // the Adam moments on this handle continue a rule with t > 0
    int final_buf = 0;                      // which ping-pong buffer holds the result
    double* d_hist = nullptr;               // 2*iters
    int hist_cap = 0;
    int* d_ctrl = nullptr;                  // [0]=stopped [1]=final_iter [2]=misses
    double* d_ctrl_f = nullptr;             // [0]=previous objective
    int* h_ctrl = nullptr;                  // pinned mirror of d_ctrl

    // GCW -------------------------------------------------------------------------------
    double* omega = nullptr;    // m
    double* isd = nullptr;      // n: 1/sqrt(d_i)
    double* X[2] = {nullptr, nullptr};  // 9n each
    double* gcw_coef = nullptr; // m: omega_e / sqrt(d_i d_j)
    double* gcw_coef_adj = nullptr;  // 2m: the same in adjacency order (streamed by the SpMV)
    std::vector<cudaEvent_t> spmv_events;
    double* gcw_red = nullptr;  // reduction scratch
    double* gcw_small = nullptr;  // 3x3 transforms etc.
    double* gcw_res = nullptr;  // residual history (device)
    double* gcw_res_host = nullptr;  // pinned mirror
    double gcw_last_res = 0.0;
    double gcw_theta[3] = {0.0, 0.0, 0.0};  // Ritz values of the last gcw call
    double* R_est = nullptr;    // 9n
    double* d_Sin = nullptr;    // m: S_vec passed to gcw from the host
    bool have_gcw = false;
    int laa_cg_iters = 0;       // CG iterations of the last refine call
    int gcw_weight_rule = 0;    // 0: GCW.m:20 (s^1.5), 1: CEMP_GCW.m:141 (s)

    // CEMP (cemp.cu) --------------------------------------------------------------------
    double* cemp_S[2] = {nullptr, nullptr};  // m each (ping-pong)
    int cemp_final = 0;
    bool have_cemp = false;
    double* R_mst = nullptr;    // 9n: CEMP+MST rotations of the last mst_init
    bool have_mst = false;

    // make_plots diagnostics (diag.cu): per-iteration S_vec error, GCW, alignment (DESC.m:235-239)
    bool diag_on = false;
    const double* diag_err = nullptr;   // ErrVec on the device (m)
    const double* diag_Rgt = nullptr;   // R_orig on the device (9n)
    double* diag_out = nullptr;         // host, 3 per iteration
    int diag_cap = 0;
    double* diag_work = nullptr;        // device scratch of the alignment
    unsigned* diag_hist = nullptr;      // radix-select histogram

    // scratch ---------------------------------------------------------------------------
    int* d_err = nullptr;       // device error flags
    desc_b200_timings tm = {};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr, ev3 = nullptr;
};

// ---- stage implementations (one .cu each) ---------------------------------------------
int desc_graph_setup(desc_b200_handle* h, const double* d_Ind);
int desc_build_incidence_impl(desc_b200_handle* h, int n_sample, uint64_t seed,
                              const int64_t* cyc_ptr, const int32_t* cyc_apex);
int desc_cycle_impl(desc_b200_handle* h);
int desc_pgd_impl(desc_b200_handle* h, int iters, desc_b200_step_rule* rule, int* iters_run);
int desc_gcw_impl(desc_b200_handle* h, const double* d_S);
// per-iteration parameters of the MPLS loop (MPLS.m:39-63), padded to `len` by the caller; nullptr = DESC.m:265-312
struct desc_laa_sched {
    const double* beta;    // reweighting
    const double* tau;     // thresholding
    const double* alpha;   // cycle_info_ratio
    int len;
    double empty_value;    // HVec of edges without a 3-cycle: acos(-1/2)/pi (zero R_cycle, MPLS.m:125-135)
};
int desc_laa_impl(desc_b200_handle* h, const double* d_S, const double* d_Rinit, double* d_Rout, int max_iters,
                  double stop_threshold, int* iters_run, double* scores_host, const desc_laa_sched* mpls = nullptr);
// MPLS.m:152-195: minimum spanning tree of SVec+1 and rotations multiplied along it from node 1 (mpls.cu)
int desc_mst_init_impl(desc_b200_handle* h, const double* d_S, double* d_R);
int desc_cemp_impl(desc_b200_handle* h, int max_iter, const double* beta, int n_beta);
int desc_cemp_reweight(desc_b200_handle* h, const double* x_cur, double* x_next, double beta, double empty_value);
// Rotation_Alignment.m on the device: out[0]=mean error, out[1]=median error (degrees), out[2..10]=R_align;
// d_Rout (may be null) receives R_est*R_align
int desc_align_impl(desc_b200_handle* h, const double* d_Rest, const double* d_Rgt, double* d_Rout, double out[11]);
// called by the PGD loop after iteration t when h->diag_on (DESC.m:235-239)
int desc_diag_record(desc_b200_handle* h, int t, const double* d_S);
// k-th smallest (1-based) of non-negative doubles on the device (laa.cu); d_hist: 2048 unsigned
int desc_select_kth(desc_b200_handle* h, const double* X, int64_t m, int64_t k, unsigned* d_hist, double* out);
int desc_exclusive_scan_i64(desc_b200_handle* h, const int* in, int64_t* out, int64_t count);

// multi-GPU collectives (comm.cu); no-ops when world==1
int desc_comm_init(desc_b200_handle* h, const void* nccl_id);
void desc_comm_destroy(desc_b200_handle* h);
int desc_allreduce_sum(desc_b200_handle* h, double* buf, int64_t count);
int desc_allgather_ranges(desc_b200_handle* h, void* buf, size_t elem_bytes,
                          const std::vector<int64_t>& bounds);
int desc_reduce_to_owners(desc_b200_handle* h, double* buf, int width, const std::vector<int64_t>& bounds,
                          int tail);
// Peer-memory exchanges of the PGD iteration (comm.cu): S[0], S[1] and a receive scratch live in a region that every
// rank maps from every peer (CUDA IPC over NVLink); the exchanges are plain stores into the peers' memory plus a
// flag barrier.  desc_sym_setup returns DESC_B200_OK with h->sym == nullptr when peer mapping is unavailable or
// DESC_B200_COMM selects NCCL.
int desc_sym_setup(desc_b200_handle* h, int64_t m, const std::vector<int64_t>& bounds);
double* desc_sym_S_buffer(desc_b200_handle* h, int which);
int desc_sym_barrier(desc_b200_handle* h);
int desc_sym_allgather_S(desc_b200_handle* h, int which, const std::vector<int64_t>& bounds);
int desc_sym_reduce_to_owners(desc_b200_handle* h, double* buf, const std::vector<int64_t>& bounds);

// ---- device helpers -----------------------------------------------------------------
#ifdef __CUDACC__
// 64-bit sampler key of (edge, apex); bit-identical to oracle/desc_oracle.py::sampler_keys
__host__ __device__ __forceinline__ uint64_t desc_key(uint64_t seed, uint64_t edge, uint64_t k) {
    uint64_t z = seed + 0x9E3779B97F4A7C15ull * (edge + 1ull);
    z ^= 0xD1B54A32D192ED03ull * (k + 1ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// number of neighbours of `row` that are < v, and whether v is a neighbour
__device__ __forceinline__ int desc_rank(const uint32_t* __restrict__ bm,
                                         const int* __restrict__ bmprefix, int nwords, int row,
                                         int v) {
    const size_t o = (size_t)row * nwords + (v >> 5);
    return bmprefix[o] + __popc(bm[o] & ((1u << (v & 31)) - 1u));
}

template <int G>
__device__ __forceinline__ double group_sum(double v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
template <int G>
__device__ __forceinline__ int group_sum_int(int v) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#endif
