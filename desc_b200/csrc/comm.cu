// Multi-GPU plumbing: one process per GPU, NCCL over NVLink/NVSwitch (SURVEY 8e).
//
// The reference has no communication layer at all (single MATLAB process); what is exchanged
// here follows from sharding DESC.m's per-edge loops over contiguous edge ranges:
//   * per PGD iteration: all-reduce (sum) of the 2m partner-sum accumulators + 2 scalars
//     (DESC.m:189-190 in scatter form, DESC.m:232-233) and all-gather of the S_vec shards
//     (DESC.m:193 gathers S at arbitrary edges);
//   * per GCW power step: all-gather of the per-node 3x3 blocks (9n doubles);
//   * once in the build: all-gather of co-degrees and apex lists.
//
// NCCL is bound at run time with dlopen, so the single-GPU library (and the MEX file that wraps
// it) has no link-time dependency on NCCL; inside a torch process the already-loaded
// torch-bundled libnccl.so.2 is reused.
#include "internal.cuh"

#include <dlfcn.h>
#include <nccl.h>

#include <algorithm>
#include <map>
#include <mutex>

namespace {
struct NcclApi {
    void* lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void*, void*, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
NcclApi g_nccl;

int nccl_load() {
    if (g_nccl.ok) return DESC_B200_OK;
    const char* names[] = {"libnccl.so.2", "libnccl.so"};
    for (const char* nm : names) {
        g_nccl.lib = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (g_nccl.lib) break;
    }
    if (!g_nccl.lib) {
        desc_set_error("multi-GPU requested but libnccl.so.2 cannot be loaded: %s", dlerror());
        return DESC_B200_ERR_NCCL;
    }
#define LOAD(field, sym)                                                              \
    *(void**)(&g_nccl.field) = dlsym(g_nccl.lib, sym);                                \
    if (!g_nccl.field) {                                                              \
        desc_set_error("libnccl is missing symbol %s", sym);                          \
        return DESC_B200_ERR_NCCL;                                                    \
    }
    LOAD(GetUniqueId, "ncclGetUniqueId");
    LOAD(CommInitRank, "ncclCommInitRank");
    LOAD(CommDestroy, "ncclCommDestroy");
    LOAD(AllReduce, "ncclAllReduce");
    LOAD(Broadcast, "ncclBroadcast");
    LOAD(AllGather, "ncclAllGather");
    LOAD(Send, "ncclSend");
    LOAD(Recv, "ncclRecv");
    LOAD(GroupStart, "ncclGroupStart");
    LOAD(GroupEnd, "ncclGroupEnd");
    LOAD(GetErrorString, "ncclGetErrorString");
#undef LOAD
    g_nccl.ok = true;
    return DESC_B200_OK;
}
}  // namespace

#define NCCL_TRY(expr)                                                                        \
    do {                                                                                      \
        ncclResult_t _r = (expr);                                                             \
        if (_r != ncclSuccess) {                                                              \
            desc_set_error("NCCL error at %s:%d: %s", __FILE__, __LINE__, g_nccl.GetErrorString(_r)); \
            return DESC_B200_ERR_NCCL;                                                        \
        }                                                                                     \
    } while (0)

extern "C" int desc_b200_nccl_unique_id(void* out128) {
    if (!out128) {
        desc_set_error("null output");
        return DESC_B200_ERR_ARG;
    }
    DESC_TRY(nccl_load());
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    NCCL_TRY(g_nccl.GetUniqueId(&id));
    memcpy(out128, &id, sizeof(id));
    return DESC_B200_OK;
}

// Communicators are cached per (unique id, rank, world, device): a ncclUniqueId can initialise one
// communicator only, while a caller typically solves many graphs (many handles) with the id it
// broadcast once.  Handles borrow the cached communicator; desc_b200_comm_finalize() frees them.
namespace {
std::map<std::string, ncclComm_t> g_comms;
std::mutex g_comms_mu;
}  // namespace

int desc_comm_init(desc_b200_handle* h, const void* nccl_id) {
    if (h->world <= 1) return DESC_B200_OK;
    if (!nccl_id) {
        desc_set_error("world=%d but no nccl_id in opts", h->world);
        return DESC_B200_ERR_ARG;
    }
    DESC_TRY(nccl_load());
    std::string key((const char*)nccl_id, 128);
    key += "/" + std::to_string(h->rank) + "/" + std::to_string(h->world) + "/" + std::to_string(h->device);
    std::lock_guard<std::mutex> lock(g_comms_mu);
    auto it = g_comms.find(key);
    if (it != g_comms.end()) {
        h->comm = it->second;
        return DESC_B200_OK;
    }
    ncclUniqueId id;
    memcpy(&id, nccl_id, sizeof(id));
    ncclComm_t comm;
    NCCL_TRY(g_nccl.CommInitRank(&comm, h->world, id, h->rank));
    g_comms[key] = comm;
    h->comm = comm;
    return DESC_B200_OK;
}

void desc_sym_release(desc_b200_handle* h);
void desc_comm_destroy(desc_b200_handle* h) {
    desc_sym_release(h);
    h->comm = nullptr;
}

void desc_sym_finalize();
extern "C" int desc_b200_comm_finalize(void) {
    desc_sym_finalize();
    std::lock_guard<std::mutex> lock(g_comms_mu);
    if (g_nccl.ok)
        for (auto& kv : g_comms) g_nccl.CommDestroy(kv.second);
    g_comms.clear();
    return DESC_B200_OK;
}

int desc_allreduce_sum(desc_b200_handle* h, double* buf, int64_t count) {
    if (h->world <= 1 || count <= 0) return DESC_B200_OK;
    NCCL_TRY(g_nccl.AllReduce(buf, buf, (size_t)count, ncclFloat64, ncclSum, (ncclComm_t)h->comm, h->stream));
    h->collectives++;
    return DESC_B200_OK;
}

// receive buffer of desc_reduce_to_owners, grown to `need` bytes
static int comm_scratch_need(desc_b200_handle* h, size_t need) {
    if (h->comm_scratch_bytes < need) {
        if (h->comm_scratch) cudaFree(h->comm_scratch);
        h->comm_scratch = nullptr;
        h->comm_scratch_bytes = 0;
        CUDA_TRY(cudaMalloc(&h->comm_scratch, need));
        h->comm_scratch_bytes = need;
    }
    return DESC_B200_OK;
}

// in-place ragged all-gather: rank r owns elements [bounds[r], bounds[r+1]) of buf.  Point-to-point
// sends/receives in one group (all pairs move concurrently over NVSwitch) instead of `world`
// broadcasts, which NCCL runs one after the other.
int desc_allgather_ranges(desc_b200_handle* h, void* buf, size_t elem_bytes,
                          const std::vector<int64_t>& bounds) {
    if (h->world <= 1) return DESC_B200_OK;
    const int me = h->rank;
    char* mine = (char*)buf + (size_t)bounds[me] * elem_bytes;
    const size_t my_bytes = (size_t)(bounds[me + 1] - bounds[me]) * elem_bytes;
    NCCL_TRY(g_nccl.GroupStart());
    for (int d = 1; d < h->world; d++) {
        const int to = (me + d) % h->world, from = (me - d + h->world) % h->world;
        const size_t from_bytes = (size_t)(bounds[from + 1] - bounds[from]) * elem_bytes;
        if (my_bytes > 0) NCCL_TRY(g_nccl.Send(mine, my_bytes, ncclInt8, to, (ncclComm_t)h->comm, h->stream));
        if (from_bytes > 0)
            NCCL_TRY(g_nccl.Recv((char*)buf + (size_t)bounds[from] * elem_bytes, from_bytes, ncclInt8, from,
                                 (ncclComm_t)h->comm, h->stream));
    }
    NCCL_TRY(g_nccl.GroupEnd());
    h->collectives++;
    return DESC_B200_OK;
}

// sum over ranks of buf[bounds[r]*width .. bounds[r+1]*width) delivered to rank r only (a ragged
// reduce-scatter), plus an all-reduce of the `tail` doubles at buf[total*width ..].  Every rank
// sends its partial of range r to rank r and adds the received partials IN RANK ORDER: half the
// bytes of an all-reduce, and a summation order that does not depend on NCCL's algorithm choice.
__global__ void k_sum_partials(double* __restrict__ own, const double* __restrict__ scratch, int64_t count,
                               int64_t stride, int world, int me) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    double acc = 0.0;
    int slot = 0;
    for (int r = 0; r < world; r++) {
        if (r == me)
            acc += own[i];
        else
            acc += scratch[(int64_t)(slot++) * stride + i];
    }
    own[i] = acc;
}

int desc_reduce_to_owners(desc_b200_handle* h, double* buf, int width, const std::vector<int64_t>& bounds,
                          int tail) {
    if (h->world <= 1) return DESC_B200_OK;
    const int me = h->rank, W = h->world;
    const int64_t total = bounds[W];
    int64_t maxr = 0;
    for (int r = 0; r < W; r++) maxr = std::max<int64_t>(maxr, bounds[r + 1] - bounds[r]);
    const int64_t stride = maxr * width + tail;            // doubles per received partial
    DESC_TRY(comm_scratch_need(h, (size_t)(W - 1) * stride * sizeof(double)));
    double* scratch = (double*)h->comm_scratch;
    const int64_t my_cnt = (bounds[me + 1] - bounds[me]) * width;
    NCCL_TRY(g_nccl.GroupStart());
    int slot_of[64];
    {
        int sl = 0;
        for (int r = 0; r < W; r++) slot_of[r] = (r == me) ? -1 : sl++;
    }
    for (int d = 1; d < W; d++) {
        const int to = (me + d) % W, from = (me - d + W) % W;
        const int64_t to_cnt = (bounds[to + 1] - bounds[to]) * width;
        if (to_cnt > 0)
            NCCL_TRY(g_nccl.Send(buf + bounds[to] * width, (size_t)to_cnt, ncclFloat64, to, (ncclComm_t)h->comm, h->stream));
        if (my_cnt > 0)
            NCCL_TRY(g_nccl.Recv(scratch + (int64_t)slot_of[from] * stride, (size_t)my_cnt, ncclFloat64, from,
                                 (ncclComm_t)h->comm, h->stream));
        if (tail > 0) {
            NCCL_TRY(g_nccl.Send(buf + total * width, (size_t)tail, ncclFloat64, to, (ncclComm_t)h->comm, h->stream));
            NCCL_TRY(g_nccl.Recv(scratch + (int64_t)slot_of[from] * stride + maxr * width, (size_t)tail, ncclFloat64, from,
                                 (ncclComm_t)h->comm, h->stream));
        }
    }
    NCCL_TRY(g_nccl.GroupEnd());
    if (my_cnt > 0) {
        k_sum_partials<<<(unsigned)((my_cnt + 255) / 256), 256, 0, h->stream>>>(buf + bounds[me] * width, scratch, my_cnt,
                                                                              stride, W, me);
        KERNEL_CHECK(h);
    }
    if (tail > 0) {
        k_sum_partials<<<1, 32, 0, h->stream>>>(buf + total * width, scratch + maxr * width, tail, stride, W, me);
        KERNEL_CHECK(h);
    }
    h->collectives++;
    return DESC_B200_OK;
}


// ------------------------------------------------------------------------------------------
// Peer-memory exchanges (DESC_B200_COMM=peer, the default when CUDA IPC peer mapping works)
// ------------------------------------------------------------------------------------------
// One region per (communicator, rank), allocated once and kept across handles like the communicator itself:
//     [ flags: 2 x 64 u64 ][ S0: cap_m doubles ][ S1: cap_m doubles ][ scratch: (W-1) x cap_stride doubles ]
// Every rank opens every peer's region with cudaIpcOpenMemHandle.  Exchanges:
//   * all-gather of S: each rank STORES its own slice of S into the same offset of every peer's S buffer (16-byte
//     coalesced stores over NVLink, all peers from one kernel), then a flag barrier;
//   * reduce-to-owners of the partner-sum partials: each rank stores its partial of range q (+ the 2 tail doubles)
//     into slot(me) of rank q's scratch, flag barrier, and the owner adds the W partials in rank order (same
//     arithmetic as the NCCL version: deterministic).
// The barrier is a one-CTA kernel: thread q writes this barrier's epoch into rank q's flag[me] (system-scope release)
// and spins (with a timeout) until flag[q] of its own region reaches the epoch.  Ranks are separate processes on
// separate GPUs, so the spinning kernels always run concurrently.
namespace {
struct SymRegion {
    unsigned char* local = nullptr;
    size_t bytes = 0;
    int64_t cap_m = 0, cap_stride = 0;
    int world = 0, me = 0;
    std::vector<unsigned char*> peer;   // peer[me] == local
    uint64_t epoch = 0;
    int users = 0;          // handles whose S buffers point into the region
    bool failed = false;
};
std::map<std::string, SymRegion*> g_sym;
std::mutex g_sym_mu;
constexpr size_t SYM_FLAG_BYTES = 2 * 64 * sizeof(uint64_t);

struct PeerPtrs {
    unsigned char* p[64];
};
struct RangeTab {
    int64_t b[65];
    int world;
};

__global__ void k_sym_barrier(PeerPtrs pp, int me, int W, unsigned long long epoch, int* __restrict__ err) {
    const int q = threadIdx.x;
    if (q >= W || q == me) return;
    volatile unsigned long long* theirs = reinterpret_cast<volatile unsigned long long*>(pp.p[q]) + me;
    volatile unsigned long long* mine = reinterpret_cast<volatile unsigned long long*>(pp.p[me]) + q;
    __threadfence_system();
    *theirs = epoch;
    __threadfence_system();
    const long long t0 = clock64();
    while (*mine < epoch) {
        if (clock64() - t0 > 20000000000ll) {   // ~10 s: a peer died; fail instead of hanging the GPU
            atomicOr(err, 16);
            break;
        }
    }
    __threadfence_system();
}

// my slice [off, off+count) of a buffer at byte offset `base` of the region -> the same place in every peer's region
__global__ void k_sym_push_same(PeerPtrs pp, int me, int W, size_t base, int64_t off, int64_t count) {
    const int q0 = blockIdx.y;
    const int q = q0 < me ? q0 : q0 + 1;          // W-1 peers
    const double* src = reinterpret_cast<const double*>(pp.p[me] + base) + off;
    double* dst = reinterpret_cast<double*>(pp.p[q] + base) + off;
    const int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    // 16-byte stores where the alignment allows (off may be odd)
    const int64_t head = (off & 1) ? 1 : 0;
    if (i0 == 0 && head && count > 0) dst[0] = src[0];
    const int64_t pairs = (count - head) / 2;
    const double2* s2 = reinterpret_cast<const double2*>(src + head);
    double2* d2 = reinterpret_cast<double2*>(dst + head);
    for (int64_t i = i0; i < pairs; i += stride) d2[i] = s2[i];
    if (i0 == 0 && head + 2 * pairs < count) dst[count - 1] = src[count - 1];
    __threadfence_system();
}

// partial of range q (width 2) + the 2 tail doubles -> slot(me) of rank q's scratch
__global__ void k_sym_push_partials(PeerPtrs pp, int me, int W, size_t scratch_base, int64_t cap_stride,
                                    const double* __restrict__ buf, RangeTab t) {
    const int q0 = blockIdx.y;
    const int q = q0 < me ? q0 : q0 + 1;
    const int slot = me < q ? me : me - 1;
    const int64_t n = (t.b[q + 1] - t.b[q]) * 2;
    const double* src = buf + t.b[q] * 2;         // even offset: 16-byte aligned
    double* dst = reinterpret_cast<double*>(pp.p[q] + scratch_base) + (int64_t)slot * cap_stride;
    const int64_t i0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x, stride = (int64_t)gridDim.x * blockDim.x;
    const double2* s2 = reinterpret_cast<const double2*>(src);
    double2* d2 = reinterpret_cast<double2*>(dst);
    for (int64_t i = i0; i < n / 2; i += stride) d2[i] = s2[i];
    if (i0 == 0) {
        const double* tail = buf + t.b[t.world] * 2;
        dst[cap_stride - 2] = tail[0];
        dst[cap_stride - 1] = tail[1];
    }
    __threadfence_system();
}
// own range += the W-1 received partials, in rank order; tail likewise
__global__ void k_sym_sum(double* __restrict__ own, double* __restrict__ tail, const double* __restrict__ scratch,
                          int64_t count, int64_t cap_stride, int W, int me) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= count + 2) return;
    const bool is_tail = i >= count;
    const int64_t si = is_tail ? cap_stride - 2 + (i - count) : i;
    double* o = is_tail ? tail + (i - count) : own + i;
    double acc = 0.0;
    for (int r = 0; r < W; r++) {
        if (r == me)
            acc += *o;
        else
            acc += scratch[(int64_t)(r < me ? r : r - 1) * cap_stride + si];
    }
    *o = acc;
}

int sym_barrier(desc_b200_handle* h, SymRegion* R) {
    PeerPtrs pp;
    for (int q = 0; q < R->world; q++) pp.p[q] = R->peer[q];
    R->epoch++;
    k_sym_barrier<<<1, 64, 0, h->stream>>>(pp, R->me, R->world, (unsigned long long)R->epoch, h->d_err);
    KERNEL_CHECK(h);
    return DESC_B200_OK;
}
}  // namespace

int desc_sym_setup(desc_b200_handle* h, int64_t m, const std::vector<int64_t>& bounds) {
    if (h->sym) return DESC_B200_OK;   // this handle already uses the region (its sizes do not change)
    if (h->world <= 1 || h->world > 64) return DESC_B200_OK;
    {   // DESC_B200_COMM = peer (default) | p2p: any value but peer exchanges through NCCL point-to-point
        const char* e = getenv("DESC_B200_COMM");
        if (e && strcmp(e, "peer") != 0) return DESC_B200_OK;
    }
    const int W = h->world, me = h->rank;
    int64_t maxr = 0;
    for (int r = 0; r < W; r++) maxr = std::max<int64_t>(maxr, bounds[r + 1] - bounds[r]);
    const int64_t need_m = (m + 4 + 1) & ~(int64_t)1, need_stride = maxr * 2 + 2;
    char keyb[64];
    snprintf(keyb, sizeof(keyb), "%p/%d", h->comm, h->device);
    std::lock_guard<std::mutex> lock(g_sym_mu);
    SymRegion*& R = g_sym[keyb];
    if (!R) R = new SymRegion();
    if (R->failed) return DESC_B200_OK;
    if (h->sym == nullptr && R->local && (R->cap_m < need_m || R->cap_stride < need_stride) && R->users > 0)
        return DESC_B200_OK;   // another live handle points into the region: this handle exchanges through NCCL
    if (!R->local || R->cap_m < need_m || R->cap_stride < need_stride) {
        // (re)allocate: collective -- every rank takes the same decision because the sizes follow from the graph
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        for (int q = 0; q < (int)R->peer.size(); q++)
            if (q != R->me && R->peer[q]) cudaIpcCloseMemHandle(R->peer[q]);
        if (R->local) desc_raw_free(R->local);
        R->peer.assign(W, nullptr);
        R->local = nullptr;
        R->world = W;
        R->me = me;
        // headroom: later graphs of similar size reuse it.  Multiples of 16 doubles: the PGD kernels bulk-copy (TMA)
        // from S, which needs 16-byte aligned bases
        R->cap_m = (std::max<int64_t>(need_m, R->cap_m) + need_m / 8 + 15) & ~(int64_t)15;
        R->cap_stride = ((std::max<int64_t>(need_stride, R->cap_stride) + need_stride / 8) + 15) & ~(int64_t)15;
        R->bytes = SYM_FLAG_BYTES + (size_t)(2 * R->cap_m + (int64_t)(W - 1) * R->cap_stride) * sizeof(double);
        R->epoch = 0;
        void* p = nullptr;
        if (desc_raw_malloc(&p, R->bytes) != cudaSuccess) {
            cudaGetLastError();
            R->failed = true;
            return DESC_B200_OK;
        }
        R->local = (unsigned char*)p;
        CUDA_TRY(cudaMemsetAsync(R->local, 0, SYM_FLAG_BYTES, h->stream));
        cudaIpcMemHandle_t mine;
        bool ok = cudaIpcGetMemHandle(&mine, R->local) == cudaSuccess;
        if (!ok) cudaGetLastError();
        // all-gather the handles (+ an ok byte) through NCCL
        const size_t rec = sizeof(cudaIpcMemHandle_t) + 8;
        unsigned char* d_all = nullptr;
        CUDA_TRY(cudaMalloc(&d_all, rec * W));
        std::vector<unsigned char> hall(rec * W, 0);
        memcpy(hall.data() + rec * me, &mine, sizeof(mine));
        hall[rec * me + sizeof(mine)] = ok ? 1 : 0;
        CUDA_TRY(cudaMemcpyAsync(d_all + rec * me, hall.data() + rec * me, rec, cudaMemcpyHostToDevice, h->stream));
        NCCL_TRY(g_nccl.AllGather(d_all + rec * me, d_all, rec, ncclInt8, (ncclComm_t)h->comm, h->stream));
        CUDA_TRY(cudaMemcpyAsync(hall.data(), d_all, rec * W, cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        CUDA_TRY(cudaFree(d_all));
        for (int q = 0; q < W; q++) ok = ok && hall[rec * q + sizeof(mine)] == 1;
        R->peer[me] = R->local;
        for (int q = 0; q < W && ok; q++) {
            if (q == me) continue;
            cudaIpcMemHandle_t hq;
            memcpy(&hq, hall.data() + rec * q, sizeof(hq));
            void* pq = nullptr;
            if (cudaIpcOpenMemHandle(&pq, hq, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
                cudaGetLastError();
                ok = false;
            }
            R->peer[q] = (unsigned char*)pq;
        }
        // every rank must agree on success (a rank that failed to map would wait forever in a barrier)
        double* d_ok = nullptr;
        CUDA_TRY(cudaMalloc(&d_ok, sizeof(double)));
        const double okv = ok ? 0.0 : 1.0;
        CUDA_TRY(cudaMemcpyAsync(d_ok, &okv, sizeof(double), cudaMemcpyHostToDevice, h->stream));
        NCCL_TRY(g_nccl.AllReduce(d_ok, d_ok, 1, ncclFloat64, ncclSum, (ncclComm_t)h->comm, h->stream));
        double bad = 0.0;
        CUDA_TRY(cudaMemcpyAsync(&bad, d_ok, sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        CUDA_TRY(cudaFree(d_ok));
        if (bad != 0.0) {
            for (int q = 0; q < W; q++)
                if (q != me && R->peer[q]) cudaIpcCloseMemHandle(R->peer[q]);
            desc_raw_free(R->local);
            R->local = nullptr;
            R->peer.clear();
            R->failed = true;
            return DESC_B200_OK;
        }
    }
    h->sym = R;
    R->users++;
    return DESC_B200_OK;
}

// flag barrier over all ranks of the handle's communicator (no-op without a peer-mapped region)
int desc_sym_barrier(desc_b200_handle* h) {
    if (!h->sym) return DESC_B200_OK;
    return sym_barrier(h, (SymRegion*)h->sym);
}

static double* sym_S(SymRegion* R, int which) {
    return reinterpret_cast<double*>(R->local + SYM_FLAG_BYTES) + (int64_t)which * R->cap_m;
}
// the S buffers of a multi-GPU handle live in the region (pgd.cu asks for them here)
double* desc_sym_S_buffer(desc_b200_handle* h, int which) {
    return h->sym ? sym_S((SymRegion*)h->sym, which) : nullptr;
}

int desc_sym_allgather_S(desc_b200_handle* h, int which, const std::vector<int64_t>& bounds) {
    SymRegion* R = (SymRegion*)h->sym;
    const int W = R->world, me = R->me;
    PeerPtrs pp;
    for (int q = 0; q < W; q++) pp.p[q] = R->peer[q];
    const int64_t cnt = bounds[me + 1] - bounds[me];
    if (cnt > 0) {
        dim3 g(std::max(1, (2 * DESC_SMS) / (W - 1)), W - 1);
        k_sym_push_same<<<g, 256, 0, h->stream>>>(pp, me, W, SYM_FLAG_BYTES + (size_t)which * R->cap_m * sizeof(double),
                                                 bounds[me], cnt);
        KERNEL_CHECK(h);
    }
    DESC_TRY(sym_barrier(h, R));
    h->collectives++;
    return DESC_B200_OK;
}

int desc_sym_reduce_to_owners(desc_b200_handle* h, double* buf, const std::vector<int64_t>& bounds) {
    SymRegion* R = (SymRegion*)h->sym;
    const int W = R->world, me = R->me;
    {   // a re-built incidence may have moved the shard boundaries: larger ranges than the scratch go through NCCL
        int64_t maxr = 0;
        for (int r = 0; r < W; r++) maxr = std::max<int64_t>(maxr, bounds[r + 1] - bounds[r]);
        if (maxr * 2 + 2 > R->cap_stride) return desc_reduce_to_owners(h, buf, 2, bounds, 2);
    }
    PeerPtrs pp;
    for (int q = 0; q < W; q++) pp.p[q] = R->peer[q];
    RangeTab t;
    t.world = W;
    for (int r = 0; r <= W; r++) t.b[r] = bounds[r];
    const size_t scratch_base = SYM_FLAG_BYTES + (size_t)2 * R->cap_m * sizeof(double);
    dim3 g(std::max(1, (2 * DESC_SMS) / (W - 1)), W - 1);
    k_sym_push_partials<<<g, 256, 0, h->stream>>>(pp, me, W, scratch_base, R->cap_stride, buf, t);
    KERNEL_CHECK(h);
    DESC_TRY(sym_barrier(h, R));
    const int64_t n = (bounds[me + 1] - bounds[me]) * 2;
    k_sym_sum<<<(unsigned)((n + 2 + 255) / 256), 256, 0, h->stream>>>(buf + bounds[me] * 2, buf + bounds[W] * 2,
                                                                     reinterpret_cast<const double*>(R->local + scratch_base), n,
                                                                     R->cap_stride, W, me);
    KERNEL_CHECK(h);
    h->collectives++;
    return DESC_B200_OK;
}

void desc_sym_release(desc_b200_handle* h) {
    if (!h->sym) return;
    std::lock_guard<std::mutex> lock(g_sym_mu);
    ((SymRegion*)h->sym)->users--;
    h->sym = nullptr;
}

void desc_sym_finalize() {
    std::lock_guard<std::mutex> lock(g_sym_mu);
    for (auto& kv : g_sym) {
        SymRegion* R = kv.second;
        for (int q = 0; q < (int)R->peer.size(); q++)
            if (q != R->me && R->peer[q]) cudaIpcCloseMemHandle(R->peer[q]);
        if (R->local) desc_raw_free(R->local);
        delete R;
    }
    g_sym.clear();
}
