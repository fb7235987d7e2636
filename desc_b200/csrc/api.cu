// C ABI of libdesc_b200.so (include/desc_b200.h): argument checking, stage ordering, host<->device
// copies and stage timing.  The kernels live in build.cu / cycle.cu / pgd.cu / gcw.cu.
#include "internal.cuh"

#include <stdarg.h>

#include <algorithm>
#include <cmath>

static thread_local char g_err[1024] = "";

void desc_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

namespace {
struct StageTimer {
    desc_b200_handle* h;
    double* slot;
    bool started = false;
    StageTimer(desc_b200_handle* h_, double* slot_) : h(h_), slot(slot_) {
        started = cudaEventRecord(h->ev0, h->stream) == cudaSuccess;
    }
    int stop() {
        if (!started) return DESC_B200_OK;
        started = false;
        CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
        CUDA_TRY(cudaEventSynchronize(h->ev1));
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, h->ev0, h->ev1));
        *slot = ms;
        return DESC_B200_OK;
    }
};

int check_handle(desc_b200_handle* h) {
    if (!h) {
        desc_set_error("null handle");
        return DESC_B200_ERR_ARG;
    }
    CUDA_TRY(cudaSetDevice(h->device));
    return DESC_B200_OK;
}
}  // namespace

extern "C" {

const char* desc_b200_last_error(void) { return g_err; }
int desc_b200_version(void) { return DESC_B200_VERSION; }

int desc_b200_device_count(void) {
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (e != cudaSuccess) {
        cudaGetLastError();
        desc_set_error("no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e));
        return DESC_B200_ERR_CUDA;
    }
    return c;
}

void desc_b200_destroy(desc_b200_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    desc_comm_destroy(h);
    if (h->S_in_sym) h->S[0] = h->S[1] = nullptr;   // they live in the communicator's peer-mapped region
    void* ptrs[] = {h->ei, h->ej, h->Rij_owned, h->bm, h->bmprefix, h->rowstart, h->adj_nbr, h->adj_eid,
                    h->codeg, h->rowptr, h->apex, h->pk_jk, h->pk_ki, h->S0, h->w[0], h->w[1],
                    h->S[0], h->S[1], h->acc[0], h->acc[1], h->adam_m, h->adam_v, h->d_hist, h->d_ctrl,
                    h->d_ctrl_f, h->omega, h->isd, h->X[0], h->X[1], h->gcw_coef, h->gcw_red,
                    h->gcw_small, h->gcw_res, h->R_est, h->d_err, h->d_Sin, h->rk_i, h->rk_j, h->estart,
                    h->pgd_partial, h->jhdr, h->sjk, h->thr_key, h->thr_k, h->comm_scratch,
                    h->cemp_S[0], h->cemp_S[1], h->diag_work, h->diag_hist, h->R_mst, h->gcw_coef_adj, h->P1,
                    h->S_adj[0], h->S_adj[1], h->adj_mirror};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (h->h_ctrl) cudaFreeHost(h->h_ctrl);
    if (h->gcw_res_host) cudaFreeHost(h->gcw_res_host);
    for (cudaEvent_t e : h->iter_events) cudaEventDestroy(e);
    for (cudaEvent_t e : h->spmv_events) cudaEventDestroy(e);
    cudaEvent_t evs[] = {h->ev0, h->ev1, h->ev2, h->ev3};
    for (cudaEvent_t e : evs)
        if (e) cudaEventDestroy(e);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int desc_b200_create(desc_b200_handle** out, int32_t n, int64_t m, const double* Ind,
                     const double* RijMat, const desc_b200_opts* opts) {
    if (!out) {
        desc_set_error("null output handle");
        return DESC_B200_ERR_ARG;
    }
    *out = nullptr;
    if (!Ind || !RijMat || m <= 0 || n < 0) {
        desc_set_error("bad arguments: Ind/RijMat null, or m <= 0 (m=%lld, n=%d)", (long long)m, n);
        return DESC_B200_ERR_ARG;
    }
    if (m > DESC_MAX_EDGES) {
        desc_set_error("m=%lld exceeds the 30-bit edge-id limit", (long long)m);
        return DESC_B200_ERR_LIMIT;
    }
    int ndev = desc_b200_device_count();
    if (ndev <= 0) {
        if (ndev == 0) desc_set_error("no CUDA device (this library has no CPU fallback)");
        return DESC_B200_ERR_CUDA;
    }
    desc_b200_opts o = {};
    o.device = -1;
    o.world = 1;
    if (opts) o = *opts;
    if (o.world < 1) o.world = 1;
    if (o.rank < 0 || o.rank >= o.world) {
        desc_set_error("rank %d outside world %d", o.rank, o.world);
        return DESC_B200_ERR_ARG;
    }
    int dev = o.device;
    if (dev < 0) CUDA_TRY(cudaGetDevice(&dev));
    if (dev >= ndev) {
        desc_set_error("device %d requested but only %d visible", dev, ndev);
        return DESC_B200_ERR_ARG;
    }
    CUDA_TRY(cudaSetDevice(dev));
    desc_b200_handle* h = new desc_b200_handle();
    h->device = dev;
    h->rank = o.rank;
    h->world = o.world;
    h->n = n;
    h->m = m;
    int rc = DESC_B200_OK;
    auto fail = [&](int code) {
        desc_b200_destroy(h);
        return code;
    };
    if (o.stream) {
        h->stream = (cudaStream_t)o.stream;
    } else {
        if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess) {
            desc_set_error("cudaStreamCreate failed: %s", cudaGetErrorString(cudaGetLastError()));
            return fail(DESC_B200_ERR_CUDA);
        }
        h->own_stream = true;
    }
    cudaEvent_t* evs[] = {&h->ev0, &h->ev1, &h->ev2, &h->ev3};
    for (cudaEvent_t* e : evs)
        if (cudaEventCreate(e) != cudaSuccess) {
            desc_set_error("cudaEventCreate failed");
            return fail(DESC_B200_ERR_CUDA);
        }
    auto body = [&]() -> int {
        const double* d_Ind = Ind;
        DescTmp t_ind;   // device copy of Ind: only needed until the graph is set up (freed on error returns too)
        double* d_Ind_owned = nullptr;
        if (o.flags & DESC_B200_INPUTS_ON_DEVICE) {
            h->Rij = RijMat;
        } else {
            StageTimer t(h, &h->tm.h2d_ms);
            CUDA_TRY(t_ind.alloc(2 * m * sizeof(double)));
            d_Ind_owned = t_ind.as<double>();
            CUDA_TRY(cudaMalloc(&h->Rij_owned, 9 * m * sizeof(double)));
            if (h->world > 1) {
                // every rank was given the same host arrays (the contract of a sharded solve): each uploads 1/world of
                // them over PCIe and the slices are all-gathered over NVLink -- with 8 ranks on one host the full
                // upload per rank (440 MB at cfg 4, 8 x in parallel through one host) cost ~20 ms per solve
                DESC_TRY(desc_comm_init(h, o.nccl_id));
                std::vector<int64_t> b(h->world + 1);
                for (int r = 0; r <= h->world; r++) b[r] = (m * r) / h->world;
                const int64_t b0 = b[h->rank], cnt = b[h->rank + 1] - b[h->rank];
                if (cnt > 0) {
                    CUDA_TRY(cudaMemcpyAsync(d_Ind_owned + b0, Ind + b0, cnt * sizeof(double), cudaMemcpyHostToDevice, h->stream));
                    CUDA_TRY(cudaMemcpyAsync(d_Ind_owned + m + b0, Ind + m + b0, cnt * sizeof(double), cudaMemcpyHostToDevice, h->stream));
                    CUDA_TRY(cudaMemcpyAsync(h->Rij_owned + 9 * b0, RijMat + 9 * b0, 9 * cnt * sizeof(double), cudaMemcpyHostToDevice, h->stream));
                }
                DESC_TRY(desc_allgather_ranges(h, d_Ind_owned, sizeof(double), b));
                DESC_TRY(desc_allgather_ranges(h, d_Ind_owned + m, sizeof(double), b));
                DESC_TRY(desc_allgather_ranges(h, h->Rij_owned, 9 * sizeof(double), b));
            } else {
                CUDA_TRY(cudaMemcpyAsync(d_Ind_owned, Ind, 2 * m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
                CUDA_TRY(cudaMemcpyAsync(h->Rij_owned, RijMat, 9 * m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
            }
            DESC_TRY(t.stop());
            d_Ind = d_Ind_owned;
            h->Rij = h->Rij_owned;
        }
        int r;
        {
            StageTimer t(h, &h->tm.graph_ms);
            r = desc_graph_setup(h, d_Ind);
            if (r == DESC_B200_OK) r = t.stop();
        }
        t_ind.release();
        DESC_TRY(r);
        if (!h->comm) DESC_TRY(desc_comm_init(h, o.nccl_id));
        return DESC_B200_OK;
    };
    rc = body();
    if (rc != DESC_B200_OK) return fail(rc);
    h->tm.total_launches = h->launches;
    *out = h;
    return DESC_B200_OK;
}

int desc_b200_build_incidence(desc_b200_handle* h, int32_t n_sample, uint64_t seed,
                              const int64_t* cyc_ptr, const int32_t* cyc_apex) {
    DESC_TRY(check_handle(h));
    StageTimer t(h, &h->tm.build_ms);
    DESC_TRY(desc_build_incidence_impl(h, n_sample, seed, cyc_ptr, cyc_apex));
    DESC_TRY(t.stop());
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

int desc_b200_cycle_inconsistency(desc_b200_handle* h) {
    DESC_TRY(check_handle(h));
    StageTimer t(h, &h->tm.cycle_ms);
    DESC_TRY(desc_cycle_impl(h));
    DESC_TRY(t.stop());
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

int desc_b200_pgd(desc_b200_handle* h, int32_t iters, desc_b200_step_rule* rule, double* S_vec_out,
                  double* hist_out, int32_t* iters_run_out) {
    DESC_TRY(check_handle(h));
    int iters_run = 0;
    {
        StageTimer t(h, &h->tm.pgd_ms);
        DESC_TRY(desc_pgd_impl(h, iters, rule, &iters_run));
        DESC_TRY(t.stop());
    }
    {
        StageTimer t(h, &h->tm.d2h_ms);
        if (S_vec_out)
            CUDA_TRY(cudaMemcpyAsync(S_vec_out, h->S[h->final_buf], h->m * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        if (hist_out && iters > 0) {
            CUDA_TRY(cudaMemcpyAsync(hist_out, h->d_hist, (size_t)2 * iters * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        }
        DESC_TRY(t.stop());
    }
    if (hist_out)
        for (int t = iters_run; t < iters; t++) hist_out[2 * t] = hist_out[2 * t + 1] = 0.0;
    if (iters_run_out) *iters_run_out = iters_run;
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

int desc_b200_gcw(desc_b200_handle* h, const double* S_vec, double* R_out) {
    DESC_TRY(check_handle(h));
    const double* d_S = nullptr;
    if (S_vec) {
        if (!h->d_Sin) CUDA_TRY(cudaMalloc(&h->d_Sin, h->m * sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(h->d_Sin, S_vec, h->m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        d_S = h->d_Sin;
    } else {
        if (!h->have_pgd) {
            desc_set_error("gcw with S_vec=NULL needs a previous pgd on this handle");
            return DESC_B200_ERR_STATE;
        }
        d_S = h->S[h->final_buf];
    }
    {
        StageTimer t(h, &h->tm.gcw_ms);
        DESC_TRY(desc_gcw_impl(h, d_S));
        DESC_TRY(t.stop());
    }
    h->have_gcw = true;
    if (R_out) {
        StageTimer t(h, &h->tm.d2h_ms);
        CUDA_TRY(cudaMemcpyAsync(R_out, h->R_est, 9 * (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        DESC_TRY(t.stop());
    }
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

int desc_b200_refine(desc_b200_handle* h, const double* S_vec, const double* R_init, double* R_out,
                     int32_t* iters_run, double* scores) {
    DESC_TRY(check_handle(h));
    const double* d_S = nullptr;
    if (S_vec) {
        if (!h->d_Sin) CUDA_TRY(cudaMalloc(&h->d_Sin, h->m * sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(h->d_Sin, S_vec, h->m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        d_S = h->d_Sin;
    } else {
        if (!h->have_pgd) {
            desc_set_error("refine with S_vec=NULL needs a previous pgd on this handle");
            return DESC_B200_ERR_STATE;
        }
        d_S = h->S[h->final_buf];
    }
    DescTmp t_R, t_out;   // returned to the pool on every exit path
    double* d_R = nullptr;
    if (R_init) {
        CUDA_TRY(t_R.alloc(9 * (size_t)h->n * sizeof(double)));
        d_R = t_R.as<double>();
        CUDA_TRY(cudaMemcpyAsync(d_R, R_init, 9 * (size_t)h->n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    } else if (!h->have_gcw) {
        desc_set_error("refine with R_init=NULL needs a previous gcw on this handle");
        return DESC_B200_ERR_STATE;
    }
    CUDA_TRY(t_out.alloc(9 * (size_t)h->n * sizeof(double)));
    double* d_out = t_out.as<double>();
    int run = 0, rc;
    {
        StageTimer t(h, &h->tm.laa_ms);
        rc = desc_laa_impl(h, d_S, d_R ? d_R : h->R_est, d_out, 100, 1e-3, &run, scores);
        if (rc == DESC_B200_OK) rc = t.stop();
    }
    if (rc == DESC_B200_OK && R_out) {
        cudaError_t e = cudaMemcpyAsync(R_out, d_out, 9 * (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) {
            desc_set_error("CUDA error %s copying the refined rotations", cudaGetErrorString(e));
            rc = DESC_B200_ERR_CUDA;
        }
    }
    if (iters_run) *iters_run = run;
    h->tm.laa_iters = run;
    h->tm.laa_cg_iters = h->laa_cg_iters;
    h->tm.total_launches = h->launches;
    return rc;
}

int desc_b200_solve(desc_b200_handle* h, int32_t n_sample, uint64_t seed, int32_t iters,
                    desc_b200_step_rule* rule, double* S_vec_out, double* R_out, double* hist_out,
                    int32_t* iters_run_out) {
    DESC_TRY(desc_b200_build_incidence(h, n_sample, seed, nullptr, nullptr));
    DESC_TRY(desc_b200_cycle_inconsistency(h));
    DESC_TRY(desc_b200_pgd(h, iters, rule, S_vec_out, hist_out, iters_run_out));
    if (R_out) {
        const double d2h = h->tm.d2h_ms;
        DESC_TRY(desc_b200_gcw(h, nullptr, R_out));
        h->tm.d2h_ms += d2h;
    }
    return DESC_B200_OK;
}

// ---- SURVEY 8(f) #3: CEMP / CEMP+GCW on the same incidence ---------------------------------
int desc_b200_cemp(desc_b200_handle* h, int32_t max_iter, const double* reweighting, int32_t n_reweighting,
                   double* SVec_out) {
    DESC_TRY(check_handle(h));
    {
        StageTimer t(h, &h->tm.cemp_ms);
        DESC_TRY(desc_cemp_impl(h, max_iter, reweighting, n_reweighting));
        DESC_TRY(t.stop());
    }
    h->tm.cemp_iters = max_iter;
    if (SVec_out) {
        CUDA_TRY(cudaMemcpyAsync(SVec_out, h->cemp_S[h->cemp_final], h->m * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    }
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

int desc_b200_cemp_gcw(desc_b200_handle* h, const double* SVec, double* R_out) {
    DESC_TRY(check_handle(h));
    const double* d_S = nullptr;
    if (SVec) {
        if (!h->d_Sin) CUDA_TRY(cudaMalloc(&h->d_Sin, h->m * sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(h->d_Sin, SVec, h->m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        d_S = h->d_Sin;
    } else {
        if (!h->have_cemp) {
            desc_set_error("cemp_gcw with SVec=NULL needs a previous cemp on this handle");
            return DESC_B200_ERR_STATE;
        }
        d_S = h->cemp_S[h->cemp_final];
    }
    int rc;
    {
        StageTimer t(h, &h->tm.gcw_ms);
        h->gcw_weight_rule = 1;   // CEMP_GCW.m:141
        rc = desc_gcw_impl(h, d_S);
        h->gcw_weight_rule = 0;
        if (rc == DESC_B200_OK) rc = t.stop();
    }
    DESC_TRY(rc);
    h->have_gcw = true;
    if (R_out) {
        CUDA_TRY(cudaMemcpyAsync(R_out, h->R_est, 9 * (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    }
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

// Spectral.m:15-47
int desc_b200_spectral(desc_b200_handle* h, double* R_out) {
    DESC_TRY(check_handle(h));
    int rc;
    {
        StageTimer t(h, &h->tm.gcw_ms);
        h->gcw_weight_rule = 2;
        rc = desc_gcw_impl(h, nullptr);
        h->gcw_weight_rule = 0;
        if (rc == DESC_B200_OK) rc = t.stop();
    }
    DESC_TRY(rc);
    h->have_gcw = true;
    if (R_out) {
        CUDA_TRY(cudaMemcpyAsync(R_out, h->R_est, 9 * (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    }
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

int desc_b200_cycle_reweight(desc_b200_handle* h, const double* x, double beta, double empty_value, double* out) {
    DESC_TRY(check_handle(h));
    if (!h->have_s0) {
        desc_set_error("cycle_reweight before cycle_inconsistency");
        return DESC_B200_ERR_STATE;
    }
    if (!x || !out) {
        desc_set_error("cycle_reweight: null vector");
        return DESC_B200_ERR_ARG;
    }
    double* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, (size_t)2 * h->m * sizeof(double)));
    int rc = DESC_B200_OK;
    cudaError_t e = cudaMemcpyAsync(d, x, h->m * sizeof(double), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) rc = desc_cemp_reweight(h, d, d + h->m, beta, empty_value);
    if (e == cudaSuccess && rc == DESC_B200_OK)
        e = cudaMemcpyAsync(out, d + h->m, h->m * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    if (e != cudaSuccess) {
        desc_set_error("CUDA error %s in cycle_reweight", cudaGetErrorString(e));
        return DESC_B200_ERR_CUDA;
    }
    h->tm.total_launches = h->launches;
    return rc;
}

// MPLS.m:152-195: CEMP+MST initialisation
int desc_b200_mst_init(desc_b200_handle* h, const double* SVec, double* R_out) {
    DESC_TRY(check_handle(h));
    const double* d_S = nullptr;
    if (SVec) {
        if (!h->d_Sin) CUDA_TRY(cudaMalloc(&h->d_Sin, h->m * sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(h->d_Sin, SVec, h->m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        d_S = h->d_Sin;
    } else {
        if (!h->have_cemp) {
            desc_set_error("mst_init with SVec=NULL needs a previous cemp on this handle");
            return DESC_B200_ERR_STATE;
        }
        d_S = h->cemp_S[h->cemp_final];
    }
    if (!h->R_mst) CUDA_TRY(cudaMalloc(&h->R_mst, 9 * (size_t)h->n * sizeof(double)));
    h->have_mst = false;
    {
        StageTimer t(h, &h->tm.mst_ms);
        DESC_TRY(desc_mst_init_impl(h, d_S, h->R_mst));
        DESC_TRY(t.stop());
    }
    h->have_mst = true;
    if (R_out) {
        CUDA_TRY(cudaMemcpyAsync(R_out, h->R_mst, 9 * (size_t)h->n * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
    }
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

// MPLS.m:198-256: the reweighting loop
int desc_b200_mpls_refine(desc_b200_handle* h, const double* SVec, const double* R_init,
                          const desc_b200_mpls_params* p, double* R_out, int32_t* iters_run, double* scores) {
    DESC_TRY(check_handle(h));
    if (!p || p->max_iter < 1 || !p->reweighting || !p->thresholding || !p->cycle_info_ratio || p->n_reweighting < 1 ||
        p->n_thresholding < 1 || p->n_cycle_info_ratio < 1) {
        desc_set_error("mpls_refine: MPLS_parameters need max_iter >= 1 and non-empty reweighting / thresholding / "
                       "cycle_info_ratio");
        return DESC_B200_ERR_ARG;
    }
    if (!h->have_s0) {
        desc_set_error("mpls_refine before cycle_inconsistency");
        return DESC_B200_ERR_STATE;
    }
    const double* d_S = nullptr;
    if (SVec) {
        if (!h->d_Sin) CUDA_TRY(cudaMalloc(&h->d_Sin, h->m * sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(h->d_Sin, SVec, h->m * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        d_S = h->d_Sin;
    } else {
        if (!h->have_cemp) {
            desc_set_error("mpls_refine with SVec=NULL needs a previous cemp on this handle");
            return DESC_B200_ERR_STATE;
        }
        d_S = h->cemp_S[h->cemp_final];
    }
    if (!R_init && !h->have_mst) {
        desc_set_error("mpls_refine with R_init=NULL needs a previous mst_init on this handle");
        return DESC_B200_ERR_STATE;
    }
    // MPLS.m:43-63: short parameter vectors are padded with their last element
    const int len = p->max_iter;
    std::vector<double> beta(len), tau(len), alpha(len);
    for (int t = 0; t < len; t++) {
        beta[t] = p->reweighting[std::min(t, p->n_reweighting - 1)];
        tau[t] = p->thresholding[std::min(t, p->n_thresholding - 1)];
        alpha[t] = p->cycle_info_ratio[std::min(t, p->n_cycle_info_ratio - 1)];
    }
    desc_laa_sched sched = {beta.data(), tau.data(), alpha.data(), len, std::acos(-0.5) / 3.14159265358979323846};
    double *d_R = nullptr, *d_out = nullptr;
    const size_t n9 = 9 * (size_t)h->n;
    CUDA_TRY(cudaMalloc(&d_out, n9 * sizeof(double)));
    if (R_init) {
        CUDA_TRY(cudaMalloc(&d_R, n9 * sizeof(double)));
        CUDA_TRY(cudaMemcpyAsync(d_R, R_init, n9 * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    }
    int run = 0, rc;
    {
        StageTimer t(h, &h->tm.laa_ms);
        rc = desc_laa_impl(h, d_S, d_R ? d_R : h->R_mst, d_out, p->max_iter, p->stop_threshold, &run, scores, &sched);
        if (rc == DESC_B200_OK) rc = t.stop();
    }
    if (rc == DESC_B200_OK && R_out) {
        cudaError_t e = cudaMemcpyAsync(R_out, d_out, n9 * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        if (e != cudaSuccess) {
            desc_set_error("CUDA error %s copying the MPLS rotations", cudaGetErrorString(e));
            rc = DESC_B200_ERR_CUDA;
        }
    }
    cudaFree(d_out);
    if (d_R) cudaFree(d_R);
    if (iters_run) *iters_run = run;
    h->tm.laa_iters = run;
    h->tm.laa_cg_iters = h->laa_cg_iters;
    h->tm.total_launches = h->launches;
    return rc;
}

// ---- SURVEY 8(f) #4: evaluation / diagnostics -----------------------------------------------
int desc_b200_rotation_alignment(desc_b200_handle* h, const double* R_est, const double* R_gt, double* R_out,
                                 double* R_align, double* mean_error, double* median_error) {
    DESC_TRY(check_handle(h));
    if (!R_est || !R_gt) {
        desc_set_error("rotation_alignment: null rotations");
        return DESC_B200_ERR_ARG;
    }
    const size_t n9 = 9 * (size_t)h->n;
    double* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, 3 * n9 * sizeof(double)));
    double a[11];
    int rc = DESC_B200_OK;
    cudaError_t e = cudaMemcpyAsync(d, R_est, n9 * sizeof(double), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + n9, R_gt, n9 * sizeof(double), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) rc = desc_align_impl(h, d, d + n9, d + 2 * n9, a);
    if (e == cudaSuccess && rc == DESC_B200_OK && R_out)
        e = cudaMemcpyAsync(R_out, d + 2 * n9, n9 * sizeof(double), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d);
    if (e != cudaSuccess) {
        desc_set_error("CUDA error %s in rotation_alignment", cudaGetErrorString(e));
        return DESC_B200_ERR_CUDA;
    }
    DESC_TRY(rc);
    if (mean_error) *mean_error = a[0];
    if (median_error) *median_error = a[1];
    if (R_align) memcpy(R_align, a + 2, 9 * sizeof(double));
    h->tm.total_launches = h->launches;
    return DESC_B200_OK;
}

int desc_b200_pgd_diag(desc_b200_handle* h, int32_t iters, desc_b200_step_rule* rule, const double* ErrVec,
                       const double* R_orig, double* S_vec_out, double* hist_out, double* diag_out,
                       int32_t* iters_run_out) {
    DESC_TRY(check_handle(h));
    if (!ErrVec || !R_orig || !diag_out || iters < 0) {
        desc_set_error("pgd_diag needs ErrVec (m), R_orig (3x3xn) and diag_out (3*iters)");
        return DESC_B200_ERR_ARG;
    }
    const size_t n9 = 9 * (size_t)h->n;
    double* d = nullptr;
    CUDA_TRY(cudaMalloc(&d, ((size_t)h->m + n9) * sizeof(double)));
    cudaError_t e = cudaMemcpyAsync(d, ErrVec, h->m * sizeof(double), cudaMemcpyHostToDevice, h->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + h->m, R_orig, n9 * sizeof(double), cudaMemcpyHostToDevice, h->stream);
    if (e != cudaSuccess) {
        cudaFree(d);
        desc_set_error("CUDA error %s in pgd_diag", cudaGetErrorString(e));
        return DESC_B200_ERR_CUDA;
    }
    for (int t = 0; t < 3 * iters; t++) diag_out[t] = 0.0;
    h->diag_on = true;
    h->diag_err = d;
    h->diag_Rgt = d + h->m;
    h->diag_out = diag_out;
    h->diag_cap = iters;
    const int rc = desc_b200_pgd(h, iters, rule, S_vec_out, hist_out, iters_run_out);
    h->diag_on = false;
    h->diag_err = h->diag_Rgt = nullptr;
    h->diag_out = nullptr;
    h->diag_cap = 0;
    cudaFree(d);
    if (rc == DESC_B200_OK && iters_run_out)
        for (int t = 3 * *iters_run_out; t < 3 * iters; t++) diag_out[t] = 0.0;
    return rc;
}

// ---- getters ---------------------------------------------------------------------------
int desc_b200_get_info(desc_b200_handle* h, int64_t info[10]) {
    DESC_TRY(check_handle(h));
    if (!info) {
        desc_set_error("null info");
        return DESC_B200_ERR_ARG;
    }
    info[0] = h->n;
    info[1] = h->m;
    info[2] = h->m_pos;
    info[3] = h->m_cycle;
    info[4] = h->n_sample;
    info[5] = h->max_ns;
    info[6] = h->e_begin;
    info[7] = h->e_end;
    info[8] = h->n_slots;
    info[9] = h->max_codeg;
    return DESC_B200_OK;
}

#define NEED_BUILT(h)                                                \
    if (!(h)->built) {                                               \
        desc_set_error("incidence not built yet");                   \
        return DESC_B200_ERR_STATE;                                  \
    }

int desc_b200_get_codeg(desc_b200_handle* h, int32_t* codeg) {
    DESC_TRY(check_handle(h));
    NEED_BUILT(h);
    if (codeg) CUDA_TRY(cudaMemcpyAsync(codeg, h->codeg, h->m * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return DESC_B200_OK;
}

int desc_b200_get_incidence(desc_b200_handle* h, int64_t* rowptr, int32_t* apex) {
    DESC_TRY(check_handle(h));
    NEED_BUILT(h);
    if (rowptr) CUDA_TRY(cudaMemcpyAsync(rowptr, h->rowptr, (h->m + 1) * sizeof(int64_t), cudaMemcpyDeviceToHost, h->stream));
    if (apex && h->m_cycle > 0)
        CUDA_TRY(cudaMemcpyAsync(apex, h->apex, h->m_cycle * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return DESC_B200_OK;
}

__global__ void k_unpack(const uint32_t* __restrict__ pk, int64_t ns, int32_t* __restrict__ eid,
                         uint8_t* __restrict__ app) {
    int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (s >= ns) return;
    uint32_t v = pk[s];
    if (eid) eid[s] = (int32_t)(v & PK_MASK);
    if (app) app[s] = (v & PK_APP) ? 1 : 0;
}

int desc_b200_get_slots(desc_b200_handle* h, int32_t* e_jk, int32_t* e_ki, uint8_t* ikj_appears,
                        uint8_t* jki_appears) {
    DESC_TRY(check_handle(h));
    NEED_BUILT(h);
    const int64_t ns = h->n_slots;
    if (ns == 0) return DESC_B200_OK;
    int32_t* d_e = nullptr;
    uint8_t* d_a = nullptr;
    CUDA_TRY(cudaMalloc(&d_e, ns * sizeof(int32_t)));
    CUDA_TRY(cudaMalloc(&d_a, ns));
    const unsigned gb = (unsigned)((ns + 255) / 256);
    // pk_jk carries JKI_appears, pk_ki carries IKJ_appears (internal.cuh)
    k_unpack<<<gb, 256, 0, h->stream>>>(h->pk_jk, ns, d_e, d_a);
    KERNEL_CHECK(h);
    if (e_jk) CUDA_TRY(cudaMemcpyAsync(e_jk, d_e, ns * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (jki_appears) CUDA_TRY(cudaMemcpyAsync(jki_appears, d_a, ns, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    k_unpack<<<gb, 256, 0, h->stream>>>(h->pk_ki, ns, d_e, d_a);
    KERNEL_CHECK(h);
    if (e_ki) CUDA_TRY(cudaMemcpyAsync(e_ki, d_e, ns * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (ikj_appears) CUDA_TRY(cudaMemcpyAsync(ikj_appears, d_a, ns, cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    cudaFree(d_e);
    cudaFree(d_a);
    return DESC_B200_OK;
}

int desc_b200_get_s0(desc_b200_handle* h, double* S0_long) {
    DESC_TRY(check_handle(h));
    if (!h->have_s0) {
        desc_set_error("cycle_inconsistency has not run");
        return DESC_B200_ERR_STATE;
    }
    if (S0_long && h->n_slots > 0)
        CUDA_TRY(cudaMemcpyAsync(S0_long, h->S0, h->n_slots * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return DESC_B200_OK;
}

int desc_b200_get_w(desc_b200_handle* h, double* wijk) {
    DESC_TRY(check_handle(h));
    if (!h->have_pgd) {
        desc_set_error("pgd has not run");
        return DESC_B200_ERR_STATE;
    }
    if (wijk && h->n_slots > 0)
        CUDA_TRY(cudaMemcpyAsync(wijk, h->w[h->final_buf], h->n_slots * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return DESC_B200_OK;
}

int desc_b200_get_gcw_info(desc_b200_handle* h, double info[8]) {
    DESC_TRY(check_handle(h));
    if (!h->have_gcw || !info) {
        desc_set_error("gcw has not run");
        return DESC_B200_ERR_STATE;
    }
    info[0] = h->tm.gcw_iters;
    info[1] = h->gcw_last_res;
    info[2] = h->gcw_theta[0];
    info[3] = h->gcw_theta[1];
    info[4] = h->gcw_theta[2];
    info[5] = info[6] = info[7] = 0.0;
    return DESC_B200_OK;
}

int desc_b200_get_timings(desc_b200_handle* h, desc_b200_timings* t) {
    DESC_TRY(check_handle(h));
    if (!t) {
        desc_set_error("null timings");
        return DESC_B200_ERR_ARG;
    }
    h->tm.total_launches = h->launches;
    *t = h->tm;
    return DESC_B200_OK;
}

int desc_b200_sync(desc_b200_handle* h) {
    DESC_TRY(check_handle(h));
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    return DESC_B200_OK;
}

}  // extern "C"
