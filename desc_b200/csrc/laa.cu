// DESC step 5: weighted Lie-algebraic averaging refinement (reference: Algorithms/DESC.m:265-312,
// Utils/Weighted_LAA.m:4-52, Build_Amatrix.m, R2Q.m, q2R.m).  SURVEY 8(f) "next" #1.
//
// Per IRLS iteration:
//   * per edge: residual quaternion inv(Qj) Qij Qi and its log map B (Weighted_LAA.m:12-36)
//   * weighted least squares (diag(W) A) \ (W .* B), A = signed edge-node incidence with node 1
//     grounded (Build_Amatrix.m): the reference calls sparse QR; the minimiser is unique, so the
//     normal equations (A' W^2 A) x = A' W^2 B - a grounded weighted graph Laplacian, SPD - are solved
//     here by Jacobi-preconditioned CG for the three right-hand sides at once (block-sparse SpMV over
//     the symmetric adjacency, warp per node, no atomics, fixed-order reductions)
//   * exponential map + quaternion update of every node (Weighted_LAA.m:42-52)
//   * per edge: residual of the UPDATE QUATERNION (DESC.m:290 multiplies A with the quaternion part
//     the reference returns in W, not with the rotation vector - reproduced as is), mixing with S_vec,
//     new weights, and the MATLAB-quantile threshold (DESC.m:291-303) by radix selection.
#include "internal.cuh"

#include <algorithm>
#include <cstdlib>
#include <cmath>

namespace {
constexpr int LAA_RED_BLOCKS = 256;   // partial-sum blocks of the reductions (fixed: deterministic)
constexpr int LAA_TB = 256;
constexpr double LAA_PI = 3.14159265358979323846;

// Utils/R2Q.m:9-12.  transposed=1: quaternion of R' (DESC.m:265 `permute`)
__global__ void k_laa_r2q(const double* __restrict__ R, int64_t count, int transposed, double* __restrict__ Q) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i >= count) return;
    const double* r = R + 9 * i;   // MATLAB layout: (row, col) at row + 3 col
    double q0 = (r[0] + r[4] + r[8] - 1.0) / 2.0;
    double v1 = (r[2 + 3 * 1] - r[1 + 3 * 2]) / 2.0;   // R(3,2) - R(2,3)
    double v2 = (r[0 + 3 * 2] - r[2 + 3 * 0]) / 2.0;   // R(1,3) - R(3,1)
    double v3 = (r[1 + 3 * 0] - r[0 + 3 * 1]) / 2.0;   // R(2,1) - R(1,2)
    if (transposed) {
        v1 = -v1;
        v2 = -v2;
        v3 = -v3;
    }
    q0 = sqrt((q0 + 1.0) / 2.0);
    Q[4 * i] = q0;
    Q[4 * i + 1] = (v1 / q0) / 2.0;
    Q[4 * i + 2] = (v2 / q0) / 2.0;
    Q[4 * i + 3] = (v3 / q0) / 2.0;
}

// initial weights (DESC.m:276-282): thresh = quantile(S, 1) = max(S), so no edge is truncated
__global__ void k_laa_init_weights(const double* __restrict__ S, int64_t m, double wmax, double* __restrict__ W) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    const double w = 1.0 / pow(S[e], 0.75);
    W[e] = w > wmax ? wmax : w;
}

// Weighted_LAA.m:12-36: B = log map of inv(Qj) * Qij * Qi
__global__ void k_laa_residual(const int* __restrict__ ei, const int* __restrict__ ej, const double* __restrict__ Q,
                               const double* __restrict__ QQ, int64_t m, double* __restrict__ B) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    const double* qi = Q + 4 * (int64_t)ei[e];
    const double* qj = Q + 4 * (int64_t)ej[e];
    const double* qq = QQ + 4 * e;
    const double a0 = qq[0], a1 = qq[1], a2 = qq[2], a3 = qq[3];
    const double b0 = qi[0], b1 = qi[1], b2 = qi[2], b3 = qi[3];
    // w = Qij * Qi
    const double w0 = a0 * b0 - (a1 * b1 + a2 * b2 + a3 * b3);
    const double w1 = a0 * b1 + b0 * a1 + (a2 * b3 - a3 * b2);
    const double w2 = a0 * b2 + b0 * a2 + (a3 * b1 - a1 * b3);
    const double w3 = a0 * b3 + b0 * a3 + (a1 * b2 - a2 * b1);
    // w = inv(Qj) * w
    const double c0 = qj[0], c1 = qj[1], c2 = qj[2], c3 = qj[3];
    const double u0 = -c0 * w0 - (c1 * w1 + c2 * w2 + c3 * w3);
    const double u1 = -c0 * w1 + w0 * c1 + (c2 * w3 - c3 * w2);
    const double u2 = -c0 * w2 + w0 * c2 + (c3 * w1 - c1 * w3);
    const double u3 = -c0 * w3 + w0 * c3 + (c1 * w2 - c2 * w1);
    const double s2 = sqrt(u1 * u1 + u2 * u2 + u3 * u3);
    double th = 2.0 * atan2(s2, u0);
    if (th < -LAA_PI) th += 2.0 * LAA_PI;
    if (th >= LAA_PI) th -= 2.0 * LAA_PI;
    const double f = th / s2;
    double o1 = u1 * f, o2 = u2 * f, o3 = u3 * f;
    if (isnan(o1)) o1 = 0.0;   // Weighted_LAA.m:36
    if (isnan(o2)) o2 = 0.0;
    if (isnan(o3)) o3 = 0.0;
    B[3 * e] = o1;
    B[3 * e + 1] = o2;
    B[3 * e + 2] = o3;
}

// squared weights in adjacency order (read contiguously by the SpMV)
__global__ void k_laa_w2adj(const int* __restrict__ adj_eid, const double* __restrict__ W, int64_t n2m,
                            double* __restrict__ w2adj) {
    const int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (p >= n2m) return;
    const double w = W[adj_eid[p]];
    w2adj[p] = w * w;
}

// rhs = A' W^2 B and the Jacobi diagonal of A' W^2 A; node 0 is grounded (Build_Amatrix.m:12)
__global__ void __launch_bounds__(LAA_TB)
k_laa_rhs(const int* __restrict__ rowstart, const int* __restrict__ adj_nbr, const int* __restrict__ adj_eid,
          const double* __restrict__ w2adj, const double* __restrict__ B, int n, double* __restrict__ rhs,
          double* __restrict__ diag) {
    const int node = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (node >= n) return;
    double a0 = 0.0, a1 = 0.0, a2 = 0.0, d = 0.0;
    const int p1 = rowstart[node + 1];
    for (int p = rowstart[node] + lane; p < p1; p += 32) {
        const int nb = adj_nbr[p];
        const int64_t e = adj_eid[p];
        const double w2 = w2adj[p];
        const double sg = node > nb ? w2 : -w2;   // +1 at the larger endpoint j, -1 at i
        a0 += sg * B[3 * e];
        a1 += sg * B[3 * e + 1];
        a2 += sg * B[3 * e + 2];
        d += w2;
    }
    a0 = group_sum<32>(a0);
    a1 = group_sum<32>(a1);
    a2 = group_sum<32>(a2);
    d = group_sum<32>(d);
    if (lane == 0) {
        const bool g = node == 0;
        rhs[3 * node] = g ? 0.0 : a0;
        rhs[3 * node + 1] = g ? 0.0 : a1;
        rhs[3 * node + 2] = g ? 0.0 : a2;
        diag[node] = d;
    }
}

// Y = (A' W^2 A) X for the three columns; X[0,:] is pinned to zero (grounded node)
__global__ void __launch_bounds__(LAA_TB)
k_laa_matvec(const int* __restrict__ rowstart, const int* __restrict__ adj_nbr, const double* __restrict__ w2adj,
             const double* __restrict__ X, int n, double* __restrict__ Y) {
    const int node = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (node >= n) return;
    const double x0 = X[3 * node], x1 = X[3 * node + 1], x2 = X[3 * node + 2];
    double a0 = 0.0, a1 = 0.0, a2 = 0.0;
    const int p1 = rowstart[node + 1];
    for (int p = rowstart[node] + lane; p < p1; p += 32) {
        const int nb = adj_nbr[p];
        const double w2 = w2adj[p];
        a0 += w2 * (x0 - X[3 * nb]);
        a1 += w2 * (x1 - X[3 * nb + 1]);
        a2 += w2 * (x2 - X[3 * nb + 2]);
    }
    a0 = group_sum<32>(a0);
    a1 = group_sum<32>(a1);
    a2 = group_sum<32>(a2);
    if (lane == 0) {
        const bool g = node == 0;
        Y[3 * node] = g ? 0.0 : a0;
        Y[3 * node + 1] = g ? 0.0 : a1;
        Y[3 * node + 2] = g ? 0.0 : a2;
    }
}

// column-wise dot products of two n x 3 arrays -> partial[block][3] (fixed shape: deterministic)
__global__ void __launch_bounds__(LAA_TB)
k_laa_dot(const double* __restrict__ Xa, const double* __restrict__ Xb, int n, double* __restrict__ partial) {
    double s[3] = {0.0, 0.0, 0.0};
    for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x)
#pragma unroll
        for (int c = 0; c < 3; c++) s[c] += Xa[3 * v + c] * Xb[3 * v + c];
    __shared__ double sh[3][LAA_TB / 32];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        s[c] = group_sum<32>(s[c]);
        if ((threadIdx.x & 31) == 0) sh[c][threadIdx.x >> 5] = s[c];
    }
    __syncthreads();
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int w = 0; w < LAA_TB / 32; w++) t += sh[threadIdx.x][w];
        partial[3 * blockIdx.x + threadIdx.x] = t;
    }
}
// out[0..2] = sum over blocks
__global__ void k_laa_dot_finish(const double* __restrict__ partial, int nblocks, double* __restrict__ out) {
    if (threadIdx.x < 3) {
        double t = 0.0;
        for (int b = 0; b < nblocks; b++) t += partial[3 * b + threadIdx.x];
        out[threadIdx.x] = t;
    }
}

// scalars: [0..2] rz, [3..5] pAp, [6..8] rz_new, [9..11] rr, [12..14] bb
// x += alpha p ; r -= alpha Ap ; z = r / diag      (alpha = rz / pAp per column)
__global__ void k_laa_cg_update(int n, const double* __restrict__ sc, const double* __restrict__ P,
                                const double* __restrict__ AP, const double* __restrict__ diag, double* __restrict__ X,
                                double* __restrict__ R, double* __restrict__ Z) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const double dinv = v > 0 ? 1.0 / diag[v] : 0.0;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const double pap = sc[3 + c];
        const double alpha = pap != 0.0 ? sc[c] / pap : 0.0;
        X[3 * v + c] += alpha * P[3 * v + c];
        const double r = R[3 * v + c] - alpha * AP[3 * v + c];
        R[3 * v + c] = r;
        Z[3 * v + c] = r * dinv;
    }
}
// p = z + beta p (beta = rz_new / rz); then rz <- rz_new (done by the host-side swap of scalar slots)
__global__ void k_laa_cg_pupdate(int n, const double* __restrict__ sc, const double* __restrict__ Z, double* __restrict__ P) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const double rz = sc[c];
        const double beta = rz != 0.0 ? sc[6 + c] / rz : 0.0;
        P[3 * v + c] = Z[3 * v + c] + beta * P[3 * v + c];
    }
}
__global__ void k_laa_copy3(double* dst, const double* src) {
    if (threadIdx.x < 3) dst[threadIdx.x] = src[threadIdx.x];
}
// z = r / diag, p = z, x = 0 with r = rhs
__global__ void k_laa_cg_start(int n, const double* __restrict__ rhs, const double* __restrict__ diag, double* __restrict__ X,
                               double* __restrict__ R, double* __restrict__ Z, double* __restrict__ P) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const double dinv = v > 0 ? 1.0 / diag[v] : 0.0;
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const double r = rhs[3 * v + c];
        X[3 * v + c] = 0.0;
        R[3 * v + c] = r;
        Z[3 * v + c] = r * dinv;
        P[3 * v + c] = r * dinv;
    }
}

// Weighted_LAA.m:42-52: score partials, exponential map, Q <- Q * W; Wq = vector part of the update quaternion
__global__ void __launch_bounds__(LAA_TB)
k_laa_node_update(int n, const double* __restrict__ X, double* __restrict__ Q, double* __restrict__ Wq,
                  double* __restrict__ partial) {
    double sc = 0.0;
    for (int v = blockIdx.x * blockDim.x + threadIdx.x; v < n; v += gridDim.x * blockDim.x) {
        double o1 = 0.0, o2 = 0.0, o3 = 0.0;
        if (v > 0) {
            o1 = X[3 * v];
            o2 = X[3 * v + 1];
            o3 = X[3 * v + 2];
        }
        const double theta = sqrt(o1 * o1 + o2 * o2 + o3 * o3);
        if (v > 0) sc += theta;
        double w0 = cos(theta / 2.0);
        const double f = sin(theta / 2.0) / theta;
        double w1 = o1 * f, w2 = o2 * f, w3 = o3 * f;
        if (isnan(w0)) w0 = 0.0;   // Weighted_LAA.m:48
        if (isnan(w1)) w1 = 0.0;
        if (isnan(w2)) w2 = 0.0;
        if (isnan(w3)) w3 = 0.0;
        if (v == 0) {              // W(1,:) = [1 0 0 0] (:38); theta = 0 => 0/0 -> NaN -> 0, cos(0) = 1
            w0 = 1.0;
            w1 = w2 = w3 = 0.0;
        }
        Wq[3 * v] = w1;
        Wq[3 * v + 1] = w2;
        Wq[3 * v + 2] = w3;
        const double q0 = Q[4 * v], q1 = Q[4 * v + 1], q2 = Q[4 * v + 2], q3 = Q[4 * v + 3];
        Q[4 * v] = q0 * w0 - (q1 * w1 + q2 * w2 + q3 * w3);
        Q[4 * v + 1] = q0 * w1 + w0 * q1 + (q2 * w3 - q3 * w2);
        Q[4 * v + 2] = q0 * w2 + w0 * q2 + (q3 * w1 - q1 * w3);
        Q[4 * v + 3] = q0 * w3 + w0 * q3 + (q1 * w2 - q2 * w1);
    }
    sc = group_sum<32>(sc);
    __shared__ double sh[LAA_TB / 32];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = sc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < LAA_TB / 32; w++) t += sh[w];
        partial[blockIdx.x] = t;
    }
}
__global__ void k_laa_sum_finish(const double* __restrict__ partial, int nblocks, double scale, double* __restrict__ out) {
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int b = 0; b < nblocks; b++) t += partial[b];
        out[0] = t * scale;
    }
}

// DESC.m:290-298: E = A*Wq - B, ResVec = |E|/pi, RSVec = (1-lam) ResVec + lam S, Weights = min(RSVec^-0.75, wmax)
__global__ void k_laa_edge_update(const int* __restrict__ ei, const int* __restrict__ ej, const double* __restrict__ Wq,
                                  const double* __restrict__ B, const double* __restrict__ S, int64_t m, double lam,
                                  double wmax, double* __restrict__ RS, double* __restrict__ W) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int i = ei[e], j = ej[e];
    double e0 = -B[3 * e], e1 = -B[3 * e + 1], e2 = -B[3 * e + 2];
    if (j > 0) {   // (the grounded node has no column)
        e0 += Wq[3 * j];
        e1 += Wq[3 * j + 1];
        e2 += Wq[3 * j + 2];
    }
    if (i > 0) {
        e0 -= Wq[3 * i];
        e1 -= Wq[3 * i + 1];
        e2 -= Wq[3 * i + 2];
    }
    const double res = sqrt(e0 * e0 + e1 * e1 + e2 * e2) / LAA_PI;
    const double rs = (1.0 - lam) * res + lam * S[e];
    RS[e] = rs;
    const double w = 1.0 / pow(rs, 0.75);
    W[e] = w > wmax ? wmax : w;
}
// MPLS.m:241-242: RHVec = (1-alpha) ResVec + alpha HVec (in place in RS), Weights = min(RHVec^-0.75, wmax)
__global__ void k_laa_mix(const double* __restrict__ H, int64_t m, double alpha, double wmax, double* __restrict__ RS,
                          double* __restrict__ W) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    const double rs = (1.0 - alpha) * RS[e] + alpha * H[e];
    RS[e] = rs;
    const double w = 1.0 / pow(rs, 0.75);
    W[e] = w > wmax ? wmax : w;
}
__global__ void k_laa_truncate(const double* __restrict__ RS, int64_t m, double thresh, double wmin, double* __restrict__ W) {
    const int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (e >= m) return;
    if (RS[e] > thresh) W[e] = wmin;
}

// radix selection on the bit patterns of non-negative doubles (monotone): histogram of the `width`-bit
// digit at `shift` over the keys whose higher bits equal `prefix`
__global__ void __launch_bounds__(LAA_TB)
k_laa_hist(const double* __restrict__ X, int64_t m, uint64_t prefix, int shift, int width, int first,
           unsigned* __restrict__ hist) {
    __shared__ unsigned sh[2048];
    for (int b = threadIdx.x; b < 2048; b += blockDim.x) sh[b] = 0u;
    __syncthreads();
    const uint64_t mask = (1ull << width) - 1ull;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < m; e += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t k = (uint64_t)__double_as_longlong(X[e]);
        if (first || (k >> (shift + width)) == prefix) atomicAdd(&sh[(k >> shift) & mask], 1u);
    }
    __syncthreads();
    for (int b = threadIdx.x; b < 2048; b += blockDim.x)
        if (sh[b]) atomicAdd(&hist[b], sh[b]);
}

// Utils/q2R.m
__global__ void k_laa_q2r(const double* __restrict__ Q, int n, double* __restrict__ R) {
    const int v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v >= n) return;
    const double c2 = Q[4 * v];
    double* r = R + 9 * (int64_t)v;
    if (fabs(fabs(c2) - 1.0) > 1e-12) {
        const double q1 = Q[4 * v + 1], q2 = Q[4 * v + 2], q3 = Q[4 * v + 3];
        const double s2 = sqrt(q1 * q1 + q2 * q2 + q3 * q3);
        const double s = 2.0 * s2 * c2;
        const double c = 2.0 * c2 * c2 - 1.0;
        const double n1 = q1 / s2, n2 = q2 / s2, n3 = q3 / s2;
        const double cc = 1.0 - c;
        const double n12 = n1 * n2 * cc, n23 = n2 * n3 * cc, n31 = n3 * n1 * cc;
        const double n1s = n1 * s, n2s = n2 * s, n3s = n3 * s;
        r[0] = c + n1 * n1 * cc;  r[3] = n12 - n3s;         r[6] = n31 + n2s;
        r[1] = n12 + n3s;         r[4] = c + n2 * n2 * cc;  r[7] = n23 - n1s;
        r[2] = n31 - n2s;         r[5] = n23 + n1s;         r[8] = c + n3 * n3 * cc;
    } else {
        r[0] = 1.0; r[1] = 0.0; r[2] = 0.0; r[3] = 0.0; r[4] = 1.0; r[5] = 0.0; r[6] = 0.0; r[7] = 0.0; r[8] = 1.0;
    }
}

// k-th smallest (1-based) of the non-negative doubles X[0..m): six passes of 11-bit digits, MSB first
int laa_select(desc_b200_handle* h, const double* X, int64_t m, int64_t k, unsigned* d_hist, double* out) {
    uint64_t prefix = 0;
    unsigned hist[2048];
    const int shifts[6] = {53, 42, 31, 20, 9, 0};
    const int widths[6] = {11, 11, 11, 11, 11, 9};
    for (int pass = 0; pass < 6; pass++) {
        CUDA_TRY(cudaMemsetAsync(d_hist, 0, 2048 * sizeof(unsigned), h->stream));
        k_laa_hist<<<DESC_SMS * 4, LAA_TB, 0, h->stream>>>(X, m, prefix, shifts[pass], widths[pass], pass == 0, d_hist);
        KERNEL_CHECK(h);
        CUDA_TRY(cudaMemcpyAsync(hist, d_hist, sizeof(hist), cudaMemcpyDeviceToHost, h->stream));
        CUDA_TRY(cudaStreamSynchronize(h->stream));
        const int nb = 1 << widths[pass];
        int64_t cum = 0;
        int b = 0;
        for (; b < nb; b++) {
            if (cum + (int64_t)hist[b] >= k) break;
            cum += hist[b];
        }
        if (b >= nb) {
            desc_set_error("radix selection failed (NaN or negative residual?)");
            return DESC_B200_ERR_STATE;
        }
        k -= cum;
        prefix = (prefix << widths[pass]) | (uint64_t)b;
    }
    long long bits = (long long)prefix;
    memcpy(out, &bits, sizeof(double));
    return DESC_B200_OK;
}
}  // namespace

int desc_select_kth(desc_b200_handle* h, const double* X, int64_t m, int64_t k, unsigned* d_hist, double* out) {
    return laa_select(h, X, m, k, d_hist, out);
}

// MATLAB quantile(x, p) of a device vector of non-negative doubles (DESC.m:276,301)
static int laa_quantile(desc_b200_handle* h, const double* X, int64_t m, double p, unsigned* d_hist, double* out) {
    const double pos = (double)m * p + 0.5;
    int64_t lo;
    double frac = 0.0;
    if (pos <= 1.0) {
        lo = 1;
    } else if (pos >= (double)m) {
        lo = m;
    } else {
        lo = (int64_t)std::floor(pos);
        frac = pos - (double)lo;
    }
    double a = 0.0, b = 0.0;
    DESC_TRY(laa_select(h, X, m, lo, d_hist, &a));
    if (frac > 0.0 && lo < m) {
        DESC_TRY(laa_select(h, X, m, lo + 1, d_hist, &b));
        *out = a + frac * (b - a);
    } else {
        *out = a;
    }
    return DESC_B200_OK;
}

int desc_laa_impl(desc_b200_handle* h, const double* d_S, const double* d_Rinit, double* d_Rout, int max_iters,
                  double stop_threshold, int* iters_run, double* scores_host, const desc_laa_sched* mpls) {
    // Multi-GPU handles: every rank runs the whole refinement on the replicated graph and the all-gathered S_vec
    // (a 2 ms stage at cfg 4: sharding its CG would cost more in collectives than it saves).  All ranks execute the
    // same kernels on the same data, so scores / trip counts agree and the collectives inside the MPLS variant's
    // cycle reweighting (edge-sharded, desc_cemp_reweight) stay in lockstep.
    const int n = h->n;
    const int64_t m = h->m;
    cudaStream_t st = h->stream;
    const double wmax = 1e4, wmin = 1e-4, qmin = 0.8;
    double *Q, *QQ, *W, *B, *RS, *w2adj, *rhs, *diag, *X, *R, *Z, *P, *AP, *Wq, *partial, *sc;
    unsigned* d_hist;
    CUDA_TRY(cudaMalloc(&Q, (size_t)4 * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&QQ, (size_t)4 * m * sizeof(double)));
    CUDA_TRY(cudaMalloc(&W, (size_t)m * sizeof(double)));
    CUDA_TRY(cudaMalloc(&B, (size_t)3 * m * sizeof(double)));
    CUDA_TRY(cudaMalloc(&RS, (size_t)m * sizeof(double)));
    CUDA_TRY(cudaMalloc(&w2adj, (size_t)2 * m * sizeof(double)));
    CUDA_TRY(cudaMalloc(&rhs, (size_t)3 * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&diag, (size_t)n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&X, (size_t)3 * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&R, (size_t)3 * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&Z, (size_t)3 * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&P, (size_t)3 * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&AP, (size_t)3 * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&Wq, (size_t)3 * n * sizeof(double)));
    CUDA_TRY(cudaMalloc(&partial, (size_t)3 * LAA_RED_BLOCKS * sizeof(double)));
    CUDA_TRY(cudaMalloc(&sc, 32 * sizeof(double)));
    CUDA_TRY(cudaMalloc(&d_hist, 2048 * sizeof(unsigned)));
    double* H = nullptr;   // MPLS: cycle-reweighted residuals (HVec)
    if (mpls) CUDA_TRY(cudaMalloc(&H, (size_t)m * sizeof(double)));
    void* to_free[] = {Q, QQ, W, B, RS, w2adj, rhs, diag, X, R, Z, P, AP, Wq, partial, sc, d_hist, H};
    auto cleanup = [&]() {
        for (void* p : to_free)
            if (p) cudaFree(p);
    };
    const unsigned gm = (unsigned)((m + LAA_TB - 1) / LAA_TB), gn = (unsigned)((n + LAA_TB - 1) / LAA_TB);
    const unsigned gw = (unsigned)(((int64_t)n * 32 + LAA_TB - 1) / LAA_TB);
    // CG needs at most n - 1 steps in exact arithmetic; 2n leaves room for rounding on slow-mixing graphs (rings
    // need thousands of steps after the weights are truncated).  DESC_B200_LAA_CG_MAX overrides the cap (tests).
    int cg_max = std::max(1000, 2 * n);
    if (const char* o = getenv("DESC_B200_LAA_CG_MAX")) cg_max = std::max(1, atoi(o));

    k_laa_r2q<<<gn, LAA_TB, 0, st>>>(d_Rinit, n, 0, Q);
    KERNEL_CHECK(h);
    k_laa_r2q<<<gm, LAA_TB, 0, st>>>(h->Rij, m, 1, QQ);
    KERNEL_CHECK(h);
    k_laa_init_weights<<<gm, LAA_TB, 0, st>>>(d_S, m, wmax, W);
    KERNEL_CHECK(h);

    double score = INFINITY, quant_ratio = 1.0;
    int it = 1, cg_total = 0;
    int rc = DESC_B200_OK;
    while (score > stop_threshold && it < max_iters) {
        const double lam = 1.0 / (double)(it + 1);
        k_laa_residual<<<gm, LAA_TB, 0, st>>>(h->ei, h->ej, Q, QQ, m, B);
        KERNEL_CHECK(h);
        k_laa_w2adj<<<(unsigned)((2 * m + LAA_TB - 1) / LAA_TB), LAA_TB, 0, st>>>(h->adj_eid, W, 2 * m, w2adj);
        KERNEL_CHECK(h);
        k_laa_rhs<<<gw, LAA_TB, 0, st>>>(h->rowstart, h->adj_nbr, h->adj_eid, w2adj, B, n, rhs, diag);
        KERNEL_CHECK(h);
        // ---- preconditioned CG on the grounded weighted Laplacian, three right-hand sides
        k_laa_cg_start<<<gn, LAA_TB, 0, st>>>(n, rhs, diag, X, R, Z, P);
        KERNEL_CHECK(h);
        k_laa_dot<<<LAA_RED_BLOCKS, LAA_TB, 0, st>>>(R, Z, n, partial);
        k_laa_dot_finish<<<1, 32, 0, st>>>(partial, LAA_RED_BLOCKS, sc + 0);       // rz
        k_laa_dot<<<LAA_RED_BLOCKS, LAA_TB, 0, st>>>(R, R, n, partial);
        k_laa_dot_finish<<<1, 32, 0, st>>>(partial, LAA_RED_BLOCKS, sc + 12);      // bb
        h->launches += 4;
        double hs[16];
        CUDA_TRY(cudaMemcpyAsync(hs, sc, 16 * sizeof(double), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        const double bb[3] = {hs[12], hs[13], hs[14]};
        bool conv = (bb[0] == 0.0 && bb[1] == 0.0 && bb[2] == 0.0);
        for (int k = 1; k <= cg_max && !conv; k++) {
            k_laa_matvec<<<gw, LAA_TB, 0, st>>>(h->rowstart, h->adj_nbr, w2adj, P, n, AP);
            k_laa_dot<<<LAA_RED_BLOCKS, LAA_TB, 0, st>>>(P, AP, n, partial);
            k_laa_dot_finish<<<1, 32, 0, st>>>(partial, LAA_RED_BLOCKS, sc + 3);   // pAp
            k_laa_cg_update<<<gn, LAA_TB, 0, st>>>(n, sc, P, AP, diag, X, R, Z);
            k_laa_dot<<<LAA_RED_BLOCKS, LAA_TB, 0, st>>>(R, Z, n, partial);
            k_laa_dot_finish<<<1, 32, 0, st>>>(partial, LAA_RED_BLOCKS, sc + 6);   // rz_new
            k_laa_cg_pupdate<<<gn, LAA_TB, 0, st>>>(n, sc, Z, P);
            k_laa_copy3<<<1, 32, 0, st>>>(sc + 0, sc + 6);                          // rz <- rz_new
            h->launches += 8;
            cg_total++;
            if (k % 8 == 0 || k == cg_max) {
                k_laa_dot<<<LAA_RED_BLOCKS, LAA_TB, 0, st>>>(R, R, n, partial);
                k_laa_dot_finish<<<1, 32, 0, st>>>(partial, LAA_RED_BLOCKS, sc + 9);   // rr
                h->launches += 2;
                CUDA_TRY(cudaMemcpyAsync(hs, sc, 16 * sizeof(double), cudaMemcpyDeviceToHost, st));
                CUDA_TRY(cudaStreamSynchronize(st));
                conv = true;
                for (int c = 0; c < 3; c++)
                    if (hs[9 + c] > 1e-26 * bb[c]) conv = false;   // |r| <= 1e-13 |b|
            }
        }
        CUDA_TRY(cudaGetLastError());
        if (!conv) {   // an unconverged solve would move every node by a wrong step and still report success
            double rel = 0.0;
            for (int c = 0; c < 3; c++)
                if (bb[c] > 0.0) rel = std::max(rel, std::sqrt(hs[9 + c] / bb[c]));
            desc_set_error("LAA refinement: CG did not reach |r| <= 1e-13 |b| in %d iterations (relative residual %.3e) "
                           "in IRLS iteration %d", cg_max, rel, it);
            rc = DESC_B200_ERR_NOCONV;
            break;
        }
        // ---- node update, score
        k_laa_node_update<<<LAA_RED_BLOCKS, LAA_TB, 0, st>>>(n, X, Q, Wq, partial);
        KERNEL_CHECK(h);
        k_laa_sum_finish<<<1, 32, 0, st>>>(partial, LAA_RED_BLOCKS, 1.0 / (double)n, sc + 15);
        KERNEL_CHECK(h);
        CUDA_TRY(cudaMemcpyAsync(&score, sc + 15, sizeof(double), cudaMemcpyDeviceToHost, st));
        // ---- edge residuals, new weights, quantile truncation
        k_laa_edge_update<<<gm, LAA_TB, 0, st>>>(h->ei, h->ej, Wq, B, d_S, m, mpls ? 0.0 : lam, wmax, RS, W);
        KERNEL_CHECK(h);
        double thresh = 0.0;
        if (mpls) {
            // MPLS.m:224-244: RS holds ResVec (lam = 0); HVec = cycle reweighting of the residuals, convex mix, quantile
            const int idx = std::min(it - 1, mpls->len - 1);
            rc = desc_cemp_reweight(h, RS, H, mpls->beta[idx], mpls->empty_value);
            if (rc != DESC_B200_OK) break;
            k_laa_mix<<<gm, LAA_TB, 0, st>>>(H, m, mpls->alpha[idx], wmax, RS, W);
            KERNEL_CHECK(h);
            rc = laa_quantile(h, RS, m, mpls->tau[idx], d_hist, &thresh);
        } else {
            quant_ratio = std::max(qmin, quant_ratio - 0.05);
            rc = laa_quantile(h, RS, m, quant_ratio, d_hist, &thresh);   // (synchronises: score is valid after it)
        }
        if (rc != DESC_B200_OK) break;
        k_laa_truncate<<<gm, LAA_TB, 0, st>>>(RS, m, thresh, wmin, W);
        KERNEL_CHECK(h);
        if (scores_host) scores_host[it - 1] = score;
        it++;
    }
    if (rc == DESC_B200_OK) {
        k_laa_q2r<<<gn, LAA_TB, 0, st>>>(Q, n, d_Rout);
        h->launches++;
        cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            desc_set_error("CUDA error in the LAA refinement: %s", cudaGetErrorString(e));
            rc = DESC_B200_ERR_CUDA;
        }
    }
    cleanup();
    *iters_run = it - 1;
    h->laa_cg_iters = cg_total;
    return rc;
}
