// A5: cycle inconsistency d_ijk (reference: DESC.m:129-147).
//
//   S0_long(c) = abs(acos((trace(R_ij * R_jk * R_ki) - 1) / 2)) / pi
//
// R_jk = RijMat4d(:,:,j,k) is the stored matrix of edge {j,k} if j<k, else its transpose
// (DESC.m:65-66); likewise R_ki = RijMat4d(:,:,k,i).
//
// Bit-level parity (SURVEY H2): the reference accumulates the two 3x3 products with separate
// multiply and add roundings, from zero, index j = 1,2,3 (bsxfun loops DESC.m:137-143), and the
// trace as (C11+C22)+C33 (DESC.m:146).  The kernel does exactly that with __dmul_rn/__dadd_rn so
// no FMA contraction can change (trace-1)/2 -- which matters because acos is infinitely
// ill-conditioned at 1 and exactly-consistent cycles land there.  For arguments a few ulp outside
// [-1,1] MATLAB's acos goes complex and abs() takes the modulus: acosh(x) for x>1,
// sqrt(pi^2+acosh(-x)^2) for x<-1.
//
// Layout: one group of G lanes per edge (G chosen from the slot budget), lanes stride over the edge's slots, so a
// warp works on 32 slots at a time.  R_ij is loaded once per group (broadcast).  The two partner rotations of the
// warp's 32 slots (random 72-byte records, 8-byte aligned) are gathered COOPERATIVELY: in 9 rounds lane L loads the
// 8-byte word (32 t + L) of the concatenated 32 records, i.e. 9 consecutive lanes read one record as one contiguous
// 72-byte piece (1-2 L1 wavefronts per record instead of the 9 of a per-lane scalar gather, which made the first
// version load/store-pipe bound: 18 wavefronts per slot, 7.5 ms at cfg 4).  The words go through a per-warp staging
// buffer in shared memory (written contiguously, read back with stride 9 doubles: odd, conflict-free) to the lane
// that owns the slot.  HBM/L2-bound gather arithmetic; tensor cores deliberately unused (3x3 products).
#include "internal.cuh"
#include "so3.cuh"

// M(r,c) of a stored column-major 3x3, optionally transposed
#define MAT(p, r, c, tr) ((tr) ? (p)[(c) + 3 * (r)] : (p)[(r) + 3 * (c)])
#define CYC_WARPS 8
#ifndef CYC_MINB
#define CYC_MINB 3   // resident CTAs per SM the register budget is capped for (3: 80 registers, 24 warps per SM)
#endif

template <int G>
__global__ void __launch_bounds__(CYC_WARPS * 32, CYC_MINB)
k_cycle(const double* __restrict__ Rij, const int64_t* __restrict__ rowptr,
        const uint32_t* __restrict__ pk_jk, const uint32_t* __restrict__ pk_ki,
        double* __restrict__ S0, int64_t e0, int64_t e1, int64_t slot_base) {
    __shared__ double stage[CYC_WARPS][2][288];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int r = lane & (G - 1), g = lane / G;
    constexpr int GPW = 32 / G;                    // edges per warp
    const int64_t warp = (int64_t)blockIdx.x * CYC_WARPS + wib;
    const int64_t nwarps = (int64_t)gridDim.x * CYC_WARPS;
    double* sb = stage[wib][0];
    double* sc = stage[wib][1];
    for (int64_t eb = e0 + warp * GPW; eb < e1; eb += nwarps * GPW) {
        const int64_t e = eb + g;
        int64_t s0 = 0;
        int ns = 0;
        if (e < e1) {
            s0 = rowptr[e];
            ns = (int)(rowptr[e + 1] - s0);
        }
        double a[9];
#pragma unroll
        for (int x = 0; x < 9; x++) a[x] = ns > 0 ? __ldg(Rij + 9 * e + x) : 0.0;  // a[r+3c] = R_ij(r,c)
        const int trips = __reduce_max_sync(0xffffffffu, (ns + G - 1) / G);
        for (int it = 0; it < trips; it++) {
            const int idx = r + it * G;
            const bool ok = idx < ns;
            const int64_t s = s0 + idx - slot_base;
            uint32_t pj = 0u, pi = 0u;
            if (ok) {
                pj = __ldcs(pk_jk + s);
                pi = __ldcs(pk_ki + s);
            }
            const unsigned okmask = __ballot_sync(0xffffffffu, ok);
            // cooperative gather: word w = 32 t + lane of the 32 concatenated records
#pragma unroll
            for (int t = 0; t < 9; t++) {
                const int w = t * 32 + lane;
                const int rec = w / 9, el = w - 9 * rec;
                const uint32_t qj = __shfl_sync(0xffffffffu, pj, rec), qi = __shfl_sync(0xffffffffu, pi, rec);
                double vb = 0.0, vc = 0.0;
                if ((okmask >> rec) & 1u) {
                    vb = __ldg(Rij + 9 * (int64_t)(qj & PK_MASK) + el);
                    vc = __ldg(Rij + 9 * (int64_t)(qi & PK_MASK) + el);
                }
                sb[w] = vb;
                sc[w] = vc;
            }
            __syncwarp();
            double b[9], c[9];
#pragma unroll
            for (int x = 0; x < 9; x++) {
                b[x] = sb[9 * lane + x];
                c[x] = sc[9 * lane + x];
            }
            __syncwarp();
            const bool tb = !(pj & PK_SEL);  // j>k: stored (k,j) -> transpose
            const bool tc = (pi & PK_SEL);   // i<k: stored (i,k), need (k,i) -> transpose
            double d[3];
#pragma unroll
            for (int q = 0; q < 3; q++) {
                // C0(q,t) = ((0 + A(q,0)B(0,t)) + A(q,1)B(1,t)) + A(q,2)B(2,t)
                double c0[3];
#pragma unroll
                for (int t = 0; t < 3; t++) {
                    double acc = __dmul_rn(a[q + 0], MAT(b, 0, t, tb));
                    acc = __dadd_rn(acc, __dmul_rn(a[q + 3], MAT(b, 1, t, tb)));
                    acc = __dadd_rn(acc, __dmul_rn(a[q + 6], MAT(b, 2, t, tb)));
                    c0[t] = acc;
                }
                // C(q,q) = ((0 + C0(q,0)Rki(0,q)) + C0(q,1)Rki(1,q)) + C0(q,2)Rki(2,q)
                double acc = __dmul_rn(c0[0], MAT(c, 0, q, tc));
                acc = __dadd_rn(acc, __dmul_rn(c0[1], MAT(c, 1, q, tc)));
                acc = __dadd_rn(acc, __dmul_rn(c0[2], MAT(c, 2, q, tc)));
                d[q] = acc;
            }
            const double tr = __dadd_rn(__dadd_rn(d[0], d[1]), d[2]);
            const double x = __ddiv_rn(__dadd_rn(tr, -1.0), 2.0);
            if (ok) __stcs(S0 + s, __ddiv_rn(abs_acos_dev(x), 3.14159265358979323846));
        }
    }
}

int desc_cycle_impl(desc_b200_handle* h) {
    if (!h->built) {
        desc_set_error("cycle_inconsistency before build_incidence");
        return DESC_B200_ERR_STATE;
    }
    if (h->n_slots > 0) {
        const int grid = DESC_SMS * CYC_MINB;   // persistent: every resident CTA strides over the edges
        if (h->max_ns <= 8)
            k_cycle<8><<<grid, 256, 0, h->stream>>>(h->Rij, h->rowptr, h->pk_jk, h->pk_ki, h->S0, h->e_begin, h->e_end, h->slot_base);
        else if (h->max_ns <= 16)
            k_cycle<16><<<grid, 256, 0, h->stream>>>(h->Rij, h->rowptr, h->pk_jk, h->pk_ki, h->S0, h->e_begin, h->e_end, h->slot_base);
        else
            k_cycle<32><<<grid, 256, 0, h->stream>>>(h->Rij, h->rowptr, h->pk_jk, h->pk_ki, h->S0, h->e_begin, h->e_end, h->slot_base);
        KERNEL_CHECK(h);
    }
    h->have_s0 = true;
    return DESC_B200_OK;
}
