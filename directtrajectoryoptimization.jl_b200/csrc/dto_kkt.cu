// dto_kkt.cu -- device-side consumer of the callback outputs (SURVEY 8f, row N3): the KKT system
//
//        K = [ H + primal_reg I      J'          ]        h = [ grad f + J' y ]
//            [ J                -dual_reg I      ]            [ c             ]
//
// that /root/reference/examples/pendulum/pendulum.jl:138-211 assembles from the five callbacks and
// factors with QDLDL (K = L D L', quasi-definite so no pivoting is needed), for ALL problems of a
// batch at once, from the device-resident J / H / g / c arrays -- nothing but the solution crosses
// PCIe.
//
// Every problem of a batch has the same sparsity, so the host runtime computes ONE bandwidth-
// reducing ordering (reverse Cuthill-McKee, dto_kkt_host.inc) and static gather tables; trajectory
// problems chain knot to knot, so the permuted K is banded (half bandwidth 9-15 for the example
// models). The kernels:
//
//   kkt_rhs_kernel     thread = (problem, row): h in natural order, sums in the reference's loop order
//                      (ascending constraint row, un-fused multiply/add => bit-exact vs the oracle)
//   kkt_band_kernel<W,BW> group of W lanes = problem (W = 16: two problems per warp; W = 32: one):
//                      streaming right-looking banded LDL' with the forward solve fused in, then the
//                      backward solve. Lane i owns row W*blk + i; a row keeps its W band entries in
//                      registers indexed by (column mod W), a compile-time index inside the W-step
//                      unrolled block, so there is no dynamic register indexing. Two row sets
//                      (current block, next block) cover the rows a step can touch (half bandwidth
//                      <= BW < W). Per step: pivot broadcast (shuffle), one reciprocal, the column of
//                      L goes to shared memory (broadcast reads replace 2*BW shuffles) and to HBM
//                      (one coalesced <= 120-byte store; BW+1 values per column, not W), then BW
//                      DFMAs per row set. Rows two blocks ahead are gathered by cp.async. The
//                      backward solve re-reads L column-wise (lane = column, slot = row mod W) so a
//                      retired x_r costs one shuffle + one DFMA instead of a warp reduction.
//   kkt_assemble_kernel test/inspection export of the assembled band (same gather as the factor kernel)
#include <cuda_runtime.h>
#include <stdint.h>

#include "dto_kkt_dev.h"

namespace {

template <int G>
__device__ __forceinline__ double shfl_g(double v, int src)
{
    return __shfl_sync(0xffffffffu, v, src, G);
}

__device__ __forceinline__ void cp_async8_zfill(void* smem, const void* g, int src_size)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(sa), "l"(g), "r"(src_size) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem, const void* g)
{
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait()
{
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// band entries of row (blk*W + i): slot w holds the column c = w (mod W) of [row-W+1, row].
// JbmH = (this problem's J) - nnz_H, so that a table entry s >= nnz_H addresses J[s - nnz_H].
template <bool DIAG = false>
__device__ __forceinline__ double row_shift(const dto_kkt_args& a, size_t row, int64_t b, int64_t bd = -1)
{
    // diagonal shift of permuted row `row`: +primal_reg (per problem when a.preg is given), -dual_reg, 1.0 on padding;
    // DIAG: + the diagonal entry diag[bd][original index] of problem bd (variable AND constraint rows; a candidate slot's
    // regularisation is the slot's, its diagonal the problem's)
    if (a.rowfixed != nullptr && a.rowfixed[row]) return 1.0;   // pinned variable: identity row
    double reg = a.dreg[row];
    if (a.preg != nullptr || (DIAG && a.diag != nullptr)) {
        const int32_t ip = a.iperm[row];
        if (ip >= 0) {
            if (a.preg != nullptr && ip < a.N_z) reg = a.preg[b];
            if (DIAG && a.diag != nullptr) reg += a.diag[(bd >= 0 ? bd : b) * a.dim + ip];
        }
    }
    return reg;
}

// right-hand-side entry of original row ip (natural order, from kkt_rhs_kernel's array hb); padding rows (ip < 0) read 0
__device__ __forceinline__ double rhs_entry(const double* __restrict__ hb, int32_t ip) { return ip < 0 ? 0.0 : hb[ip]; }

template <int W, bool DIAG = false>
__device__ __forceinline__ void load_rows(const dto_kkt_args& a, const double* __restrict__ Hb, const double* __restrict__ JbmH,
                                          int blk, int i, double (&X)[W], int64_t b = 0, int64_t bd = -1)
{
    const int32_t* src = a.src + ((size_t)blk * W) * W + i;
    const double reg = row_shift<DIAG>(a, (size_t)blk * W + i, b, bd);
    int32_t sidx[W];
#pragma unroll
    for (int w = 0; w < W; ++w) sidx[w] = src[w * W];
#pragma unroll
    for (int w = 0; w < W; ++w) {
        const int32_t s = sidx[w];
        const double* bp = (s < a.nnz_H) ? Hb : JbmH;
        double v = 0.0;
        if (s >= 0) v = bp[s];
        // reference: H[i,i] += primal_reg / H[nz+j,nz+j] -= dual_reg after the assignment
        X[w] = (w == i) ? v + reg : v;
    }
}

template <int W, int BW>
struct KktSmem {
    static constexpr int NG = 32 / W;                       // problems per warp
    static constexpr int RING = 3;
    static constexpr int LW = (BW + 2) & ~1;                // doubles per stored column (dto_kkt_col_width)
    static constexpr int SLOT = (W * LW + W) * 8;           // one block of L columns + its y values
    static_assert(RING * SLOT >= W * W * 8, "the forward row stage lives in the ring area");
    static constexpr int PER_GROUP = RING * SLOT + 2 * W * 8;
    static constexpr int BYTES = 4 * NG * PER_GROUP;        // 4 warps per CTA
};

// ---------------- backward solve: x = L^-T y (shared by the factor and resolve kernels) ----------------
template <int W, int BW>
__device__ __forceinline__ void kkt_backward(const dto_kkt_args& a, unsigned char* gsm, const double* Lg, const double* Yg, int nblk, int i,
                                             bool valid, int64_t b)
{
    constexpr int G = W;
    using SM = KktSmem<W, BW>;
    constexpr int LW = SM::LW;
    double A[W], Bv[W];
    // Lane i owns COLUMN j = blk*W + i: slot w holds L(r, j) for the row r = w (mod W) of [j+1, j+W-1].
    // Rows are retired in descending order; the retired x_r is broadcast and the columns that reach it
    // (same block: i < s; block below: i >= s + W - BW) subtract L(r, j) x_r. The factor streams back
    // from HBM through a 3-slot cp.async ring (one 2 KB block of columns + its y per slot), two blocks
    // ahead of use.
    auto issue_cols = [&](int blk) {
        if (blk >= 0) {
            unsigned char* dst = gsm + (blk % SM::RING) * SM::SLOT;
            const unsigned char* srcL = reinterpret_cast<const unsigned char*>(Lg + (size_t)blk * W * LW);
#pragma unroll
            for (int k = 0; k < LW / 2; ++k) cp_async16(dst + (k * W + i) * 16, srcL + (k * W + i) * 16);
            if (i < W / 2) cp_async16(dst + W * LW * 8 + i * 16, reinterpret_cast<const unsigned char*>(Yg + (size_t)blk * W) + i * 16);
        }
        cp_async_commit();
    };
    // inertia: lane i owns column j = blk*W + i, slot 0 of the stored column is the pivot d_j; one load per lane
    // and block here instead of a compare + add per elimination step in the factor loop (padding rows: d = 1)
    int neg = 0;
    auto read_cols = [&](int blk, double (&C)[W], double& acc) {
        const double* sl = reinterpret_cast<const double*>(gsm + (blk % SM::RING) * SM::SLOT);
#pragma unroll
        for (int w = 0; w < W; ++w) {
            const int q = (w - i) & (W - 1);
            C[w] = (q >= 1 && q <= BW) ? sl[i * LW + q] : 0.0;   // (LW-1) odd => conflict-free over the lanes
        }
        acc = sl[W * LW + i];
        neg += sl[i * LW] < 0.0 ? 1 : 0;
    };
    double xa, xp = 0.0;
    issue_cols(nblk - 1);
    issue_cols(nblk - 2);
    issue_cols(nblk - 3);
    cp_async_wait<2>();
    __syncwarp();
    read_cols(nblk - 1, A, xa);
    double* solb = a.sol + b * a.dim;
    for (int blk = nblk - 1; blk >= 0; --blk) {
        cp_async_wait<1>();
        __syncwarp();
        if (blk >= 1) {
            read_cols(blk - 1, Bv, xp);
        } else {
#pragma unroll
            for (int w = 0; w < W; ++w) Bv[w] = 0.0;
            xp = 0.0;
        }
        __syncwarp();            // slot blk % RING (read one iteration ago) is free again
        issue_cols(blk - 3);
#pragma unroll
        for (int s = G - 1; s >= 0; --s) {
            const int p = s & (W - 1);
            const double xr = shfl_g<G>(xa, s);
            if (i < s && i >= s - BW) xa = fma(-A[p], xr, xa);
            if (s - BW < 0) {
                if (i >= s + G - BW) xp = fma(-Bv[p], xr, xp);
            }
        }
        const int32_t ip = a.iperm[(size_t)blk * W + i];
        if (ip >= 0 && valid) solb[ip] = xa;
#pragma unroll
        for (int w = 0; w < W; ++w) A[w] = Bv[w];
        xa = xp;
    }
    cp_async_wait<0>();
    if (a.nneg != nullptr) {   // number of negative pivots of the whole factor: sum over the group's lanes
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) neg += __shfl_xor_sync(0xffffffffu, neg, o, G);
        if (valid && i == 0) a.nneg[b] = neg;
    }
}

// One problem per group of W lanes (two problems per warp for W = 16). Row block = W rows.
// BW = compile-time bound on the half bandwidth (<= W - 1).
// VIRT = candidate launch (dto_kkt_args::virt): outputs and regularisation indexed by slot. A separate instantiation: as a
// run-time switch its extra live index cost the default path registers and spills (acrobot, 64 problems: 0.275 vs 0.204 ms)
// DIAG = a per-problem, per-variable diagonal is added to the Hessian block (dto_kkt_args::diag); separate for the same reason
template <int W, int BW, bool VIRT = false, bool DIAG = false>
__global__ void __launch_bounds__(128, (W == 16 ? 4 : 2)) kkt_band_kernel(const dto_kkt_args a)
{
    constexpr int G = W;
    using SM = KktSmem<W, BW>;
    constexpr int LW = SM::LW;
    extern __shared__ __align__(16) unsigned char kkt_smem[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int grp = lane / G, i = lane % G;
    const int64_t b0 = ((int64_t)blockIdx.x * 4 + wib) * SM::NG + grp;
    const bool valid = b0 < a.B;
    const int64_t bs = valid ? b0 : a.B - 1;         // idle groups shadow the last slot, stores masked
    const int64_t b = a.pidx ? (int64_t)a.pidx[bs] : bs;   // subset launch: slot -> problem
    const int64_t bo = VIRT ? bs : b;                // candidate launch: regularisation, factor, solution, pivot count by slot
    const double* Hb = a.H + b * a.nnz_H;
    const double* Jb = a.J + b * a.nnz_J - a.nnz_H;  // see load_rows
    const double* hb = a.rhs + b * a.dim;
    const int nblk = a.nblk;
    double* Lg = a.L + (size_t)bo * a.factor_stride; // [nblk*W][LW]: slot 0 = pivot d_j, slot q = L(j+q, j)
    double* Yg = Lg + (size_t)nblk * W * LW;         // [nblk*W]: D^-1 L^-1 h
    unsigned char* gsm = kkt_smem + (size_t)(wib * SM::NG + grp) * SM::PER_GROUP;
    double* stage = reinterpret_cast<double*>(gsm);                              // forward: rows of block blk+2, [w][i]
    double (*lcol)[W] = reinterpret_cast<double (*)[W]>(gsm + SM::RING * SM::SLOT);  // un-scaled column, double-buffered

    double A[W], Bv[W];
    double ra, rb = 0.0, rc = 0.0, regc = 0.0;
    int32_t nidx[W];                                  // gather indices of the rows two blocks ahead
    load_rows<W, DIAG>(a, Hb, Jb, 0, i, A, bo, b);
    ra = rhs_entry(hb, a.iperm[i]);
    if (nblk > 1) {
        load_rows<W, DIAG>(a, Hb, Jb, 1, i, Bv, bo, b);
        rb = rhs_entry(hb, a.iperm[W + i]);
    } else {
#pragma unroll
        for (int w = 0; w < W; ++w) Bv[w] = 0.0;
    }
    auto load_idx = [&](int blk) {
        if (blk < nblk) {
            const int32_t* src = a.src + ((size_t)blk * W) * W + i;
#pragma unroll
            for (int w = 0; w < W; ++w) nidx[w] = src[w * W];
        }
    };
    load_idx(2);
    // Static per-row values of the block two ahead (source row of the right-hand side, diagonal shift, pinned flag) are
    // fetched one block early and consumed without branches: a table load followed by a dependent branch or load inside
    // the block loop was a quarter of the time of a launch too small to hide it (profiles/ncu_kkt_latency_r02.txt)
    const double prim = a.preg != nullptr ? a.preg[bo] : a.primal_reg;   // diagonal shift of this slot's variable rows
    int32_t ipn = -1;
    bool fixn = false;
    auto load_static = [&](int blk) {
        if (blk < nblk) {
            const size_t row = (size_t)blk * W + i;
            ipn = a.iperm[row];
            fixn = a.rowfixed != nullptr && a.rowfixed[row];
        }
    };
    load_static(2);

    // ---------------- factor (right-looking) + forward solve ----------------
    // Step j = blk*W + s. v_r = A(r, j) (un-scaled column), l_r = v_r / d_j. The trailing update
    // A(r, c) -= l_r * v_c is applied to EVERY slot (c mod W) of a row without a lane mask: for c > r
    // that slot holds A(r, c - W), a column < j whose L value has already been published to HBM
    // and is never read from the registers again, and rows outside the band have l_r = 0.
    // Rows of block blk+2 are gathered from J / H into shared memory by cp.async while block blk is
    // being eliminated (their table indices were fetched one block earlier still).
    for (int blk = 0; blk < nblk; ++blk) {
        const bool more = blk + 2 < nblk;
        if (more) {
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const int32_t sx = nidx[w];
                const double* bp = (sx < a.nnz_H) ? Hb : Jb;
                cp_async8_zfill(stage + w * W + i, sx >= 0 ? (const void*)(bp + sx) : (const void*)Hb, sx >= 0 ? 8 : 0);
            }
            cp_async_commit();
            rc = rhs_entry(hb, ipn);
            regc = (fixn || ipn < 0) ? 1.0 : (ipn < a.N_z ? prim : -a.dual_reg);   // = row_shift(): the values of the dreg table
            if (DIAG && !fixn && ipn >= 0) regc += a.diag[b * a.dim + ipn];
            load_idx(blk + 3);
            load_static(blk + 3);
        }
        double* LA = Lg + (size_t)blk * W * LW + i;  // + s*LW + (row - j) with immediates
#pragma unroll
        for (int s = 0; s < G; ++s) {
            const int p = s & (W - 1);
            const bool inA = i > s && i <= s + BW;
            const bool hasB = (s + BW >= G);
            const bool inB = hasB && (i <= s + BW - G);
            const double vA = inA ? A[p] : 0.0;
            const double vB = (hasB && inB) ? Bv[p] : 0.0;
            double* vs = lcol[s & 1];
            // publish the un-scaled column: position q - 1 = row - j - 1
            if (inA) vs[i - s - 1] = vA;
            if (hasB && inB) vs[i + G - s - 1] = vB;
            const double d = shfl_g<G>(A[p], s);
            const double dinv = 1.0 / d;
            const double lA = vA * dinv;
            const double lB = vB * dinv;
            // (row - j) = i - s for set A (0 = the pivot slot), i + G - s for set B
            if (valid && i >= s && i <= s + BW) LA[s * LW - s] = (i == s) ? d : lA;
            if (hasB && inB && valid) LA[s * LW - s + G] = lB;
            __syncwarp();
            // forward substitution, then the D solve for row j
            const double yj = shfl_g<G>(ra, s);
            ra = fma(-lA, yj, ra);
            if (hasB) rb = fma(-lB, yj, rb);
            if (i == s) ra = yj * dinv;
            const double nlA = -lA, nlB = -lB;
#pragma unroll
            for (int q = 1; q <= BW; ++q) {
                const int c = s + q;
                const int idx = (p + q) & (W - 1);
                const double vc = vs[q - 1];
                if (c < G) A[idx] = fma(nlA, vc, A[idx]);
                if (hasB) Bv[idx] = fma(nlB, vc, Bv[idx]);
            }
        }
        if (valid) Yg[(size_t)blk * W + i] = ra;
#pragma unroll
        for (int w = 0; w < W; ++w) A[w] = Bv[w];
        ra = rb;
        if (more) {
            cp_async_wait<0>();
            __syncwarp();
#pragma unroll
            for (int w = 0; w < W; ++w) {
                const double v = stage[w * W + i];
                Bv[w] = (w == i) ? v + regc : v;
            }
            rb = rc;
            __syncwarp();   // the stage is rewritten at the top of the next block
        } else {
#pragma unroll
            for (int w = 0; w < W; ++w) Bv[w] = 0.0;
            rb = 0.0;
        }
    }
    __syncwarp();
    __threadfence_block();

    kkt_backward<W, BW>(a, gsm, Lg, Yg, nblk, i, valid, bo);
}

// ------------------------------------------------------------------------------------------------
// Solve again with the factor of the last factorisation: K unchanged, new right-hand side (a second-order
// correction re-solves with c(z) + c(z + dz), Nocedal & Wright 18.3). The forward substitution reads the stored
// columns of L block by block through the same 3-slot cp.async ring the backward solve uses and applies the
// very operations the factor kernel fuses into its elimination steps (fma(-l, y_j, r); y_j / d_j as y_j * (1/d_j)),
// so the solution is bit-identical to factorising again -- at a fraction of the latency: no trailing update,
// no gather of J and H.
template <int W, int BW>
__global__ void __launch_bounds__(128, (W == 16 ? 4 : 2)) kkt_resolve_kernel(const dto_kkt_args a)
{
    constexpr int G = W;
    using SM = KktSmem<W, BW>;
    constexpr int LW = SM::LW;
    extern __shared__ __align__(16) unsigned char kkt_smem[];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int grp = lane / G, i = lane % G;
    const int64_t b0 = ((int64_t)blockIdx.x * 4 + wib) * SM::NG + grp;
    const bool valid = b0 < a.B;
    const int64_t bs = valid ? b0 : a.B - 1;
    const int64_t b = a.pidx ? (int64_t)a.pidx[bs] : bs;
    const double* hb = a.rhs + b * a.dim;
    const int nblk = a.nblk;
    double* Lg = a.L + (size_t)b * a.factor_stride;
    double* Yg = Lg + (size_t)nblk * W * LW;
    unsigned char* gsm = kkt_smem + (size_t)(wib * SM::NG + grp) * SM::PER_GROUP;
    auto issue = [&](int blk) {
        if (blk < nblk) {
            unsigned char* dst = gsm + (blk % SM::RING) * SM::SLOT;
            const unsigned char* srcL = reinterpret_cast<const unsigned char*>(Lg + (size_t)blk * W * LW);
#pragma unroll
            for (int k = 0; k < LW / 2; ++k) cp_async16(dst + (k * W + i) * 16, srcL + (k * W + i) * 16);
        }
        cp_async_commit();
    };
    issue(0);
    issue(1);
    issue(2);
    double ra = rhs_entry(hb, a.iperm[i]);
    double rb = nblk > 1 ? rhs_entry(hb, a.iperm[W + i]) : 0.0;
    int32_t ipn = nblk > 2 ? a.iperm[2 * W + i] : -1;   // source row of the block two ahead, fetched one block early
    for (int blk = 0; blk < nblk; ++blk) {
        const double rc = blk + 2 < nblk ? rhs_entry(hb, ipn) : 0.0;
        if (blk + 3 < nblk) ipn = a.iperm[(size_t)(blk + 3) * W + i];
        cp_async_wait<2>();
        __syncwarp();
        const double* sl = reinterpret_cast<const double*>(gsm + (blk % SM::RING) * SM::SLOT);
        // y_j / d_j is applied by the lane that owns row j (i == s), to its own value: one reciprocal per lane and block
        // (of the pivot of its own column) instead of one per step -- the same 1 / d_j the factor kernel multiplies by
        const double dinv = 1.0 / sl[i * LW];
#pragma unroll
        for (int s = 0; s < G; ++s) {
            const bool inA = i > s && i <= s + BW;
            const bool hasB = (s + BW >= G);
            const bool inB = hasB && (i <= s + BW - G);
            const double lA = inA ? sl[s * LW + (i - s)] : 0.0;
            const double lB = inB ? sl[s * LW + (i + G - s)] : 0.0;
            const double yj = shfl_g<G>(ra, s);
            ra = fma(-lA, yj, ra);
            if (hasB) rb = fma(-lB, yj, rb);
            if (i == s) ra = yj * dinv;
        }
        if (valid) Yg[(size_t)blk * W + i] = ra;
        ra = rb;
        rb = rc;
        __syncwarp();            // every lane is done with slot blk % RING
        issue(blk + 3);
    }
    cp_async_wait<0>();
    __syncwarp();
    __threadfence_block();
    kkt_backward<W, BW>(a, gsm, Lg, Yg, nblk, i, valid, b);
}

template <int W>
__global__ void kkt_assemble_kernel(const dto_kkt_args a, int64_t problem, double* __restrict__ out)
{
    const int i = threadIdx.x;
    const int blk = blockIdx.x;
    const double* Hb = a.H + problem * a.nnz_H;
    const double* Jb = a.J + problem * a.nnz_J - a.nnz_H;
    double X[W];
    load_rows<W, true>(a, Hb, Jb, blk, i, X, problem);
#pragma unroll
    for (int w = 0; w < W; ++w) out[((size_t)blk * W + w) * W + i] = X[w];
}

// h = [grad f + J' y ; c], natural order. Reference loop (examples/pendulum/pendulum.jl:155-173):
// for each variable i: cy = sum over constraint rows j ascending of C[j,i]*y[j]; h[i] = grad[i] + cy.
__global__ void kkt_rhs_kernel(const dto_kkt_args a)
{
    const int64_t gid0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (gid0 >= a.B * a.dim) return;
    const int64_t slot = gid0 / a.dim;
    const int i = (int)(gid0 - slot * a.dim);
    const int64_t b = a.pidx ? (int64_t)a.pidx[slot] : slot;
    const int64_t gid = b * a.dim + i;
    double h;
    if (i < a.N_z) {
        const double* Jb = a.J + b * a.nnz_J;
        const double* yb = a.y + b * a.N_c;
        double cy = 0.0;
        for (int k = a.colptr[i]; k < a.colptr[i + 1]; ++k)
            cy = __dadd_rn(cy, __dmul_rn(Jb[a.colslot[k]], yb[a.colrow[k]]));
        h = __dadd_rn(a.g[b * a.N_z + i], cy);
        if (a.fixed != nullptr && a.fixed[i]) h = 0.0;   // pinned variable: no step
    } else {
        h = a.c[b * a.N_c + (i - a.N_z)];
    }
    a.rhs[gid] = h;
}

}  // namespace

extern "C" int dto_kkt_launch_rhs(const dto_kkt_args* a, void* stream)
{
    const int64_t n = a->B * a->dim;
    if (n == 0) return 0;
    kkt_rhs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(*a);
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 1 : -(int)e;
}

using kkt_kernel_t = void (*)(dto_kkt_args);

// the factor kernel instantiation for the launch's options
struct BandKernel {
    template <int W, int BW>
    static kkt_kernel_t get(const dto_kkt_args* a)
    {
        if (a->diag) return a->virt ? kkt_band_kernel<W, BW, true, true> : kkt_band_kernel<W, BW, false, true>;
        return a->virt ? kkt_band_kernel<W, BW, true, false> : kkt_band_kernel<W, BW, false, false>;
    }
};
struct ResolveKernel {
    template <int W, int BW>
    static kkt_kernel_t get(const dto_kkt_args*) { return kkt_resolve_kernel<W, BW>; }
};

// one CTA = 4 warps = 4 * 32 / W problems, with the KktSmem<W, BW> layout in dynamic shared memory
template <class Kernel, int W, int BW>
static cudaError_t launch_at(const dto_kkt_args* a, cudaStream_t st)
{
    const kkt_kernel_t kernel = Kernel::template get<W, BW>(a);
    const int64_t per_block = 4 * (32 / W);
    // the opt-in is per device and a batch may span several: set it on every launch (a cheap driver call
    // next to a >= 100 us kernel) instead of caching it per process
    if (KktSmem<W, BW>::BYTES > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, KktSmem<W, BW>::BYTES);
        if (e != cudaSuccess) return e;
    }
    kernel<<<(unsigned)((a->B + per_block - 1) / per_block), 128, KktSmem<W, BW>::BYTES, st>>>(*a);
    return cudaGetLastError();
}

// W and the half bandwidth -> the <W, BW> instantiation; BW must be the bound dto_kkt_bw_bound gives, which also fixes
// the layout of the stored factor, so every bound it returns needs a case here
template <class Kernel>
static int launch_banded(const dto_kkt_args* a, void* stream)
{
    if (a->B == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaErrorInvalidValue;
    const int bound = dto_kkt_bw_bound(a->W, a->bw);
    if (a->W == 16) {
        if (bound == 6) e = launch_at<Kernel, 16, 6>(a, st);
        else if (bound == 9) e = launch_at<Kernel, 16, 9>(a, st);
        else if (bound == 12) e = launch_at<Kernel, 16, 12>(a, st);
        else e = launch_at<Kernel, 16, 15>(a, st);
    } else if (a->W == 32) {
        if (bound == 20) e = launch_at<Kernel, 32, 20>(a, st);
        else e = launch_at<Kernel, 32, 31>(a, st);
    }
    return e == cudaSuccess ? 1 : -(int)e;
}

extern "C" int dto_kkt_launch_band(const dto_kkt_args* a, void* stream) { return launch_banded<BandKernel>(a, stream); }

// forward + backward solve with the factor the last factor kernel launch stored
extern "C" int dto_kkt_launch_resolve(const dto_kkt_args* a, void* stream) { return launch_banded<ResolveKernel>(a, stream); }

extern "C" int dto_kkt_launch_assemble(const dto_kkt_args* a, int64_t problem, double* out, void* stream)
{
    if (a->W == 16)
        kkt_assemble_kernel<16><<<(unsigned)a->nblk, 16, 0, (cudaStream_t)stream>>>(*a, problem, out);
    else if (a->W == 32)
        kkt_assemble_kernel<32><<<(unsigned)a->nblk, 32, 0, (cudaStream_t)stream>>>(*a, problem, out);
    else
        return -(int)cudaErrorInvalidValue;
    const cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? 1 : -(int)e;
}
