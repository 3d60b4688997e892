// Hand-written sm_100a kernels for the batched NLP callbacks. Included by every generated
// model translation unit AFTER the generated `struct DtoModel` (element device functions +
// kind dispatchers), so that the element code inlines into the kernels.
//
// Work decomposition (replaces the reference's serial `for t` loops,
// /root/reference/src/dynamics.jl:103-127, src/costs.jl:49-73, src/constraints.jl:80-104):
//   * one LANE per (problem, knot) item, items numbered flat g = b*T + t so warps stay full
//     even when T is not a multiple of 32 (a warp may straddle two problems);
//   * one WARP is an independent tile of 32 consecutive items (31 + 1 halo item when a
//     dynamics Hessian reaches next-state rows): no __syncthreads anywhere;
//   * every lane writes its element values into the warp's shared-memory segments at the
//     item's flat offset, then the warp streams each segment to HBM with coalesced stores:
//     problem-major outputs J[b][:], H[b][:] are contiguous per (segment, problem) range;
//   * Hessian slots are gathered owner-computes: the warp owns the slots whose ROW belongs to
//     its knots and sums the contributing terms in the reference's += order
//     (cost, dynamics t-1 (as y), dynamics t (as x), stage; /root/reference/src/moi.jl:88-111),
//     so results are deterministic and no atomics / zero-fill are needed.
//   * the GeneralConstraint block (/root/reference/src/general_constraint.jl:73-91) runs as a
//     second tiny kernel on the same stream: J slots assigned, H slots += (it is last in the
//     reference's order too).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <mutex>
#include <type_traits>
#include <vector>

#include "dto_model_abi.h"

#define DTO_WARPS 2          /* warps per CTA of the plain knot kernel */
#define DTO_MIN_CTAS 6       /* resident CTAs per SM asked of __launch_bounds__ (caps registers per thread) */
#define DTO_GATHER_UNROLL 4  /* table-gather records in flight per lane */
#define DTO_PWARPS 12        /* warps per persistent CTA (upper bound; fewer are launched if shared memory is short) */
#define DTO_PCTAS 1          /* persistent CTAs per SM */
#define DTO_KT_SMEM_MAX 384  /* knot-table entries (64 B each) staged in shared memory */
// Kernel selection, set per model library through DTO_TUNE (codegen._tuning); the tests force each alternative
#ifndef DTO_PERSIST
#define DTO_PERSIST 1      /* use the persistent pipeline kernel when the shape allows */
#endif
#ifndef DTO_WS
#define DTO_WS 1           /* use the warp-specialised kernel when the shape allows */
#endif
#ifndef DTO_WS_PLAN
#define DTO_WS_PLAN 1      /* precomputed tile-plan table for the ws kernel (0: helpers compute every tile's records) */
#endif
#ifndef DTO_WS_ALL_MODES
#define DTO_WS_ALL_MODES 0 /* 1: ws kernel also for the gradient / residual / Jacobian-only passes */
#endif
#define DTO_SMEM_LIMIT (227 * 1024)

#define DTO_MODE_G 1
#define DTO_MODE_C 2
#define DTO_MODE_J 4
#define DTO_MODE_H 8

namespace dto {

__device__ __forceinline__ dto_knot_entry load_knot(const dto_knot_entry* __restrict__ tab, int t)
{
    // 64-byte entry = 4 x 16-byte read-only loads
    const int4* p = reinterpret_cast<const int4*>(tab + t);
    int4 a = __ldg(p), b = __ldg(p + 1), c = __ldg(p + 2), d = __ldg(p + 3);
    dto_knot_entry e;
    e.zofs = a.x; e.nx = a.y; e.wofs = a.z; e.kdyn = a.w;
    e.kcost = b.x; e.kstage = b.y; e.rdyn = b.z; e.rstage = b.w;
    e.jdyn = c.x; e.jstage = c.y; e.hterm = c.z; e.hslot = c.w;
    e.hclass = d.x; e.hprev = d.y; e.pad0 = d.z; e.pad1 = d.w;
    return e;
}

// flat item index -> (problem, knot) without an integer divide (magic number from the runtime)
__device__ __forceinline__ void split_item(const dto_launch_args& a, int g, int& b, int& t)
{
    b = (int)(((unsigned long long)(unsigned)g * a.div_mul) >> a.div_shift);
    t = g - b * a.T;
}

__device__ __forceinline__ void warp_stream_out(double* __restrict__ dst, const double* __restrict__ src, int n, int lane)
{
    // dst is 8-byte aligned only (slot ranges start anywhere); one 256-byte row per warp instruction,
    // four rows in flight per trip
    int i = lane;
    for (; i + 96 < n; i += 128) {
        const double v0 = src[i], v1 = src[i + 32], v2 = src[i + 64], v3 = src[i + 96];
        dst[i] = v0;
        dst[i + 32] = v1;
        dst[i + 64] = v2;
        dst[i + 96] = v3;
    }
    for (; i < n; i += 32) dst[i] = src[i];
}

template <int MODE>
__host__ __device__ constexpr bool seg_active(int s)
{
    return (s == DTO_SEG_G && (MODE & DTO_MODE_G)) || ((s == DTO_SEG_CDYN || s == DTO_SEG_CSTAGE) && (MODE & DTO_MODE_C)) ||
           ((s == DTO_SEG_JDYN || s == DTO_SEG_JSTAGE) && (MODE & DTO_MODE_J)) || (s == DTO_SEG_HTERM && (MODE & DTO_MODE_H));
}

template <int MODE>
__host__ __device__ inline int smem_doubles_per_warp(const dto_launch_args& a, int* base)
{
    int per_warp = 0;
    for (int s = 0; s < 6; ++s) {
        if (seg_active<MODE>(s)) {
            if (base) base[s] = per_warp + a.seg_pad[s];
            per_warp += a.seg_pad[s] + a.seg_cap[s];
        } else if (base) {
            base[s] = 0;
        }
    }
    return (per_warp + 1) & ~1;  // keep warps 16-byte aligned
}

// ---------------------------------------------------------------------------------------
// per-knot kernel: gradient / residuals / Jacobian / Hessian / fused Jacobian+Hessian
// ---------------------------------------------------------------------------------------
template <class M, int MODE>
__global__ void __launch_bounds__(DTO_WARPS * 32, DTO_MIN_CTAS) knot_kernel(const __grid_constant__ dto_launch_args a)
{
    extern __shared__ __align__(16) double dto_smem[];
    constexpr bool DO_G = (MODE & DTO_MODE_G) != 0, DO_C = (MODE & DTO_MODE_C) != 0;
    constexpr bool DO_J = (MODE & DTO_MODE_J) != 0, DO_H = (MODE & DTO_MODE_H) != 0;
    constexpr bool HALO = DO_H && (M::HESS_HALO != 0);
    constexpr int OWN = HALO ? 31 : 32;
    // launched with programmatic stream serialization: wait for the previous kernel before touching data, so only the
    // launch latency overlaps (cartpole B=4096 gradient 10.3 -> 9.6 us, constraint 18.7 -> 17.1, Jacobian 24.3 -> 21.7)
    asm volatile("griddepcontrol.launch_dependents;");
    asm volatile("griddepcontrol.wait;" ::: "memory");

    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int T = a.T;
    const int total = (int)(a.B * T);  // the runtime guarantees B*T < 2^31 per shard
    const int g0 = (int)((blockIdx.x * DTO_WARPS + wib) * OWN);  // first OWN item of this warp
    if (g0 >= total) return;
    const int g1 = (g0 + OWN < total) ? g0 + OWN : total;
    int b0, t0;
    split_item(a, g0, b0, t0);

    // L2 prefetch of the inputs of the tile that will start when this one retires (the grid is
    // consumed in order, `tiles_in_flight` warps at a time): its loads then hit L2, not HBM.
    if (a.tiles_in_flight > 0) {
        const long long ga = (long long)g0 + (long long)a.tiles_in_flight * OWN;
        if (ga < total) {
            int ba, ta_;
            split_item(a, (int)ga, ba, ta_);
            const size_t zf = (size_t)ba * a.N_z + (size_t)ta_ * a.z_per_knot;   // approximate start is fine
            const size_t lf = (size_t)ba * a.N_c + (size_t)ta_ * a.c_per_knot;
            const int zl = ((OWN + 1) * a.z_per_knot) / 16 + 2;                   // 128-byte lines of the z range
            const int ll = (OWN * a.c_per_knot) / 16 + 2;
            if (lane < zl) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.z + zf + lane * 16));
            if ((MODE & DTO_MODE_H) && lane < ll) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.lam + lf + lane * 16));
        }
    }

    int base[6];
    const int per_warp = smem_doubles_per_warp<MODE>(a, base);
    double* __restrict__ sm = dto_smem + (size_t)wib * per_warp;

    const dto_knot_entry k0 = load_knot(a.knot, t0);
    const dto_knot_entry kb = load_knot(a.knot, 0);
    const dto_knot_entry kT = load_knot(a.knot, T);
    const int L_g = kT.zofs, L_cd = kT.rdyn - kb.rdyn, L_cs = kT.rstage - kb.rstage;
    const int L_jd = kT.jdyn - kb.jdyn, L_js = kT.jstage - kb.jstage, L_h = kT.hterm;

    // ---- compute phase: one item per lane ----
    {
        const int g = g0 + lane - (HALO ? 1 : 0);
        const bool in = (g < g1) && (g >= g0 || (HALO && t0 > 0));
        if (in) {
            const bool own = g >= g0;
            int b, t;
            split_item(a, g, b, t);
            const int db = b - b0;
            const dto_knot_entry ke = load_knot(a.knot, t);
            const dto_knot_entry kn = load_knot(a.knot, t + 1);
            const double* __restrict__ zb = a.z + (size_t)b * a.N_z;
            const double* __restrict__ x = zb + ke.zofs;
            const double* __restrict__ u = x + ke.nx;
            const double* __restrict__ y = zb + kn.zofs;
            const double* __restrict__ w = a.w + (size_t)b * a.N_w + ke.wofs;
            const double* __restrict__ lam = a.lam + (size_t)b * a.N_c;

            double* hterm = sm + base[DTO_SEG_HTERM] + db * L_h + (ke.hterm - k0.hterm);
            // cost
            if (own) {
                if (DO_G) M::cost_grad(ke.kcost, x, u, w, sm + base[DTO_SEG_G] + db * L_g + (ke.zofs - k0.zofs));
                if (DO_H) M::cost_hess(ke.kcost, x, u, w, __ldg(a.sigma + b), hterm);
            }
            if (DO_H) hterm += M::cost_nh(ke.kcost);
            // dynamics (also evaluated by the halo lane: its y-row Hessian terms feed our first knot)
            if (ke.kdyn >= 0) {
                if (DO_C) M::dyn_res(ke.kdyn, y, x, u, w, sm + base[DTO_SEG_CDYN] + db * L_cd + (ke.rdyn - k0.rdyn));
                double* jd = sm + base[DTO_SEG_JDYN] + db * L_jd + (ke.jdyn - k0.jdyn);
                if (DO_J && DO_H) M::dyn_jac_hess(ke.kdyn, y, x, u, w, lam + ke.rdyn, jd, hterm);
                else if (DO_J) M::dyn_jac(ke.kdyn, y, x, u, w, jd);
                else if (DO_H) M::dyn_hess(ke.kdyn, y, x, u, w, lam + ke.rdyn, hterm);
                if (DO_H) hterm += M::dyn_nh(ke.kdyn);
            }
            // stage constraint
            if (own && ke.kstage >= 0) {
                if (DO_C) M::stage_res(ke.kstage, x, u, w, sm + base[DTO_SEG_CSTAGE] + db * L_cs + (ke.rstage - k0.rstage));
                double* js = sm + base[DTO_SEG_JSTAGE] + db * L_js + (ke.jstage - k0.jstage);
                if (DO_J && DO_H) M::stage_jac_hess(ke.kstage, x, u, w, lam + ke.rstage, js, hterm);
                else if (DO_J) M::stage_jac(ke.kstage, x, u, w, js);
                else if (DO_H) M::stage_hess(ke.kstage, x, u, w, lam + ke.rstage, hterm);
            }
        }
    }
    __syncwarp();

    // ---- compiled Hessian gather (recipes.py): each lane sums the terms of ITS knot's slots with
    // straight-line code (no table loads), then the slot values overwrite the (now dead) term
    // buffer so that the stream-out below is a plain coalesced copy.
    constexpr bool HG = DO_H && (M::HG_NCLASS > 0);
    if (HG && a.use_hclass) {
        double v[M::HG_VMAX > 0 ? M::HG_VMAX : 1];
        const int g = g0 + lane - (HALO ? 1 : 0);
        const bool own = (g < g1) && (g >= g0);
        int cls = -1;
        double* dst = nullptr;
        int b = 0, t = 0;
        if (own) {
            split_item(a, g, b, t);
            const dto_knot_entry ke = load_knot(a.knot, t);
            const double* ownp = sm + base[DTO_SEG_HTERM] + (b - b0) * L_h + (ke.hterm - k0.hterm);
            cls = ke.hclass;
            dst = sm + base[DTO_SEG_HTERM] + (b - b0) * a.nnz_H + (ke.hslot - k0.hslot);
            M::hg_compute(cls, ownp, ownp - ke.hprev, v);
        }
        __syncwarp();
        if (own) M::hg_store(cls, v, dst);
        __syncwarp();
        // general-constraint Hessian entries owned by this lane's knot: last in the reference's +=
        // order (src/moi.jl:112-118), added in shared memory so H is written to HBM exactly once
        if (a.gen_nhess > 0) {
            if (own) {
                const int p0 = __ldg(a.gh_ptr + t), p1 = __ldg(a.gh_ptr + t + 1);
                const int khs = load_knot(a.knot, t).hslot;
                for (int p = p0; p < p1; ++p) {
                    const int2 e = __ldg(reinterpret_cast<const int2*>(a.gh_ent) + p);  // slot, instance
                    const int4 inst = __ldg(reinterpret_cast<const int4*>(a.gen_inst[2]) + e.y);
                    const double val = M::gen_eval(2, inst.x, a.z + (size_t)b * a.N_z + inst.y, a.w + (size_t)b * a.N_w + inst.z,
                                                   a.lam + (size_t)b * a.N_c + a.gen_row0 + inst.w);
                    dst[e.x - khs] += val;
                }
            }
            __syncwarp();
        }
    }

    // ---- stream-out phase: per (problem) sub-tile, coalesced ----
    {
        int b = b0, ta = t0;
        int rem = g1 - g0;
        while (rem > 0) {
            const int cnt = (rem < T - ta) ? rem : (T - ta);
            const int tb = ta + cnt;
            const int db = b - b0;
            const dto_knot_entry ea = load_knot(a.knot, ta);
            const dto_knot_entry eb = load_knot(a.knot, tb);
            if (DO_G)
                warp_stream_out(a.g + (size_t)b * a.N_z + ea.zofs, sm + base[DTO_SEG_G] + db * L_g + (ea.zofs - k0.zofs),
                                eb.zofs - ea.zofs, lane);
            if (DO_C) {
                warp_stream_out(a.c + (size_t)b * a.N_c + ea.rdyn, sm + base[DTO_SEG_CDYN] + db * L_cd + (ea.rdyn - k0.rdyn),
                                eb.rdyn - ea.rdyn, lane);
                warp_stream_out(a.c + (size_t)b * a.N_c + ea.rstage,
                                sm + base[DTO_SEG_CSTAGE] + db * L_cs + (ea.rstage - k0.rstage), eb.rstage - ea.rstage, lane);
            }
            if (DO_J) {
                warp_stream_out(a.J + (size_t)b * a.nnz_J + ea.jdyn, sm + base[DTO_SEG_JDYN] + db * L_jd + (ea.jdyn - k0.jdyn),
                                eb.jdyn - ea.jdyn, lane);
                warp_stream_out(a.J + (size_t)b * a.nnz_J + ea.jstage,
                                sm + base[DTO_SEG_JSTAGE] + db * L_js + (ea.jstage - k0.jstage), eb.jstage - ea.jstage, lane);
            }
            if (HG && a.use_hclass) {
                warp_stream_out(a.H + (size_t)b * a.nnz_H + ea.hslot,
                                sm + base[DTO_SEG_HTERM] + db * a.nnz_H + (ea.hslot - k0.hslot), eb.hslot - ea.hslot, lane);
            } else if (DO_H) {
                const double* __restrict__ smh = sm + base[DTO_SEG_HTERM] + db * L_h - k0.hterm;
                double* __restrict__ Hb = a.H + (size_t)b * a.nnz_H;
                const int4* __restrict__ src4 = reinterpret_cast<const int4*>(a.hsrc4);
                // DTO_GATHER_UNROLL table records per lane are in flight before the first use: the
                // records live in L2 (one 16-byte coalesced load each), so the exposed latency is
                // one L2 round trip per 32*UNROLL slots instead of one per 32 slots.
                int s = ea.hslot + lane;
                for (; s + 32 * (DTO_GATHER_UNROLL - 1) < eb.hslot; s += 32 * DTO_GATHER_UNROLL) {
                    int4 q[DTO_GATHER_UNROLL];
#pragma unroll
                    for (int k = 0; k < DTO_GATHER_UNROLL; ++k) q[k] = __ldg(src4 + s + 32 * k);
#pragma unroll
                    for (int k = 0; k < DTO_GATHER_UNROLL; ++k) {
                        double acc = q[k].x >= 0 ? smh[q[k].x] : 0.0;
                        if (q[k].y >= 0) acc += smh[q[k].y];
                        if (q[k].z >= 0) acc += smh[q[k].z];
                        if (q[k].w >= 0) acc += smh[q[k].w];
                        Hb[s + 32 * k] = acc;
                    }
                }
                for (; s < eb.hslot; s += 32) {
                    const int4 q0 = __ldg(src4 + s);
                    double acc = q0.x >= 0 ? smh[q0.x] : 0.0;
                    if (q0.y >= 0) acc += smh[q0.y];
                    if (q0.z >= 0) acc += smh[q0.z];
                    if (q0.w >= 0) acc += smh[q0.w];
                    Hb[s] = acc;
                }
            }
            rem -= cnt;
            ++b;
            ta = 0;
        }
    }
}

// ---------------------------------------------------------------------------------------
// persistent pipeline variant of the per-knot kernel (the default; knot_kernel above is the
// fallback for shapes it does not cover). Same lane = item / warp = tile decomposition and the
// same arithmetic, but:
//   * one CTA per SM for the whole launch, each warp walks tiles gw, gw+stride, ...;
//   * the knot table is staged in shared memory once per CTA;
//   * a tile's inputs (z, sigma, w: one flat range each; dynamics / stage multipliers: one range
//     per problem touched) are fetched one tile AHEAD by bulk async copies (cp.async.bulk, TMA
//     engine) into a double-buffered per-warp staging area, completion on a per-warp mbarrier:
//     the compute phase reads shared memory only, no HBM latency is exposed;
//   * outputs leave by bulk async stores (shared -> global) issued by one lane per
//     (segment, problem) piece, so the warp starts the next tile while they drain.
// Bulk copies need 16-byte aligned addresses and sizes: every staged range is placed at
// slot + (global_index & 1), i.e. with the parity of its global position, and the copy moves the
// 16-byte aligned hull (inputs) or the aligned body plus at most two single stores (outputs).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(bar), "r"(parity)
                     : "memory");
    } while (!ok);
}
__device__ __forceinline__ void bulk_load(uint32_t dst_smem, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void bulk_store(void* dst, uint32_t src_smem, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src_smem), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// knot entry through a generic pointer (shared-memory copy or the global table)
__device__ __forceinline__ dto_knot_entry ld_knot(const dto_knot_entry* tab, int t)
{
    const int4* p = reinterpret_cast<const int4*>(tab + t);
    const int4 a = p[0], b = p[1], c = p[2], d = p[3];
    dto_knot_entry e;
    e.zofs = a.x; e.nx = a.y; e.wofs = a.z; e.kdyn = a.w;
    e.kcost = b.x; e.kstage = b.y; e.rdyn = b.z; e.rstage = b.w;
    e.jdyn = c.x; e.jstage = c.y; e.hterm = c.z; e.hslot = c.w;
    e.hclass = d.x; e.hprev = d.y; e.pad0 = d.z; e.pad1 = d.w;
    return e;
}

// the prefix-sum field of a knot entry that positions output segment s (HTERM: the slot prefix)
__device__ __forceinline__ int seg_field(const dto_knot_entry& e, int s)
{
    return s == DTO_SEG_G ? e.zofs : s == DTO_SEG_CDYN ? e.rdyn : s == DTO_SEG_CSTAGE ? e.rstage : s == DTO_SEG_JDYN ? e.jdyn
           : s == DTO_SEG_JSTAGE ? e.jstage : e.hslot;
}

// offset (relative to the segment base) of the value `kex` of item (db, b) in the parity-aligned
// piece layout: piece db starts at even_up(flat start) + 2*db + parity of its global start ADDRESS
// (pb = parity of the array base pointer in doubles)
__device__ __forceinline__ int piece_off(int db, int b, int N_s, int pb, int k0x, int kbx, int kTx, int kex)
{
    const int eax = db == 0 ? k0x : kbx;
    const int flat = db == 0 ? 0 : (kTx - k0x) + (db - 1) * (kTx - kbx);
    return ((flat + 1) & ~1) + 2 * db + (((b & N_s) ^ eax ^ pb) & 1) + (kex - eax);
}
__device__ __forceinline__ int ptr_parity(const void* p) { return (int)((reinterpret_cast<uintptr_t>(p) >> 3) & 1); }

struct tile_t {
    int g0, g1, b0, t0, bl, tl, tf, nsub;
};
template <bool HALO>
__device__ __forceinline__ tile_t tile_geom(const dto_launch_args& a, int tile, int total)
{
    constexpr int OWN = HALO ? 31 : 32;
    tile_t q;
    q.g0 = tile * OWN;
    q.g1 = (q.g0 + OWN < total) ? q.g0 + OWN : total;
    split_item(a, q.g0, q.b0, q.t0);
    split_item(a, q.g1 - 1, q.bl, q.tl);
    q.tf = q.t0 - ((HALO && q.t0 > 0) ? 1 : 0);
    q.nsub = q.bl - q.b0 + 1;
    return q;
}
struct item_t {
    int b, t, db;
    bool in, own;
};
template <bool HALO>
__device__ __forceinline__ item_t tile_item(const dto_launch_args& a, const tile_t& q, int lane)
{
    item_t m;
    const int g = q.g0 + lane - (HALO ? 1 : 0);
    m.in = (g < q.g1) && (g >= q.g0 || (HALO && q.t0 > 0));
    m.own = (g < q.g1) && (g >= q.g0);
    m.b = q.b0;
    m.t = q.t0;
    if (m.in) split_item(a, g, m.b, m.t);
    m.db = m.b - q.b0;
    return m;
}
// make the compiler forget what it knows about v: everything derived from it afterwards is recomputed
// instead of being kept live in registers across the FP64 section
__device__ __forceinline__ void forget(int& v) { asm volatile("" : "+r"(v)); }

template <int MODE>
__host__ __device__ inline int p_layout(const dto_launch_args& a, int* base, int* ioff, int* in_sz)
{
    constexpr bool DO_H = (MODE & DTO_MODE_H) != 0;
    int n = 0;
    for (int k = 0; k < 5; ++k) {
        const bool need = (k == DTO_IN_Z) || (k == DTO_IN_W && a.w_flat) || (DO_H && k != DTO_IN_W);
        if (ioff) ioff[k] = n;
        if (need) n += a.in_cap[k];
    }
    if (in_sz) *in_sz = n;
    int off = 2 + 2 * n;  // two mbarriers, two input buffers
    for (int s = 0; s < 6; ++s) {
        if (seg_active<MODE>(s)) {
            const int pad = (a.seg_pad[s] + 1) & ~1;
            if (base) base[s] = off + pad;
            off += pad + ((a.seg_cap[s] + 1) & ~1) + 2 * a.nsub_max + 2;
        } else if (base) {
            base[s] = 0;
        }
    }
    return (off + 1) & ~1;
}

template <class M, int MODE>
__global__ void __launch_bounds__(DTO_PWARPS * 32, DTO_PCTAS) knot_kernel_p(const __grid_constant__ dto_launch_args a)
{
    extern __shared__ __align__(16) double dto_smem[];
    constexpr bool DO_G = (MODE & DTO_MODE_G) != 0, DO_C = (MODE & DTO_MODE_C) != 0;
    constexpr bool DO_J = (MODE & DTO_MODE_J) != 0, DO_H = (MODE & DTO_MODE_H) != 0;
    constexpr bool HALO = DO_H && (M::HESS_HALO != 0);
    constexpr int OWN = HALO ? 31 : 32;
    constexpr bool HG = DO_H && (M::HG_NCLASS > 0);
    // bulk-stored segments, piece order = segment order (at most 3 per instantiated MODE, 8 problems each)
    static_assert((DO_G ? 1 : 0) + (DO_C ? 2 : 0) + (DO_J ? 2 : 0) + (HG ? 1 : 0) <= 4, "piece map needs <= 4 segments per mode");

    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    const int nwarps = blockDim.x >> 5;
    const int T = a.T;
    const int total = (int)(a.B * T);  // the runtime guarantees B*T < 2^31 per shard
    const int tiles = (total + OWN - 1) / OWN;

    const int kt_doubles = a.kt_smem ? (T + 1) * 8 : 0;
    if (a.kt_smem) {
        const int4* src = reinterpret_cast<const int4*>(a.knot);
        int4* dst = reinterpret_cast<int4*>(dto_smem);
        for (int i = threadIdx.x; i < (T + 1) * 4; i += blockDim.x) dst[i] = __ldg(src + i);
    }
    const dto_knot_entry* tab = a.kt_smem ? reinterpret_cast<const dto_knot_entry*>(dto_smem) : a.knot;

    int base[6], ioff[5], in_sz;
    const int per_warp = p_layout<MODE>(a, base, ioff, &in_sz);
    double* __restrict__ sm = dto_smem + kt_doubles + (size_t)wib * per_warp;
    const uint32_t bar0 = smem_u32(sm);
    if (lane == 0) {
        mbar_init(bar0, 1);
        mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    __syncthreads();

    const bool hg_on = HG && a.use_hclass;
    const int gw = blockIdx.x * nwarps + wib;
    const int stride = gridDim.x * nwarps;
    int it = -1;
    int tile = gw - stride;
    while (true) {
        const int nxt = tile + stride;
        const bool have_next = nxt < tiles;
        // ---- producer: bulk-fetch the inputs of tile `nxt` into staging buffer (it+1)&1 ----
        if (have_next) {
            const tile_t q = tile_geom<HALO>(a, nxt, total);
            const dto_knot_entry kT = ld_knot(tab, T);
            double* ib = sm + 2 + ((it + 1) & 1) * in_sz;
            const uint32_t bar = bar0 + ((it + 1) & 1) * 8;
            const dto_knot_entry ktf = ld_knot(tab, q.tf);
            const double* src = nullptr;
            int len = 0, slot = 0;
            if (lane == 0) {
                const dto_knot_entry kl1 = ld_knot(tab, q.tl + 1);
                src = a.z + (size_t)q.b0 * a.N_z + ktf.zofs;
                len = (q.bl - q.b0) * a.N_z + kl1.zofs + (q.tl + 1 < T ? kl1.nx : 0) - ktf.zofs;
                slot = ioff[DTO_IN_Z];
            } else if (lane == 1) {
                if (DO_H) {
                    src = a.sigma + q.b0;
                    len = q.nsub;
                    slot = ioff[DTO_IN_SIGMA];
                }
            } else if (lane == 2) {
                if (a.w_flat) {
                    const dto_knot_entry kl = ld_knot(tab, q.tl);
                    src = a.w + (size_t)q.b0 * a.N_w + ktf.wofs;
                    len = (q.bl - q.b0) * a.N_w + kl.wofs + kl.pad0 - ktf.wofs;
                    slot = ioff[DTO_IN_W];
                }
            } else if (DO_H) {
                const int j = (lane - 3) >> 1, st = (lane - 3) & 1;
                if (j < q.nsub) {
                    const dto_knot_entry ea = ld_knot(tab, j == 0 ? q.tf : 0);
                    const dto_knot_entry eb = ld_knot(tab, j == q.nsub - 1 ? q.tl + 1 : T);
                    const int r0 = st ? ea.rstage : ea.rdyn, r1 = st ? eb.rstage : eb.rdyn;
                    const int rT = st ? kT.rstage : kT.rdyn;
                    const int Ls = st ? kT.rstage - kT.rdyn : kT.rdyn;  // rows per problem: stage rows follow the dynamics rows
                    const int flat = j == 0 ? 0 : (rT - (st ? ktf.rstage : ktf.rdyn)) + (j - 1) * Ls;
                    src = a.lam + (size_t)(q.b0 + j) * a.N_c + r0;
                    len = r1 - r0;
                    slot = ioff[st ? DTO_IN_LSTAGE : DTO_IN_LDYN] + ((flat + 1) & ~1) + 2 * j;
                }
            }
            if (len > 0) {
                const int mis = ptr_parity(src);  // the range lands at slot + mis: same 16-byte phase as in HBM
                const uint32_t bytes = (uint32_t)((len + mis + 1) & ~1) * 8u;
                mbar_expect_tx(bar, bytes);
                bulk_load(smem_u32(ib + slot), src - mis, bytes, bar);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar);
        }

        // ---- consumer: tile `tile` from staging buffer it&1 ----
        if (it >= 0) {
            mbar_wait(bar0 + (it & 1) * 8, (it >> 1) & 1);  // this tile's inputs have landed
            bulk_wait_read();                               // the previous tile's output staging has been read
            __syncwarp();
            {   // -- compute phase: one item per lane; only pointers derived here are live inside it
                const tile_t q = tile_geom<HALO>(a, tile, total);
                const item_t m = tile_item<HALO>(a, q, lane);
                if (m.in) {
                    const dto_knot_entry kb = ld_knot(tab, 0), kT = ld_knot(tab, T);
                    const dto_knot_entry k0 = ld_knot(tab, q.t0), ktf = ld_knot(tab, q.tf), ke = ld_knot(tab, m.t);
                    const double* __restrict__ ib = sm + 2 + (it & 1) * in_sz;
                    const int b = m.b, db = m.db;
                    const int kn_zofs = ld_knot(tab, m.t + 1).zofs;
                    const double* __restrict__ x =
                        ib + ioff[DTO_IN_Z] + (((q.b0 & a.N_z) ^ ktf.zofs ^ ptr_parity(a.z)) & 1) + db * a.N_z + (ke.zofs - ktf.zofs);
                    const double* __restrict__ u = x + ke.nx;
                    const double* __restrict__ y = x + (kn_zofs - ke.zofs);
                    const double* __restrict__ w =
                        a.w_flat ? ib + ioff[DTO_IN_W] + (((q.b0 & a.N_w) ^ ktf.wofs ^ ptr_parity(a.w)) & 1) + db * a.N_w + (ke.wofs - ktf.wofs)
                                 : a.w + (size_t)b * a.N_w + ke.wofs;
                    const double* __restrict__ lam_d = nullptr;
                    const double* __restrict__ lam_s = nullptr;
                    if (DO_H) {
                        const int pl = ptr_parity(a.lam);
                        lam_d = ib + ioff[DTO_IN_LDYN] + piece_off(db, b, a.N_c, pl, ktf.rdyn, kb.rdyn, kT.rdyn, ke.rdyn);
                        lam_s = ib + ioff[DTO_IN_LSTAGE] + piece_off(db, b, a.N_c, pl, ktf.rstage, kb.rstage, kT.rstage, ke.rstage);
                    }
                    double* hterm = sm + base[DTO_SEG_HTERM] + db * kT.hterm + (ke.hterm - k0.hterm);
                    if (m.own) {
                        if (DO_G)
                            M::cost_grad(ke.kcost, x, u, w,
                                         sm + base[DTO_SEG_G] + piece_off(db, b, a.N_z, ptr_parity(a.g), k0.zofs, kb.zofs, kT.zofs, ke.zofs));
                        if (DO_H)
                            M::cost_hess(ke.kcost, x, u, w, ib[ioff[DTO_IN_SIGMA] + ((q.b0 ^ ptr_parity(a.sigma)) & 1) + db], hterm);
                    }
                    if (DO_H) hterm += M::cost_nh(ke.kcost);
                    if (ke.kdyn >= 0) {
                        if (DO_C)
                            M::dyn_res(ke.kdyn, y, x, u, w,
                                       sm + base[DTO_SEG_CDYN] + piece_off(db, b, a.N_c, ptr_parity(a.c), k0.rdyn, kb.rdyn, kT.rdyn, ke.rdyn));
                        double* jd = sm + base[DTO_SEG_JDYN] + piece_off(db, b, a.nnz_J, ptr_parity(a.J), k0.jdyn, kb.jdyn, kT.jdyn, ke.jdyn);
                        if (DO_J && DO_H) M::dyn_jac_hess(ke.kdyn, y, x, u, w, lam_d, jd, hterm);
                        else if (DO_J) M::dyn_jac(ke.kdyn, y, x, u, w, jd);
                        else if (DO_H) M::dyn_hess(ke.kdyn, y, x, u, w, lam_d, hterm);
                        if (DO_H) hterm += M::dyn_nh(ke.kdyn);
                    }
                    if (m.own && ke.kstage >= 0) {
                        if (DO_C)
                            M::stage_res(ke.kstage, x, u, w,
                                         sm + base[DTO_SEG_CSTAGE] +
                                             piece_off(db, b, a.N_c, ptr_parity(a.c), k0.rstage, kb.rstage, kT.rstage, ke.rstage));
                        double* js =
                            sm + base[DTO_SEG_JSTAGE] + piece_off(db, b, a.nnz_J, ptr_parity(a.J), k0.jstage, kb.jstage, kT.jstage, ke.jstage);
                        if (DO_J && DO_H) M::stage_jac_hess(ke.kstage, x, u, w, lam_s, js, hterm);
                        else if (DO_J) M::stage_jac(ke.kstage, x, u, w, js);
                        else if (DO_H) M::stage_hess(ke.kstage, x, u, w, lam_s, hterm);
                    }
                }
            }
            forget(tile);
            __syncwarp();

            // ---- compiled Hessian gather: terms -> slot values, in place, parity-aligned pieces ----
            if (hg_on) {
                const tile_t q = tile_geom<HALO>(a, tile, total);
                const item_t m = tile_item<HALO>(a, q, lane);
                const dto_knot_entry kb = ld_knot(tab, 0), kT = ld_knot(tab, T);
                const dto_knot_entry k0 = ld_knot(tab, q.t0), ke = ld_knot(tab, m.t);
                double v[M::HG_VMAX > 0 ? M::HG_VMAX : 1];
                double* dst = sm + base[DTO_SEG_HTERM] + piece_off(m.db, m.b, a.nnz_H, ptr_parity(a.H), k0.hslot, kb.hslot, kT.hslot, ke.hslot);
                if (m.own) {
                    const double* ownp = sm + base[DTO_SEG_HTERM] + m.db * kT.hterm + (ke.hterm - k0.hterm);
                    M::hg_compute(ke.hclass, ownp, ownp - ke.hprev, v);
                }
                __syncwarp();
                if (m.own) M::hg_store(ke.hclass, v, dst);
                if (a.gen_nhess > 0) {
                    __syncwarp();
                    if (m.own) {
                        const int b = m.b;
                        const int p0 = __ldg(a.gh_ptr + m.t), p1 = __ldg(a.gh_ptr + m.t + 1);
                        for (int p = p0; p < p1; ++p) {
                            const int2 e = __ldg(reinterpret_cast<const int2*>(a.gh_ent) + p);  // slot, instance
                            const int4 inst = __ldg(reinterpret_cast<const int4*>(a.gen_inst[2]) + e.y);
                            const double val = M::gen_eval(2, inst.x, a.z + (size_t)b * a.N_z + inst.y, a.w + (size_t)b * a.N_w + inst.z,
                                                           a.lam + (size_t)b * a.N_c + a.gen_row0 + inst.w);
                            dst[e.x - ke.hslot] += val;
                        }
                    }
                }
            }
            fence_async_smem();  // generic-proxy writes of this lane -> visible to the bulk-store engine
            __syncwarp();

            // ---- stream-out: one lane per (segment, problem) piece: lane = 8*segment + problem ----
            {
                const tile_t q = tile_geom<HALO>(a, tile, total);
                const int si = lane >> 3, j = lane & 7;
                int sg = -1;
                {
                    int c = 0;
#pragma unroll
                    for (int k = 0; k < 6; ++k)
                        if (seg_active<MODE>(k) && (k != DTO_SEG_HTERM || HG)) {
                            if (c == si && (k != DTO_SEG_HTERM || hg_on)) sg = k;
                            ++c;
                        }
                }
                if (sg >= 0 && j < q.nsub) {
                    const dto_knot_entry kb = ld_knot(tab, 0), kT = ld_knot(tab, T), k0 = ld_knot(tab, q.t0);
                    const dto_knot_entry ea = ld_knot(tab, j == 0 ? q.t0 : 0);
                    const dto_knot_entry eb = ld_knot(tab, j == q.nsub - 1 ? q.tl + 1 : T);
                    const int x0 = seg_field(ea, sg);
                    int len = seg_field(eb, sg) - x0;
                    const bool isc = sg == DTO_SEG_CDYN || sg == DTO_SEG_CSTAGE, isj = sg == DTO_SEG_JDYN || sg == DTO_SEG_JSTAGE;
                    const int N_s = sg == DTO_SEG_G ? a.N_z : isc ? a.N_c : isj ? a.nnz_J : a.nnz_H;
                    double* arr = sg == DTO_SEG_G ? a.g : isc ? a.c : isj ? a.J : a.H;
                    double* __restrict__ dst = arr + (size_t)(q.b0 + j) * N_s + x0;
                    const int bs = sg == DTO_SEG_G ? base[0] : sg == DTO_SEG_CDYN ? base[1] : sg == DTO_SEG_CSTAGE ? base[2]
                                   : sg == DTO_SEG_JDYN ? base[3] : sg == DTO_SEG_JSTAGE ? base[4] : base[5];
                    const double* sp =
                        sm + bs + piece_off(j, q.b0 + j, N_s, ptr_parity(arr), seg_field(k0, sg), seg_field(kb, sg), seg_field(kT, sg), x0);
                    if (len > 0) {
                        if (ptr_parity(dst)) {  // odd position: single head store
                            *dst = *sp;
                            ++dst; ++sp; --len;
                        }
                        if (len & 1) {
                            dst[len - 1] = sp[len - 1];
                            --len;
                        }
                        if (len > 0) bulk_store(dst, smem_u32(sp), (uint32_t)len * 8u);
                    }
                }
                bulk_commit();
            }
            // ---- table-driven Hessian gather (shapes without compiled recipes): direct coalesced stores ----
            if (DO_H && !hg_on) {
                const tile_t q = tile_geom<HALO>(a, tile, total);
                const int k0_hterm = ld_knot(tab, q.t0).hterm, L_h = ld_knot(tab, T).hterm;
                int bq = q.b0, ta = q.t0;
                int rem = q.g1 - q.g0;
                while (rem > 0) {
                    const int cnt = (rem < T - ta) ? rem : (T - ta);
                    const dto_knot_entry ea = ld_knot(tab, ta);
                    const dto_knot_entry eb = ld_knot(tab, ta + cnt);
                    const double* __restrict__ smh = sm + base[DTO_SEG_HTERM] + (bq - q.b0) * L_h - k0_hterm;
                    double* __restrict__ Hb = a.H + (size_t)bq * a.nnz_H;
                    const int4* __restrict__ src4 = reinterpret_cast<const int4*>(a.hsrc4);
                    for (int s = ea.hslot + lane; s < eb.hslot; s += 32) {
                        const int4 q0 = __ldg(src4 + s);
                        double acc = q0.x >= 0 ? smh[q0.x] : 0.0;
                        if (q0.y >= 0) acc += smh[q0.y];
                        if (q0.z >= 0) acc += smh[q0.z];
                        if (q0.w >= 0) acc += smh[q0.w];
                        Hb[s] = acc;
                    }
                    rem -= cnt;
                    ++bq;
                    ta = 0;
                }
                __syncwarp();
            }
        }
        if (!have_next) break;
        tile = nxt;
        ++it;
    }
    bulk_wait_all();
}

#include "dto_kernel_ws.cuh"

// ---------------------------------------------------------------------------------------
// objective value: one warp per problem. The per-knot costs of 32 consecutive knots are evaluated in
// parallel (lane = knot), then added to the running sum ONE BY ONE in knot order -- the reference's serial
// `J += cost_t` (/root/reference/src/costs.jl:49-56), so the rounding of the sum is the reference's too
// (a shuffle tree would be ~T/32 times shorter but sums in another order).
// ---------------------------------------------------------------------------------------
template <class M>
__global__ void __launch_bounds__(DTO_WARPS * 32) objective_kernel(const __grid_constant__ dto_launch_args a)
{
    const int lane = threadIdx.x & 31;
    const long long b = (long long)blockIdx.x * DTO_WARPS + (threadIdx.x >> 5);
    if (b >= a.B) return;
    const double* __restrict__ zb = a.z + (size_t)b * a.N_z;
    double acc = 0.0;
    for (int t0 = 0; t0 < a.T; t0 += 32) {
        const int t = t0 + lane;
        double v = 0.0;
        if (t < a.T) {
            const dto_knot_entry ke = load_knot(a.knot, t);
            const double* x = zb + ke.zofs;
            v = M::cost_val(ke.kcost, x, x + ke.nx, a.w + (size_t)b * a.N_w + ke.wofs);
        }
        const int n = min(32, a.T - t0);  // warp-uniform
        for (int k = 0; k < n; ++k) acc = __dadd_rn(acc, __shfl_sync(0xffffffffu, v, k));
    }
    if (lane == 0) a.f[b] = acc;
}

// ---------------------------------------------------------------------------------------
// general constraint: one thread per (problem, output instance)
// ---------------------------------------------------------------------------------------
template <class M, int CLS>
__global__ void __launch_bounds__(128) general_kernel(const __grid_constant__ dto_launch_args a)
{
    const int n = (CLS == 0) ? a.gen_nrow : (CLS == 1) ? a.gen_njac : a.gen_nhess;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= a.B * (long long)n) return;
    const long long b = idx / n;
    const int i = (int)(idx - b * n);
    const int4 inst = __ldg(reinterpret_cast<const int4*>(a.gen_inst[CLS]) + i);  // tmpl, zbase, wbase, lbase
    const double* __restrict__ z = a.z + (size_t)b * a.N_z + inst.y;
    const double* __restrict__ w = a.w + (size_t)b * a.N_w + inst.z;
    if (CLS == 0) {
        a.c[(size_t)b * a.N_c + a.gen_row0 + i] = M::gen_eval(0, inst.x, z, w, nullptr);
    } else if (CLS == 1) {
        a.J[(size_t)b * a.nnz_J + a.gen_jac0 + i] = M::gen_eval(1, inst.x, z, w, nullptr);
    } else {
        const double* __restrict__ lam = a.lam + (size_t)b * a.N_c + a.gen_row0 + inst.w;
        double* h = a.H + (size_t)b * a.nnz_H + __ldg(a.gen_hslot + i);
        *h += M::gen_eval(2, inst.x, z, w, lam);  // general is last in the reference's += order
    }
}

// ---------------------------------------------------------------------------------------
// host side of the model library
// ---------------------------------------------------------------------------------------
template <int MODE>
inline int64_t knot_smem_bytes(const dto_launch_args& a)
{
    return (int64_t)smem_doubles_per_warp<MODE>(a, nullptr) * DTO_WARPS * (int64_t)sizeof(double);
}

// persistent kernel launch plan: warps per CTA and shared memory, or warps = 0 if the shape is not covered
template <int MODE>
inline int plan_persistent(dto_launch_args& b, int64_t* smem_out, int min_ops_ok = 1)
{
    if (!DTO_PERSIST || !b.persist_ok || min_ops_ok == 0) return 0;
    const int64_t per_warp = (int64_t)p_layout<MODE>(b, nullptr, nullptr, nullptr) * (int64_t)sizeof(double);
    for (int kt = 1; kt >= 0; --kt) {
        if (kt && b.T + 1 > DTO_KT_SMEM_MAX) continue;
        const int64_t ktb = kt ? (int64_t)(b.T + 1) * 64 : 0;
        int64_t nw = (DTO_SMEM_LIMIT / DTO_PCTAS - 1024 - ktb) / per_warp;
        if (nw > DTO_PWARPS) nw = DTO_PWARPS;
        if (nw >= 4 || (kt == 0 && nw >= 2)) {
            b.kt_smem = kt;
            *smem_out = ktb + nw * per_warp;
            return (int)nw;
        }
    }
    return 0;
}

// launch with programmatic stream serialization: the kernel may be scheduled while the previous kernel of the stream
// drains. A kernel launched here may read, before griddepcontrol.wait, anything that no kernel launched here writes.
// It must execute the wait before its first global write.
// The kernels launched here (knot_kernel, knot_kernel_ws) write only g, c, J and H. z, lambda, sigma, w, the knot
// table and the plan table are written only by copies and by kernels that do not execute launch_dependents, so such
// a writer has completed before any later kernel launched here starts, also along a chain of launches made here.
// knot_kernel waits at its top; knot_kernel_ws reads and computes first and waits before its first store.
template <class K>
inline cudaError_t launch_pdl(K kernel, unsigned grid, unsigned block, size_t smem, cudaStream_t st, const dto_launch_args& args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // not while the stream is being captured into a CUDA graph: programmatic edges made the replay of the solver's
    // line-search graph 2x slower (3.5 vs 1.5 s for config 3); a captured launch is an ordinary kernel node
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) {
        cudaGetLastError();
        cap = cudaStreamCaptureStatusNone;
    }
    if (cap != cudaStreamCaptureStatusNone) cfg.numAttrs = 0;
    return cudaLaunchKernelEx(&cfg, kernel, args);
}

template <class M, int MODE>
inline int launch_knot(const dto_launch_args& a, cudaStream_t st)
{
    constexpr bool HALO = ((MODE & DTO_MODE_H) != 0) && (M::HESS_HALO != 0);
    const long long own = HALO ? 31 : 32;
    const long long total = a.B * (long long)a.T;
    if (total == 0) return 0;
    const long long warps = (total + own - 1) / own;
    dto_launch_args b = a;
    b.tiles_in_flight = 0;
    {
        const int64_t wsmem = plan_ws<M, MODE>(b);
        if (wsmem > 0) {
            static int sms[16] = {0};
            static int64_t attr_smem[16] = {0};
            int dev = 0;
            cudaGetDevice(&dev);
            dev = (dev >= 0 && dev < 16) ? dev : 0;
            if (sms[dev] == 0) cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
            if (wsmem > attr_smem[dev]) {
                cudaError_t e = cudaFuncSetAttribute(knot_kernel_ws<M, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem);
                if (e != cudaSuccess) {
                    fprintf(stderr, "[dto] cudaFuncSetAttribute(ws mode %d, smem %lld) failed: %s\n", MODE, (long long)wsmem, cudaGetErrorString(e));
                    return (int)e;
                }
                attr_smem[dev] = wsmem;
            }
            long long ctas = (warps + DTO_WS_COMPUTE - 1) / DTO_WS_COMPUTE;
            if (ctas > sms[dev]) ctas = sms[dev];
            b.ws_plan = ws_get_plan<M, MODE>(b, st);
            cudaError_t e = launch_pdl(knot_kernel_ws<M, MODE>, (unsigned)ctas, (DTO_WS_COMPUTE + DTO_WS_HELPERS) * 32, (size_t)wsmem, st, b);
            if (e != cudaSuccess)
                fprintf(stderr, "[dto] knot_kernel_ws<mode %d> launch failed: %s (grid %lld, smem %lld)\n", MODE, cudaGetErrorString(e), ctas,
                        (long long)wsmem);
            return (int)e;
        }
    }
    {
        int64_t psmem = 0;
        const int nw = plan_persistent<MODE>(b, &psmem, (MODE & DTO_MODE_H) != 0 && M::OPS_FUSED >= 100);  // persistent fallback: FP64-heavy models only
        if (nw > 0) {
            static int sms[16] = {0};
            static int64_t attr_smem[16] = {0};
            int dev = 0;
            cudaGetDevice(&dev);
            dev = (dev >= 0 && dev < 16) ? dev : 0;
            if (sms[dev] == 0) cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
            if (psmem > attr_smem[dev]) {
                cudaError_t e = cudaFuncSetAttribute(knot_kernel_p<M, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psmem);
                if (e != cudaSuccess) {
                    fprintf(stderr, "[dto] cudaFuncSetAttribute(persistent mode %d, smem %lld) failed: %s\n", MODE, (long long)psmem,
                            cudaGetErrorString(e));
                    return (int)e;
                }
                attr_smem[dev] = psmem;
            }
            long long ctas = (warps + nw - 1) / nw;
            if (ctas > (long long)sms[dev] * DTO_PCTAS) ctas = (long long)sms[dev] * DTO_PCTAS;
            knot_kernel_p<M, MODE><<<(unsigned)ctas, nw * 32, (size_t)psmem, st>>>(b);
            cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess)
                fprintf(stderr, "[dto] knot_kernel_p<mode %d> launch failed: %s (grid %lld, block %d, smem %lld)\n", MODE,
                        cudaGetErrorString(e), ctas, nw * 32, (long long)psmem);
            return (int)e;
        }
    }
    const long long ctas = (warps + DTO_WARPS - 1) / DTO_WARPS;
    const int64_t smem = knot_smem_bytes<MODE>(a);
    if (smem > 48 * 1024) {  // opt in to large dynamic shared memory (per device, cheap)
        cudaError_t e = cudaFuncSetAttribute(knot_kernel<M, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            fprintf(stderr, "[dto] cudaFuncSetAttribute(mode %d, smem %lld) failed: %s\n", MODE, (long long)smem, cudaGetErrorString(e));
            return (int)e;
        }
    }
    {
        static int resident_warps[16] = {0};  // per device, for the shared-memory size it was computed with
        static int64_t resident_smem[16] = {0};
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 16) {
            if (resident_warps[dev] == 0 || resident_smem[dev] != smem) {
                resident_smem[dev] = smem;
                int sms = 0, per_sm = 0;
                cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
                if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, knot_kernel<M, MODE>, DTO_WARPS * 32, (size_t)smem) != cudaSuccess)
                    per_sm = 0;
                resident_warps[dev] = sms * per_sm * DTO_WARPS;
                cudaGetLastError();
            }
            b.tiles_in_flight = resident_warps[dev];
        }
    }
    cudaError_t e = launch_pdl(knot_kernel<M, MODE>, (unsigned)ctas, DTO_WARPS * 32, (size_t)smem, st, b);
    if (e != cudaSuccess)
        fprintf(stderr, "[dto] knot_kernel<mode %d> launch failed: %s (grid %lld, block %d, smem %lld)\n", MODE, cudaGetErrorString(e),
                ctas, DTO_WARPS * 32, (long long)smem);
    return (int)e;
}

template <class M, int CLS>
inline int launch_general(const dto_launch_args& a, cudaStream_t st)
{
    const int n = (CLS == 0) ? a.gen_nrow : (CLS == 1) ? a.gen_njac : a.gen_nhess;
    const long long total = a.B * (long long)n;
    if (total == 0) return 0;
    general_kernel<M, CLS><<<(unsigned)((total + 127) / 128), 128, 0, st>>>(a);
    return (int)cudaGetLastError();
}

// Enqueue the kernels of one callback. Returns the number of kernels launched (>= 0) or minus the
// cudaError_t of the first failure.
template <class M>
inline int launch(int kernel_id, const dto_launch_args* pa, void* stream)
{
    const dto_launch_args& a = *pa;
    cudaStream_t st = (cudaStream_t)stream;
    int e = 0, n = 0;
    auto general = [&](auto cls, int count) -> int {  // companion kernel over the general-constraint block
        if (count <= 0 || a.B == 0) return 0;
        if ((e = launch_general<M, decltype(cls)::value>(a, st))) return -e;
        ++n;
        return 0;
    };
    using C0 = std::integral_constant<int, 0>;
    using C1 = std::integral_constant<int, 1>;
    using C2 = std::integral_constant<int, 2>;
    if (a.B == 0) return 0;
    switch (kernel_id) {
    case DTO_K_OBJECTIVE:
        // (no programmatic launch here: measured slower for this kernel of many tiny CTAs, 10.3 -> 12.7 us)
        objective_kernel<M><<<(unsigned)((a.B + DTO_WARPS - 1) / DTO_WARPS), DTO_WARPS * 32, 0, st>>>(a);
        e = (int)cudaGetLastError();
        return e ? -e : 1;
    case DTO_K_GRADIENT:
        e = launch_knot<M, DTO_MODE_G>(a, st);
        return e ? -e : 1;
    case DTO_K_CONSTRAINT:
        if ((e = launch_knot<M, DTO_MODE_C>(a, st))) return -e;
        ++n;
        if (general(C0{}, a.gen_nrow)) return -e;
        return n;
    case DTO_K_JACOBIAN:
        if ((e = launch_knot<M, DTO_MODE_J>(a, st))) return -e;
        ++n;
        if (general(C1{}, a.gen_njac)) return -e;
        return n;
    case DTO_K_HESSIAN:
    case DTO_K_JAC_HESS: {
        if (kernel_id == DTO_K_HESSIAN) e = launch_knot<M, DTO_MODE_H>(a, st);
        else e = launch_knot<M, DTO_MODE_J | DTO_MODE_H>(a, st);
        if (e) return -e;
        ++n;
        if (kernel_id == DTO_K_JAC_HESS && general(C1{}, a.gen_njac)) return -e;
        // general-constraint Hessian: fused into the knot kernel when the compiled gather is in use
        const bool fused = M::HG_NCLASS > 0 && a.use_hclass;
        if (!fused && general(C2{}, a.gen_nhess)) return -e;
        return n;
    }
    default:
        return -(int)cudaErrorInvalidValue;
    }
}

template <class M, int MODE>
inline int64_t mode_smem_bytes(const dto_launch_args& a)
{
    dto_launch_args b = a;
    const int64_t ws = plan_ws<M, MODE>(b);
    if (ws > 0) return ws;
    int64_t ps = 0;
    if (plan_persistent<MODE>(b, &ps, (MODE & DTO_MODE_H) != 0 && M::OPS_FUSED >= 100) > 0) return ps;
    return knot_smem_bytes<MODE>(a);
}

// dynamic shared memory of the kernel that launch<M>() would pick for kernel_id
template <class M>
inline int64_t smem_bytes(int kernel_id, const dto_launch_args* pa)
{
    switch (kernel_id) {
    case DTO_K_GRADIENT: return mode_smem_bytes<M, DTO_MODE_G>(*pa);
    case DTO_K_CONSTRAINT: return mode_smem_bytes<M, DTO_MODE_C>(*pa);
    case DTO_K_JACOBIAN: return mode_smem_bytes<M, DTO_MODE_J>(*pa);
    case DTO_K_HESSIAN: return mode_smem_bytes<M, DTO_MODE_H>(*pa);
    case DTO_K_JAC_HESS: return mode_smem_bytes<M, DTO_MODE_J | DTO_MODE_H>(*pa);
    default: return 0;
    }
}

}  // namespace dto
