// Warp-specialised per-knot kernel (the default for the Hessian passes of FP64-heavy models).
// Included by dto_kernels.cuh inside namespace dto, after the shared helpers.
//
// One CTA of 12 warps per SM for the whole launch:
//   * warps 0-3 ("helpers", DTO_WS_HREG registers after setmaxnreg.dec) move data: per tile they
//     bulk-copy (cp.async.bulk, completion on the stage's mbarrier) the tile's inputs and the tile's
//     PLAN RECORDS into a shared-memory stage, and later stream the finished tile out with bulk stores;
//   * warps 4-11 ("compute", DTO_WS_CREG registers after setmaxnreg.inc: no spills, room for ILP)
//     wait on the stage's mbarrier, load their item descriptor (3 x LDS.128), run the generated FP64
//     code of /root/reference/src/dynamics.jl:103-127, src/costs.jl:58-73, src/constraints.jl:80-104
//     with the Hessian terms in registers and sum the Hessian slots in the reference's += order
//     (src/moi.jl:88-118) into the output staging.
// Helper h serves compute warps h and h+4 (all three live on SM sub-partition h, whose 512 registers
// per lane are split DTO_WS_HREG + 2 x DTO_WS_CREG). Per compute warp: two input stages (mbarrier
// full[2]) and one or two output staging buffers (mbarriers out_full / out_empty). Round kk of a
// helper, per served compute warp: wait out_full(kk-2) -> issue that tile's bulk stores -> produce
// tile kk into the input stage tile kk-2 just vacated -> wait for the stores' shared-memory reads ->
// arrive out_empty.
//
// TILE PLANS. Everything integer about a full 32-item tile -- where each item's inputs and output
// slots sit in the stage / staging buffers, which ranges to copy in and out and how they are aligned
// -- depends only on the tile's first knot t0 and on the parity of its first problem b0 (16-byte
// alignment of the 8-byte-granular ranges). A one-off kernel (plan_kernel) computes these records for
// all (t0, b0 & 1) into a table in HBM (L2-resident afterwards); the helpers then copy one 2 KB block
// per tile instead of recomputing ~500 integer instructions. The ragged last tile of a launch takes
// the slow path, which computes the same records in place.
#pragma once

#define DTO_WS_COMPUTE 8          /* compute warps per CTA (2 per SM sub-partition) */
#ifndef DTO_WS_HELPERS
#define DTO_WS_HELPERS 8          /* helper h serves compute warps h, h + HELPERS, ...: COMPUTE must be a multiple (DTO_TUNE ws_helpers) */
#endif
#define DTO_WS_HREG 40            /* registers per helper-warp thread after setmaxnreg.dec */
/* registers per thread the launch allocates: 64 K registers per SM over the CTA's threads ROUNDED UP TO 128 (ptxas
 * sizes the pool per group of four warps: 18 warps get 65536/640 = 96, not 112), multiple of 8 */
#define DTO_WS_WARPS (DTO_WS_COMPUTE + DTO_WS_HELPERS)
#define DTO_WS_BASE_REGS ((65536 / (128 * ((DTO_WS_WARPS + 3) / 4))) > 255 ? 248 : ((65536 / (128 * ((DTO_WS_WARPS + 3) / 4))) & ~7))
/* registers per compute-warp thread after setmaxnreg.inc: what the helpers leave of the launch's registers, at most 232
 * (8 helpers: 216; 4 helpers: 232) */
#define DTO_WS_CREG_LEFT ((((DTO_WS_WARPS * DTO_WS_BASE_REGS) - DTO_WS_HELPERS * DTO_WS_HREG) / DTO_WS_COMPUTE) & ~7)
#define DTO_WS_CREG (DTO_WS_CREG_LEFT < 232 ? DTO_WS_CREG_LEFT : 232)
#define DTO_WS_DESC_DOUBLES 192   /* 3 x int4 per item, 32 items */
#define DTO_WS_PIECE_DOUBLES 64   /* 1 x int4 per piece, 32 pieces */
#define DTO_WS_HDR_DOUBLES 2      /* 1 x int4: b0, ... */
#define DTO_WS_PLAN_INT4 160      /* per (t0, parity): copy[32], d0[32], d1[32], d2[32], piece[32] (+ general records) */
#define DTO_WS_GEN_K 2            /* general-constraint Hessian entries per knot carried as plan records */
#define DTO_WS_GEN_LCAP 32        /* general-constraint multipliers staged per problem of a tile (doubles, even) */
#define DTO_WS_GEN_INT4 (32 * DTO_WS_GEN_K + 8)  /* records[32][K] + count[32] */

// shapes with a general-constraint Hessian carry DTO_WS_GEN_INT4 more int4 per plan block / stage
template <int MODE>
__host__ __device__ inline int ws_gen_int4(const dto_launch_args& a)
{
    return ((MODE & DTO_MODE_H) != 0 && a.gen_nhess > 0) ? DTO_WS_GEN_INT4 : 0;
}

template <int MODE>
__host__ __device__ inline int ws_layout(const dto_launch_args& a, int* base, int* ioff, int* in_sz, int* stage_sz, int* out0, int* out_sz,
                                         int* gl_off = nullptr)
{
    constexpr bool DO_H = (MODE & DTO_MODE_H) != 0;
    int n = 0;
    for (int k = 0; k < 5; ++k) {
        const bool need = (k == DTO_IN_Z) || (k == DTO_IN_W && a.w_flat) || (DO_H && k != DTO_IN_W);
        if (ioff) ioff[k] = n;
        if (need) n += a.in_cap[k];
    }
    // general-constraint multipliers the tile's Hessian entries read: one staged range per problem touched
    if (gl_off) *gl_off = n;
    if (ws_gen_int4<MODE>(a)) n += 4 * (DTO_WS_GEN_LCAP + 2);
    if (in_sz) *in_sz = n;
    const int st = n + DTO_WS_DESC_DOUBLES + DTO_WS_PIECE_DOUBLES + 2 * ws_gen_int4<MODE>(a) + DTO_WS_HDR_DOUBLES;
    if (stage_sz) *stage_sz = st;
    int off = 8 + 2 * st;  // six mbarriers (8 doubles reserved), two input stages
    const int out_begin = off;
    if (out0) *out0 = off;
    for (int s = 0; s < 6; ++s) {
        if (seg_active<MODE>(s)) {
            // Hessian terms stay in registers here: the HTERM segment stages slot values only
            const int pad = s == DTO_SEG_HTERM ? 0 : (a.seg_pad[s] + 1) & ~1;
            const int cap = s == DTO_SEG_HTERM ? a.hslot_cap : a.seg_cap[s];
            if (base) base[s] = off + pad;
            off += pad + ((cap + 1) & ~1) + 2 * a.nsub_max + 2;
        } else if (base) {
            base[s] = 0;
        }
    }
    off = (off + 1) & ~1;
    if (out_sz) *out_sz = off - out_begin;
    return off;  // size with ONE output buffer; a second one adds *out_sz
}

// geometry of the tile whose first own item is g0 (flat item index) with `n` own items
template <bool HALO>
__device__ __forceinline__ tile_t tile_geom_at(const dto_launch_args& a, int g0, int n)
{
    tile_t q;
    q.g0 = g0;
    q.g1 = g0 + n;
    split_item(a, q.g0, q.b0, q.t0);
    split_item(a, q.g1 - 1, q.bl, q.tl);
    q.tf = q.t0 - ((HALO && q.t0 > 0) ? 1 : 0);
    q.nsub = q.bl - q.b0 + 1;
    return q;
}

// array ids of the records: inputs 0 z, 1 sigma, 2 w, 3 lambda; outputs 0 g, 1 c, 2 J, 3 H
__device__ __forceinline__ const double* ws_in_array(const dto_launch_args& a, int id, int b0)
{
    return id == 0 ? a.z + (size_t)b0 * a.N_z : id == 1 ? a.sigma + b0 : id == 2 ? a.w + (size_t)b0 * a.N_w : a.lam + (size_t)b0 * a.N_c;
}
__device__ __forceinline__ double* ws_out_array(const dto_launch_args& a, int id, int b0)
{
    return id == 0 ? a.g + (size_t)b0 * a.N_z : id == 1 ? a.c + (size_t)b0 * a.N_c : id == 2 ? a.J + (size_t)b0 * a.nnz_J : a.H + (size_t)b0 * a.nnz_H;
}

// The five records of lane `lane` for tile q, all offsets for input stage 0 / output buffer 0
// (sbase0 = offset of stage 0 in the region; the consumer adds st*stage_sz / o*out_sz):
//   copy  = {src offset (doubles, from the array's row of problem b0, 16-byte aligned address), bytes, stage offset, input array id}
//   piece = {dst offset (doubles, from the array's row of problem b0), output array id, staging offset, length in doubles}
//   d0,d1,d2 = the item descriptor of the lane's (problem, knot) item (packed 16-bit region offsets)
// lane = 4*row + j addresses the (segment row, problem) ranges: rows 0..5 the output segments (G, CDYN,
// CSTAGE, JDYN, JSTAGE, Hessian slots), rows 6,7 the dynamics / stage multipliers; lanes 0..2 also
// carry the flat z / sigma / w input ranges (their rows 0 are outputs, so the copy slot is free).
template <class M, int MODE>
__device__ __forceinline__ void ws_tile_records(const dto_launch_args& a, const dto_knot_entry* tab, const tile_t& q, int lane, const int* base,
                                                const int* ioff, int sbase0, int4& copy, int4& piece, int4& d0, int4& d1, int4& d2)
{
    constexpr bool DO_G = (MODE & DTO_MODE_G) != 0, DO_C = (MODE & DTO_MODE_C) != 0;
    constexpr bool DO_J = (MODE & DTO_MODE_J) != 0, DO_H = (MODE & DTO_MODE_H) != 0;
    constexpr bool HALO = DO_H && (M::HESS_HALO != 0);
    constexpr bool HG = DO_H && (M::HG_NCLASS > 0);
    const int T = a.T;
    const int* tabw = reinterpret_cast<const int*>(tab);  // knot entry = 16 words
    const int tfz = tabw[q.tf * 16 + 0], tfw = tabw[q.tf * 16 + 2];
    copy = make_int4(0, 0, 0, 0);
    piece = make_int4(0, 0, 0, 0);
    // ---- flat input ranges z / sigma / w: lanes 0..2 ----
    {
        const double* src = nullptr;
        int len = 0, slot = 0, rel = 0, id = 0;
        if (lane == 0) {
            const int e1z = tabw[(q.tl + 1) * 16 + 0], e1n = tabw[(q.tl + 1) * 16 + 1];
            src = a.z + (size_t)q.b0 * a.N_z + tfz;
            rel = tfz;
            len = (q.bl - q.b0) * a.N_z + e1z + (q.tl + 1 < T ? e1n : 0) - tfz;
            slot = ioff[DTO_IN_Z];
            id = 0;
        } else if (lane == 1) {
            if (DO_H) {
                src = a.sigma + q.b0;
                rel = 0;
                len = q.nsub;
                slot = ioff[DTO_IN_SIGMA];
                id = 1;
            }
        } else if (lane == 2) {
            if (a.w_flat) {
                src = a.w + (size_t)q.b0 * a.N_w + tfw;
                rel = tfw;
                len = (q.bl - q.b0) * a.N_w + tabw[q.tl * 16 + 2] + tabw[q.tl * 16 + 14] - tfw;
                slot = ioff[DTO_IN_W];
                id = 2;
            }
        }
        if (len > 0) {
            const int mis = ptr_parity(src);  // the range lands at slot + mis: same 16-byte phase as in HBM
            copy = make_int4(rel - mis, ((len + mis + 1) & ~1) * 8, sbase0 + slot, id);
        }
    }
    // ---- (segment row, problem) ranges: lane = 4*row + j. cst = start - (prefix field of the range's
    // first knot), so an item of that range sits at cst + (its own prefix field).
    int cst = 0;
    {
        const int row = lane >> 2, j = lane & 3;
        const bool is_in = row >= 6;
        const bool active = is_in ? DO_H : (seg_active<MODE>(row) && (row != DTO_SEG_HTERM || HG));
        if (active && j < q.nsub) {
            const int wi = (0x76B98760u >> (4 * row)) & 15;  // word of the row's prefix field in a knot entry
            const int tfirst = is_in ? q.tf : q.t0;
            const int kfx = tabw[tfirst * 16 + wi], kTx = tabw[T * 16 + wi], kbx = tabw[wi];
            const int ea = j == 0 ? kfx : kbx;
            const int eb = tabw[(j == q.nsub - 1 ? q.tl + 1 : T) * 16 + wi];
            const int len = eb - ea;
            const bool isc = row == 1 || row == 2 || is_in, isj = row == 3 || row == 4;
            const int N_s = row == 0 ? a.N_z : isc ? a.N_c : isj ? a.nnz_J : a.nnz_H;
            const double* arr = row == 0 ? a.g : is_in ? a.lam : isc ? a.c : isj ? a.J : a.H;
            const int par = ptr_parity(arr + (size_t)(q.b0 + j) * N_s + ea);
            const int flat = j == 0 ? 0 : (kTx - kfx) + (j - 1) * (kTx - kbx);
            const int sb = row == 0 ? base[0] : row == 1 ? base[1] : row == 2 ? base[2] : row == 3 ? base[3] : row == 4 ? base[4]
                           : row == 5 ? base[5] : row == 6 ? sbase0 + ioff[DTO_IN_LDYN] : sbase0 + ioff[DTO_IN_LSTAGE];
            const int start = sb + ((flat + 1) & ~1) + 2 * j + par;
            cst = start - ea;
            if (is_in) {
                if (len > 0) copy = make_int4(j * N_s + ea - par, ((len + par + 1) & ~1) * 8, start - par, 3);
            } else {
                piece = make_int4(j * N_s + ea, row == 0 ? 0 : isc ? 1 : isj ? 2 : 3, start, len);
            }
        }
    }
    // ---- item descriptor ----
    {
        const item_t m = tile_item<HALO>(a, q, lane);
        const dto_knot_entry ke = ld_knot(tab, m.t);
        const int kn_zofs = tabw[(m.t + 1) * 16];
        const int db = m.db;
        const int x_off = sbase0 + ioff[DTO_IN_Z] + (((q.b0 & a.N_z) ^ tfz ^ ptr_parity(a.z)) & 1) + db * a.N_z + (ke.zofs - tfz);
        const int y_off = x_off + (kn_zofs - ke.zofs);
        const int w_off = a.w_flat ? sbase0 + ioff[DTO_IN_W] + (((q.b0 & a.N_w) ^ tfw ^ ptr_parity(a.w)) & 1) + db * a.N_w + (ke.wofs - tfw) : ke.wofs;
        const int g_off = __shfl_sync(0xffffffffu, cst, 0 * 4 + db) + ke.zofs;
        const int cd_off = __shfl_sync(0xffffffffu, cst, 1 * 4 + db) + ke.rdyn;
        const int cs_off = __shfl_sync(0xffffffffu, cst, 2 * 4 + db) + ke.rstage;
        const int jd_off = __shfl_sync(0xffffffffu, cst, 3 * 4 + db) + ke.jdyn;
        const int js_off = __shfl_sync(0xffffffffu, cst, 4 * 4 + db) + ke.jstage;
        const int hd_off = __shfl_sync(0xffffffffu, cst, 5 * 4 + db) + ke.hslot;
        const int ld_off = __shfl_sync(0xffffffffu, cst, 6 * 4 + db) + ke.rdyn;
        const int ls_off = __shfl_sync(0xffffffffu, cst, 7 * 4 + db) + ke.rstage;
        const int sg_off = sbase0 + ioff[DTO_IN_SIGMA] + ((q.b0 ^ ptr_parity(a.sigma)) & 1) + db;
        const int flags = (m.in ? 1 : 0) | (m.own ? 2 : 0);
        d0.x = x_off | (ke.nx << 16);
        d0.y = y_off | (w_off << 16);
        d0.z = DO_H ? (ld_off | (ls_off << 16)) : 0;
        d0.w = (DO_H ? sg_off : 0) | (flags << 16);
        d1.x = (ke.kcost & 255) | ((ke.kdyn & 255) << 8) | ((ke.kstage & 255) << 16) | ((ke.hclass & 255) << 24);
        d1.y = (DO_G ? g_off : 0) | ((DO_C ? cd_off : 0) << 16);
        d1.z = (DO_C ? cs_off : 0) | ((DO_J ? jd_off : 0) << 16);
        d1.w = DO_J ? js_off : 0;
        d2.x = DO_H ? hd_off : 0;
        d2.y = db;        // problem = b0 (stage header) + db
        d2.z = m.t;
        d2.w = ke.hslot;
    }
}

// one warp per (t0, parity of b0): the records of a full tile starting at knot t0 of problem b0
template <class M, int MODE>
__global__ void __launch_bounds__(128) plan_kernel(const __grid_constant__ dto_launch_args a, int4* __restrict__ plan)
{
    constexpr bool HALO = ((MODE & DTO_MODE_H) != 0) && (M::HESS_HALO != 0);
    constexpr int OWN = HALO ? 31 : 32;
    const int lane = threadIdx.x & 31;
    const int w = blockIdx.x * 4 + (threadIdx.x >> 5);
    if (w >= 2 * a.T) return;
    const int t0 = w >> 1, pc = w & 1;
    int base[6], ioff[5], in_sz, stage_sz, out0, out_sz, gl_off;
    ws_layout<MODE>(a, base, ioff, &in_sz, &stage_sz, &out0, &out_sz, &gl_off);
    const tile_t q = tile_geom_at<HALO>(a, pc * a.T + t0, OWN);  // problem index = its parity: same alignment as any b0 of that parity
    int4 copy, piece, d0, d1, d2;
    ws_tile_records<M, MODE>(a, a.knot, q, lane, base, ioff, 8, copy, piece, d0, d1, d2);
    const int G4 = ws_gen_int4<MODE>(a);
    int4* P = plan + (size_t)w * (DTO_WS_PLAN_INT4 + G4);
    if (G4) {
        // ---- general-constraint Hessian entries owned by this lane's knot (src/general_constraint.jl:85-91) as
        // records {slot offset | template, z offset, lambda offset, wbase}: their z comes from the staged z
        // range, their multipliers from one extra staged range per problem (copy slots of lanes 4..7), so the
        // compute lane evaluates them without a single load from HBM. A lane whose entries do not fit (more than
        // K entries, z outside the tile, multiplier range longer than LCAP) gets count -1: in-kernel table path.
        const int* tabw = reinterpret_cast<const int*>(a.knot);
        const int T = a.T;
        const int tfz = tabw[q.tf * 16 + 0];
        const bool own = ((d0.w >> 16) & 2) != 0;
        const int db = d2.y, t = d2.z;
        const int p0 = own ? a.gh_ptr[t] : 0;
        const int cnt = own ? a.gh_ptr[t + 1] - p0 : 0;
        const int4* rec = reinterpret_cast<const int4*>(a.gh_rec);
        int lmin = 0x7fffffff, lmax = -0x7fffffff;
        for (int k = 0; k < cnt; ++k) {
            const int4 r0 = rec[2 * (p0 + k)], r1 = rec[2 * (p0 + k) + 1];
            if (r1.z > 0) {
                lmin = min(lmin, r0.w);
                lmax = max(lmax, r0.w + r1.z);
            }
        }
        int glo[4], gpar[4];
        bool gst[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const bool mine = own && db == j;
            const int lo = __reduce_min_sync(0xffffffffu, mine ? lmin : 0x7fffffff);
            const int hi = __reduce_max_sync(0xffffffffu, mine ? lmax : -0x7fffffff);
            const int len = (lo != 0x7fffffff) ? hi - lo : 0;
            gst[j] = len > 0 && len <= DTO_WS_GEN_LCAP;
            glo[j] = lo;
            gpar[j] = gst[j] ? ptr_parity(a.lam + (size_t)(pc + j) * a.N_c + a.gen_row0 + lo) : 0;
            if (gst[j] && lane == 4 + j)
                copy = make_int4(j * a.N_c + a.gen_row0 + lo - gpar[j], ((len + gpar[j] + 1) & ~1) * 8, 8 + gl_off + j * (DTO_WS_GEN_LCAP + 2), 3);
        }
        const int kl1z = tabw[(q.tl + 1) * 16 + 0], kl1n = tabw[(q.tl + 1) * 16 + 1];
        const int zend_last = kl1z + (q.tl + 1 < T ? kl1n : 0);
        const int zlo = db == 0 ? tfz : 0, zhi = (db == q.nsub - 1) ? zend_last : a.N_z;
        const int zb0 = 8 + ioff[DTO_IN_Z] + (((q.b0 & a.N_z) ^ tfz ^ ptr_parity(a.z)) & 1) + db * a.N_z - tfz;  // + z index
        bool ok = cnt <= DTO_WS_GEN_K;
#pragma unroll
        for (int k = 0; k < DTO_WS_GEN_K; ++k) {
            int4 r = make_int4(0, 0, 0, 0);
            if (k < cnt) {
                const int4 r0 = rec[2 * (p0 + k)], r1 = rec[2 * (p0 + k) + 1];
                const bool zin = r1.y == 0 || (r0.z >= zlo && r0.z + r1.y <= zhi);
                bool lin = r1.z == 0;
                int loff = 0;
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (db == j && r1.z > 0) {
                        lin = gst[j];
                        loff = 8 + gl_off + j * (DTO_WS_GEN_LCAP + 2) + gpar[j] + (r0.w - glo[j]);
                    }
                const int srel = r0.x - d2.w;
                ok = ok && zin && lin && srel >= 0 && srel < 65536 && r0.y < 65536;
                r = make_int4(srel | (r0.y << 16), zb0 + r0.z, loff, r1.x);
            }
            P[160 + lane * DTO_WS_GEN_K + k] = r;
        }
        reinterpret_cast<int*>(P + 160 + 32 * DTO_WS_GEN_K)[lane] = ok ? cnt : -1;
    }
    P[lane] = copy;
    P[32 + lane] = d0;
    P[64 + lane] = d1;
    P[96 + lane] = d2;
    P[128 + lane] = piece;
}

// setmaxnreg can only hand out what the launch allocated (12 warps x 168 registers): a split that asks
// for more makes the compute warps spin in setmaxnreg.inc forever (measured: a hung launch)
static_assert(DTO_WS_HELPERS <= DTO_WS_COMPUTE && DTO_WS_WARPS <= 32, "at most one helper per compute warp, at most 32 warps");
static_assert(DTO_WS_HELPERS * DTO_WS_HREG + DTO_WS_COMPUTE * DTO_WS_CREG <= DTO_WS_WARPS * DTO_WS_BASE_REGS,
              "DTO_WS_HREG / DTO_WS_CREG exceed the registers of the launch (64 K per SM over all warps of the CTA)");
static_assert(DTO_WS_HREG % 8 == 0 && DTO_WS_CREG % 8 == 0 && DTO_WS_HREG >= 24 && DTO_WS_CREG <= 256, "setmaxnreg takes multiples of 8 in [24, 256]");

template <class M, int MODE>
__global__ void __launch_bounds__((DTO_WS_COMPUTE + DTO_WS_HELPERS) * 32, 1) knot_kernel_ws(const __grid_constant__ dto_launch_args a)
{
    extern __shared__ __align__(16) double dto_smem[];
    constexpr bool DO_G = (MODE & DTO_MODE_G) != 0, DO_C = (MODE & DTO_MODE_C) != 0;
    constexpr bool DO_J = (MODE & DTO_MODE_J) != 0, DO_H = (MODE & DTO_MODE_H) != 0;
    constexpr bool HALO = DO_H && (M::HESS_HALO != 0);
    constexpr int OWN = HALO ? 31 : 32;
    constexpr bool HG = DO_H && (M::HG_NCLASS > 0);

    const int lane = threadIdx.x & 31;
    const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);  // warp-uniform for the compiler
    const int T = a.T;
    const int total = (int)(a.B * T);
    const int tiles = (total + OWN - 1) / OWN;
    // programmatic dependent launch: the next kernel of the stream may start its CTAs as soon as SMs free up, and
    // load and compute its first tiles while this grid finishes (see launch_pdl for what it may do before its wait)
    asm volatile("griddepcontrol.launch_dependents;");

    // the knot table lives in shared memory (the launch plan guarantees it fits). Only the slow path (ragged last
    // tile, launches without a plan table) reads it, so nobody waits for it here: one bulk copy, completion on
    // its own mbarrier (the 8 bytes after the table), waited for where the table is first used
    const int kt_doubles = (T + 1) * 8 + 2;
    const uint32_t kt_bar = smem_u32(dto_smem + (T + 1) * 8);
    if (threadIdx.x == 0) {
        mbar_init(kt_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(kt_bar, (uint32_t)(T + 1) * 64u);
        bulk_load(smem_u32(dto_smem), a.knot, (uint32_t)(T + 1) * 64u, kt_bar);
        mbar_arrive(kt_bar);
    }
    const dto_knot_entry* tab = reinterpret_cast<const dto_knot_entry*>(dto_smem);
    bool kt_ready = false;

    int base[6], ioff[5], in_sz, stage_sz, out0, out_sz;
    const int NOUT = a.ws_nout;  // output staging buffers per compute warp (1 or 2)
    const int per_warp1 = ws_layout<MODE>(a, base, ioff, &in_sz, &stage_sz, &out0, &out_sz);
    const int per_warp = per_warp1 + (NOUT - 1) * out_sz;
    if (warp >= DTO_WS_HELPERS && lane == 0) {
        const uint32_t bar = smem_u32(dto_smem + kt_doubles + (size_t)(warp - DTO_WS_HELPERS) * per_warp);
        for (int i = 0; i < 6; ++i) mbar_init(bar + 8 * i, 1);  // full[2], out_full[2], out_empty[2]
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    __syncthreads();
    const int stride = gridDim.x * DTO_WS_COMPUTE;
    const int4* __restrict__ plan = reinterpret_cast<const int4*>(a.ws_plan);
    const int G4 = ws_gen_int4<MODE>(a);  // int4 of general-constraint records per plan block / stage

    // The previous kernel of the stream may still be running. It writes none of what this kernel reads (z, lambda,
    // sigma, w, the knot and plan tables: see launch_pdl), but it may still write, or not yet have written, g, c, J
    // and H. So only global WRITES wait for it: a helper executes griddepcontrol.wait before its first store, and
    // the compute warps, which write shared memory only, never wait. Helper 0 of CTA 0 always drains tile 0, so
    // this grid does not complete before the previous one has (and a later launch's wait covers both).
    if (warp < DTO_WS_HELPERS) {
        // =============================== helper warp ===============================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(DTO_WS_HREG));
        bool dep_ok = false;
        for (int kk = 0;; ++kk) {
            bool any = false;
#pragma unroll 1
            for (int ci = 0; ci < (DTO_WS_COMPUTE + DTO_WS_HELPERS - 1) / DTO_WS_HELPERS; ++ci) {
                const int c = warp + ci * DTO_WS_HELPERS;   // helper h serves compute warps h, h + HELPERS, ...
                if (c >= DTO_WS_COMPUTE) break;
                const int tile0 = blockIdx.x * DTO_WS_COMPUTE + c;
                const int tile = tile0 + kk * stride;                                // tile to produce
                const bool have_drain = kk >= 2 && tile0 + (kk - 2) * stride < tiles;  // tile kk-2 to drain
                const bool have_prod = tile < tiles;
                if (!have_drain && !have_prod) continue;
                any = true;
                double* smc = dto_smem + kt_doubles + (size_t)c * per_warp;
                const uint32_t bar0 = smem_u32(smc);
                const int st = kk & 1;  // input stage of tile kk and of tile kk-2
                const uint32_t full = bar0 + st * 8;
                const int din = st * stage_sz;                                  // stage st relative to stage 0 (doubles)
                int4* sdesc = reinterpret_cast<int4*>(smc + 8 + din + in_sz);   // d0[32] d1[32] d2[32] piece[32] header
                const int od = (kk - 2) & (NOUT - 1), nd = (kk - 2) >> (NOUT - 1);  // output buffer / use count of tile kk-2 (NOUT is 1 or 2)
                if (have_drain) {
                    if (!dep_ok) {   // first global write of this warp: wait until the previous kernel has completed
                        asm volatile("griddepcontrol.wait;" ::: "memory");
                        dep_ok = true;
                    }
                    // ---- tile kk-2 is complete in output buffer od: issue its stores (piece list of stage st)
                    mbar_wait(bar0 + 16 + od * 8, nd & 1);
                    const int4 pd = sdesc[96 + lane];
                    const int b0 = reinterpret_cast<const int*>(sdesc + 128 + G4)[0];
                    int len = pd.w;
                    if (len > 0) {
                        double* dst = ws_out_array(a, pd.y, b0) + pd.x;
                        const double* sp = smc + pd.z + od * out_sz;
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
                    bulk_commit();
                    __syncwarp();  // every lane has read its piece before the stage is refilled
                }
                if (have_prod) {
                    const int g0 = tile * OWN;
                    const int n = (g0 + OWN <= total) ? OWN : total - g0;
                    int4 copy;
                    int b0;
                    if (plan != nullptr && n == OWN) {
                        // ---- full tile: its records are block (t0, b0 & 1) of the plan table ----
                        int t0;
                        split_item(a, g0, b0, t0);
                        const int4* P = plan + (size_t)(t0 * 2 + (b0 & 1)) * (DTO_WS_PLAN_INT4 + G4);
                        copy = __ldg(P + lane);
                        if (lane == 0) {
                            mbar_expect_tx(full, (uint32_t)(128 + G4) * 16u);
                            bulk_load(smem_u32(sdesc), P + 32, (uint32_t)(128 + G4) * 16u, full);
                        }
                    } else {
                        // ---- ragged last tile (or no plan table): compute the records here ----
                        if (!kt_ready) {
                            mbar_wait(kt_bar, 0);   // the knot table has landed in shared memory
                            kt_ready = true;
                        }
                        const tile_t q = tile_geom_at<HALO>(a, g0, n);
                        b0 = q.b0;
                        int4 piece, d0, d1, d2;
                        ws_tile_records<M, MODE>(a, tab, q, lane, base, ioff, 8, copy, piece, d0, d1, d2);
                        sdesc[lane] = d0;
                        sdesc[32 + lane] = d1;
                        sdesc[64 + lane] = d2;
                        sdesc[96 + lane] = piece;
                        if (G4) reinterpret_cast<int*>(sdesc + 128 + 32 * DTO_WS_GEN_K)[lane] = -1;  // general entries: table path
                    }
                    if (copy.y > 0) {
                        mbar_expect_tx(full, (uint32_t)copy.y);
                        bulk_load(smem_u32(smc + copy.z + din), ws_in_array(a, copy.w, b0) + copy.x, (uint32_t)copy.y, full);
                    }
                    if (lane == 0) sdesc[128 + G4] = make_int4(b0, 0, 0, 0);
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full);
                }
                if (have_drain) {
                    bulk_wait_read();  // the stores of tile kk-2 have read their shared-memory source
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar0 + 32 + od * 8);  // out_empty: buffer od may be overwritten
                }
            }
            if (!any && kk >= 2) break;  // (a lone tile is produced in round 0 and drained in round 2)
        }
        // the stores only have to have READ their shared-memory source before the CTA exits; their global writes
        // complete with the grid (what a TMA-store epilogue waits for: cp.async.bulk.wait_group.read 0)
        bulk_wait_read();
        if (!kt_ready && warp == 0) mbar_wait(kt_bar, 0);  // never leave a bulk copy into this CTA's shared memory in flight
    } else {
        // =============================== compute warp ===============================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(DTO_WS_CREG));
        const int c = warp - DTO_WS_HELPERS;
        double* __restrict__ smc = dto_smem + kt_doubles + (size_t)c * per_warp;
        const uint32_t bar0 = smem_u32(smc);
        const bool hg_on = HG && a.use_hclass;
        int k = 0;
        for (int tile = blockIdx.x * DTO_WS_COMPUTE + c; tile < tiles; tile += stride, ++k) {
            const int st = k & 1;
            const int o = k & (NOUT - 1), no = k >> (NOUT - 1);
            const int4* dsc = reinterpret_cast<const int4*>(smc + 8 + st * stage_sz + in_sz);
            const int n_items = (tile * OWN + OWN <= total) ? OWN : total - tile * OWN;
            mbar_wait(bar0 + st * 8, (k >> 1) & 1);          // inputs + descriptors of this tile are in the stage
            mbar_wait(bar0 + 32 + o * 8, (no & 1) ^ 1);      // output buffer o has been drained (passes on first use)
            {
                int4 d0 = dsc[lane], d1 = dsc[32 + lane];
                const int4 d2 = dsc[64 + lane];
                // records are laid out for input stage 0 / output buffer 0: shift to stage st / buffer o
                {
                    const int din = st * stage_sz, dout = o * out_sz;
                    d0.x += din;
                    d0.y += a.w_flat ? (din | (din << 16)) : din;
                    d0.z += din | (din << 16);
                    d0.w += din;
                    d1.y += dout | (dout << 16);
                    d1.z += dout | (dout << 16);
                    d1.w += dout;
                }
                const int flags = d0.w >> 16;
                const int li = lane - (HALO ? 1 : 0);           // item position among the tile's own items
                const bool in = (flags & 1) && li < n_items;    // (the records may describe a full tile)
                const bool own = (flags & 2) && li < n_items;
                // Hessian terms of this lane's knot, by role: registers (all indices are compile-time)
                double tc[M::MAXC], td[M::MAXD], ts[M::MAXS];
                if (in) {
                    const double* __restrict__ x = smc + (d0.x & 0xffff);
                    const double* __restrict__ u = x + (d0.x >> 16);
                    const double* __restrict__ y = smc + (d0.y & 0xffff);
                    const int kcost = d1.x & 255, kdyn = (d1.x >> 8) & 255, kstage = (d1.x >> 16) & 255;
                    const double* __restrict__ w = smc + ((unsigned)d0.y >> 16);
                    if (!a.w_flat) w = a.w + (size_t)(dsc[128 + G4].x + d2.y) * a.N_w + ((unsigned)d0.y >> 16);
                    const double* __restrict__ lam_d = smc + (d0.z & 0xffff);
                    const double* __restrict__ lam_s = smc + ((unsigned)d0.z >> 16);
                    if (own) {
                        if (DO_G) M::cost_grad(kcost, x, u, w, smc + (d1.y & 0xffff));
                        if (DO_H) M::cost_hess(kcost, x, u, w, smc[d0.w & 0xffff], tc);
                    }
                    if (kdyn != 255) {
                        if (DO_C) M::dyn_res(kdyn, y, x, u, w, smc + ((unsigned)d1.y >> 16));
                        double* jd = smc + ((unsigned)d1.z >> 16);
                        if (DO_J && DO_H) M::dyn_jac_hess(kdyn, y, x, u, w, lam_d, jd, td);
                        else if (DO_J) M::dyn_jac(kdyn, y, x, u, w, jd);
                        else if (DO_H) M::dyn_hess(kdyn, y, x, u, w, lam_d, td);
                    }
                    if (own && kstage != 255) {
                        if (DO_C) M::stage_res(kstage, x, u, w, smc + (d1.z & 0xffff));
                        double* js = smc + (d1.w & 0xffff);
                        if (DO_J && DO_H) M::stage_jac_hess(kstage, x, u, w, lam_s, js, ts);
                        else if (DO_J) M::stage_jac(kstage, x, u, w, js);
                        else if (DO_H) M::stage_hess(kstage, x, u, w, lam_s, ts);
                    }
                }
                // the previous knot's dynamics terms that feed this knot's rows come from the lane below
                // (lane = consecutive items; with a halo, lane 0 is the item before the tile)
                double pd[M::MAXD];
                if (HALO) M::hg_prev_exchange(td, pd);
                // Hessian slots of this lane's knot: own terms from registers + the previous knot's
                // dynamics terms, summed in the reference's += order (src/moi.jl:88-118)
                if (hg_on && own) {
                    const int hclass = (int)((unsigned)d1.x >> 24);
                    double v[M::HG_VMAX > 0 ? M::HG_VMAX : 1];
                    double* dst = smc + d2.x + o * out_sz;
                    M::hg_compute_r(hclass, tc, td, ts, pd, v);
                    M::hg_store(hclass, v, dst);
                    if (a.gen_nhess > 0) {
                        // general-constraint entries of this knot's slots: last in the += order (src/moi.jl:112-118)
                        const int b = dsc[128 + G4].x + d2.y, t = d2.z;
                        const int gc = reinterpret_cast<const int*>(dsc + 128 + 32 * DTO_WS_GEN_K)[lane];
                        if (gc >= 0) {  // plan records: z and multipliers are in the stage
                            const int din = st * stage_sz;
#pragma unroll
                            for (int kq = 0; kq < DTO_WS_GEN_K; ++kq)
                                if (kq < gc) {
                                    const int4 r = dsc[128 + lane * DTO_WS_GEN_K + kq];
                                    const double val = M::gen_eval(2, (int)((unsigned)r.x >> 16), smc + r.y + din, a.w + (size_t)b * a.N_w + r.w, smc + r.z + din);
                                    dst[r.x & 0xffff] += val;
                                }
                        } else {  // table path (entries that do not fit the records; ragged last tile)
                            const int p0 = __ldg(a.gh_ptr + t), p1 = __ldg(a.gh_ptr + t + 1);
                            for (int p = p0; p < p1; ++p) {
                                const int2 e = __ldg(reinterpret_cast<const int2*>(a.gh_ent) + p);  // slot, instance
                                const int4 inst = __ldg(reinterpret_cast<const int4*>(a.gen_inst[2]) + e.y);
                                const double val = M::gen_eval(2, inst.x, a.z + (size_t)b * a.N_z + inst.y, a.w + (size_t)b * a.N_w + inst.z,
                                                               a.lam + (size_t)b * a.N_c + a.gen_row0 + inst.w);
                                dst[e.x - d2.w] += val;
                            }
                        }
                    }
                }
            }
            fence_async_smem();  // this lane's generic-proxy writes -> visible to the bulk-store engine
            __syncwarp();
            if (lane == 0) mbar_arrive(bar0 + 16 + o * 8);  // out_full: the helper streams the tile out and refills the stage
        }
    }
}

// launch plan: shared memory, or 0 if the shape / mode is not covered by the specialised kernel
template <class M, int MODE>
inline int64_t plan_ws(dto_launch_args& b)
{
    constexpr bool DO_H = (MODE & DTO_MODE_H) != 0;
    if (!DTO_WS || !b.persist_ok || b.nsub_max > 4) return 0;   // (segment row, problem) lane map: 8 rows x 4 problems
    // Measured selection (profiles/sweep_r01_s_per_kernel.jsonl, sweep_r01_ae_helpers.jsonl): the gradient /
    // residual / Jacobian-only passes are light and HBM-bound, the plain kernel's occupancy wins there; every
    // Hessian pass wins here (FP64-heavy models with 4 helpers + 232-register compute warps, light models
    // with one helper per compute warp: car T=201 256 -> 196 us, pendulum T=11 41 -> 36 us).
    if (!DO_H && !DTO_WS_ALL_MODES) return 0;
    if (DO_H && !(M::HG_NCLASS > 0 && b.use_hclass)) return 0;     // table gather: other kernels
    if (M::N_KINDS_MAX >= 255 || M::HG_NCLASS >= 255) return 0;    // descriptor packs kinds in 8 bits
    if (!b.w_flat && b.N_w > 65535) return 0;
    int out_sz = 0;
    const int64_t one = (int64_t)ws_layout<MODE>(b, nullptr, nullptr, nullptr, nullptr, nullptr, &out_sz);
    const int64_t kt = (int64_t)(b.T + 1) * 64 + 16;   // + the table's mbarrier
    for (int nout = 2; nout >= 1; --nout) {
        const int64_t per_warp = one + (nout - 1) * (int64_t)out_sz;
        if (per_warp > 65535) continue;  // 16-bit region offsets
        const int64_t smem = kt + per_warp * 8 * DTO_WS_COMPUTE;
        if (smem <= DTO_SMEM_LIMIT - 1024) {
            b.kt_smem = 1;
            b.ws_nout = nout;
            return smem;
        }
    }
    return 0;
}

// The tile-plan table of (shape, mode, pointer alignment): built once on first use, kept for the
// life of the process (a few hundred KB per entry; the cache is flushed when it grows past 128).
struct ws_plan_entry {
    int64_t shape_id;
    int mode, dev;
    unsigned sig;
    void* ptr;
};
inline unsigned ws_plan_sig(const dto_launch_args& a)
{
    const void* p[9] = {a.z, a.lam, a.sigma, a.w, a.g, a.c, a.J, a.H, a.f};
    unsigned s = 0;
    for (int i = 0; i < 9; ++i) s |= (unsigned)((reinterpret_cast<uintptr_t>(p[i]) >> 3) & 1) << i;
    return s;
}
template <class M, int MODE>
inline const void* ws_get_plan(const dto_launch_args& b, cudaStream_t st)
{
    static std::mutex mu;
    static std::vector<ws_plan_entry> cache;
    if (!DTO_WS_PLAN || b.shape_id == 0) return nullptr;
    int dev = 0;
    cudaGetDevice(&dev);
    const unsigned sig = ws_plan_sig(b);
    std::lock_guard<std::mutex> lock(mu);
    for (const ws_plan_entry& e : cache)
        if (e.shape_id == b.shape_id && e.mode == MODE && e.dev == dev && e.sig == sig) return e.ptr;
    if (cache.size() >= 128) {  // bounded: drop everything once nothing can still be reading it
        for (const ws_plan_entry& e : cache) {
            cudaSetDevice(e.dev);
            cudaDeviceSynchronize();
            cudaFree(e.ptr);
        }
        cudaSetDevice(dev);
        cache.clear();
    }
    void* ptr = nullptr;
    const size_t bytes = (size_t)2 * b.T * (DTO_WS_PLAN_INT4 + ws_gen_int4<MODE>(b)) * sizeof(int4);
    if (cudaMalloc(&ptr, bytes) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;  // no table: every tile takes the in-kernel path
    }
    plan_kernel<M, MODE><<<(2 * b.T + 3) / 4, 128, 0, st>>>(b, reinterpret_cast<int4*>(ptr));
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) {
        cudaFree(ptr);
        return nullptr;
    }
    cache.push_back({b.shape_id, MODE, dev, sig, ptr});
    return ptr;
}
