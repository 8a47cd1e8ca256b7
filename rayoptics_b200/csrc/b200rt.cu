/*
 * b200rt.cu -- kernels and C ABI of libb200rt.so (see include/b200rt.h).
 *
 * Kernels (sm_100a; fp64 vector pipe + coalesced SoA global traffic; no tensor
 * cores -- the path is not a contraction):
 *   k_trace_bundle<FULL,STAGE>  one ray per lane over caller-supplied start rays
 *   k_trace_grid<FULL,SUMMARY,STAGE>  start rays generated on device from the
 *                               (field, wavelength, pupil i, j) index, optional
 *                               per-chunk spot sums
 *   k_reduce_summary            fixed-order per-tile reduction of the chunk sums
 *   k_dfma_peak                 fp64 FMA microbenchmark (roofline denominator)
 *
 * The surface table (n_ifc x rt_surface_desc + n_wvl x n_ifc indices) is staged
 * into shared memory once per CTA; CTAs are persistent (grid = SMs x resident
 * CTAs): the bundle kernels walk rays with a grid stride, the warps of the grid
 * kernels draw 32-ray work items from a per-launch counter.
 */
#include <cuda_runtime.h>
#include <math_constants.h>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <type_traits>
#include <vector>

#include "rt_device.cuh"
#include "rt_lean.cuh"
#include "rt_grid.cuh"

using namespace b200rt;

#define RT_BLOCK 256          /* threads per CTA = rays per chunk */
#define RT_LEAN_MIN_CTAS 3   /* resident CTAs per SM the lean kernels are register-limited for */
#define RT_MAX_STAGE_BYTES (200*1024)

/* ------------------------------------------------------------------ errors */
static thread_local std::string g_err;
static std::atomic<int64_t> g_launches{0};

static int fail(int code, const char *fmt, const char *a = "", const char *b = "")
{
    char buf[512];
    snprintf(buf, sizeof buf, fmt, a, b);
    g_err = buf;
    return code;
}

#define CUDA_TRY(expr)                                                            \
    do {                                                                          \
        cudaError_t e_ = (expr);                                                  \
        if (e_ != cudaSuccess)                                                    \
            return fail(RT_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(e_));    \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) {
            cudaSetDevice(dev);
            changed = true;
        }
    }
    ~DeviceGuard()
    {
        if (changed) cudaSetDevice(prev);
    }
};

/* ------------------------------------------------------------------ handles */
struct rt_table {
    int32_t device, n_ifc, n_wvl, sm_count;
    rt_surface_desc *d_surfs;
    double *d_n;
    double *d_wvl;           /* [n_wvl] wavelengths in nm (NaN until rt_table_set_wavelengths) */
    bool has_phase;
    size_t stage_bytes;      /* shared memory needed to stage the table */
    bool stage;              /* false: table too large, read it from global/L1 */
    bool lean;               /* all interfaces quadric, unrotated, max_aperture clipping only */
    bool lean_poly;          /* lean, with polynomial / toroid profiles (out-of-line Newton) */
    bool wave_ok;            /* interface n_ifc-2 carries no decenter: OPD epilogue applicable */
    size_t lean_bytes;       /* shared memory of the lean plan */
    unsigned long long *d_counters;     /* ring of RT_COUNTERS work counters */
    std::atomic<unsigned> next_counter;
};
#define RT_COUNTERS 64

struct rt_grid {
    int32_t device;
    int32_t n_fields, n_wvls, nx, ny;
    int32_t apply_vignetting, flip_z_dir, paired, pupil_kind;
    double eprad, z_pupil, foc;
    rt_field_desc *d_fields;
    int32_t *d_wvl_idx;
    double *d_pupil_x, *d_pupil_y, *d_ref_img, *d_wave;
    void *d_block;           /* the one device allocation the pointers above point into */
    int64_t rays_per_tile, chunks_per_tile, n_tiles, n_chunks, n_rays;
    std::vector<int32_t> h_wvl_idx;   /* host copy: range-checked against the table in rt_trace_grid */
    unsigned char *h_stage;           /* pinned image of d_block */
    cudaEvent_t uploaded;             /* last rt_grid_update copy */
    size_t b_fields, b_px, b_py, b_ref, b_wave, o_fields, o_px, o_py, o_ref, o_wave, o_wvl, total;
    /* rt_trace_grid_to_host: two internal streams + events (created on first use) */
    cudaStream_t side[2];
    cudaEvent_t ev_in, ev_side[2];
    bool side_ok;
};

/* what the grid kernel needs, passed by value */
/* ------------------------------------------------------------------ kernels */

/* Stage the table into shared memory (8-byte words, coalesced) or, for very
 * long systems, leave it in global memory (uniform loads hit L1). */
template <bool STAGE>
__device__ __forceinline__ void stage_table(const rt_surface_desc *g_surfs, const double *g_n,
                                            int n_ifc, int n_wvl, unsigned char *smem,
                                            const rt_surface_desc *&tab, const double *&ntab)
{
    if (STAGE) {
        const int words_s = n_ifc*(int)(sizeof(rt_surface_desc)/8);
        const int words_n = n_ifc*n_wvl;
        double *dst = reinterpret_cast<double *>(smem);
        const double *src = reinterpret_cast<const double *>(g_surfs);
        for (int i = threadIdx.x; i < words_s; i += blockDim.x) dst[i] = src[i];
        for (int i = threadIdx.x; i < words_n; i += blockDim.x) dst[words_s + i] = g_n[i];
        __syncthreads();
        tab = reinterpret_cast<const rt_surface_desc *>(smem);
        ntab = dst + words_s;
    } else {
        tab = g_surfs;
        ntab = g_n;
    }
}

__device__ __forceinline__ void store_result(const rt_out &out, int64_t k, const RayResult &R)
{
    if (out.px) { out.px[k] = R.p.x; out.py[k] = R.p.y; out.pz[k] = R.p.z; }
    if (out.dx) { out.dx[k] = R.d.x; out.dy[k] = R.d.y; out.dz[k] = R.d.z; }
    if (out.nx) { out.nx[k] = R.n.x; out.ny[k] = R.n.y; out.nz[k] = R.n.z; }
    if (out.dst) out.dst[k] = R.dst;
    if (out.op) out.op[k] = R.op;
    if (out.status) out.status[k] = R.status;
    if (out.fail_surf) out.fail_surf[k] = R.fail_surf;
    if (out.n_seg) out.n_seg[k] = R.n_seg;
}

template <bool FULL, bool STAGE>
__global__ void __launch_bounds__(RT_BLOCK)
k_trace_bundle(const rt_surface_desc *__restrict__ g_surfs, const double *__restrict__ g_n,
               int n_ifc, int n_wvl, int64_t n_rays,
               const double *__restrict__ px, const double *__restrict__ py,
               const double *__restrict__ pz, const double *__restrict__ dx,
               const double *__restrict__ dy, const double *__restrict__ dz,
               const int32_t *__restrict__ wvl_idx, rt_opts o, rt_out out,
               const double *__restrict__ g_wvl)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const rt_surface_desc *tab;
    const double *ntab;
    stage_table<STAGE>(g_surfs, g_n, n_ifc, n_wvl, smem, tab, ntab);

    const int64_t step = (int64_t)gridDim.x*blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x*blockDim.x + threadIdx.x; r < n_rays; r += step) {
        Vec3 p0 = {px[r], py[r], pz[r]};
        Vec3 d0 = {dx[r], dy[r], dz[r]};
        const int w = wvl_idx ? wvl_idx[r] : o.wvl_idx;
        FullWriter fw = {FULL ? out.full + r : nullptr, out.full_stride};
        RayResult R;
        trace_ray<FULL>(tab, ntab + (int64_t)w*n_ifc, g_wvl[w], n_ifc, o, p0, d0, fw, R);
        store_result(out, r, R);
    }
}

/* ---- per-(field, wvl) spot sums.
 * Records of 16 doubles (15 values + a valid flag); slots of a tile: RT_WARPS x SL,
 * SL = min(chunks_per_tile, RT_MAX_GRID).  When chunks_per_tile <= gridDim.x
 * (chunk slots) a warp writes the record of its 32 rays of a chunk straight from
 * registers, slot = local chunk.  Otherwise every thread keeps the counts and
 * min / max in shared memory (acc[k*RT_BLOCK + tid], conflict-free); when the warp
 * moves on to another tile (or finishes) it shuffle-reduces its lanes into its
 * record of slot blockIdx.x (a warp draws its items in ascending order, so it meets
 * a tile in one run => one record), and the floating-point sums of each work item
 * are stored on their own.  The scratch buffer is zeroed before the launch,
 * k_reduce_summary adds up the valid records of a tile in slot order and the item
 * sums in item order: bit-reproducible, and no CTA barrier in the trace kernel. */
#define RT_WARPS (RT_BLOCK/32)
#define RT_MAX_GRID 2048
#define RT_ACC 15
#define RT_ACC_BYTES (RT_ACC*RT_BLOCK*sizeof(double))

__device__ __forceinline__ void acc_init(double *acc)
{
#pragma unroll
    for (int k = 0; k < RT_ACC; k++)
        acc[k*RT_BLOCK + threadIdx.x] =
            (k == 10 || k == 12) ? CUDART_INF : ((k == 11 || k == 13) ? -CUDART_INF : 0.0);
}

/* only the order-independent columns (counts, min / max) go through the per-thread
 * accumulators; the floating-point sums are reduced per work item (item_sums_store) */
__device__ __forceinline__ void acc_add(double *acc, int status, double ax, double ay)
{
    double *a = acc + threadIdx.x;
    const int ck = status == RT_RAY_OK ? 0 : (status <= RT_RAY_BLOCKED ? status : 4);
    a[ck*RT_BLOCK] += 1.0;
    if (status == RT_RAY_OK) {
        a[10*RT_BLOCK] = fmin(a[10*RT_BLOCK], ax); a[11*RT_BLOCK] = fmax(a[11*RT_BLOCK], ax);
        a[12*RT_BLOCK] = fmin(a[12*RT_BLOCK], ay); a[13*RT_BLOCK] = fmax(a[13*RT_BLOCK], ay);
    }
}

/* the six sums of one work item (32 rays) in 9 shuffles instead of 30: at the 16 / 8 / 4
 * exchanges every lane hands over the half of its values that its partner keeps, so after
 * three steps each lane owns ONE of (up to 8) values summed over 8 lanes; two more exchanges
 * finish that value.  The addition tree is fixed: same rays, same bits. */
#define RT_ITEM_SUMS 6
__device__ __forceinline__ void item_sums_store(bool ok, double ax, double ay, double op, double *dst)
{
    const int lane = threadIdx.x & 31;
    double v0 = ok ? ax : 0.0, v1 = ok ? ay : 0.0, v2 = ok ? ax*ax : 0.0, v3 = ok ? ay*ay : 0.0;
    double v4 = ok ? ax*ay : 0.0, v5 = ok ? op : 0.0, v6 = 0.0, v7 = 0.0;
    const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4;
    /* 16: lower half-warp keeps v0..v3, upper keeps v4..v7 */
    double a0 = (h16 ? v4 : v0) + __shfl_xor_sync(0xffffffffu, h16 ? v0 : v4, 16);
    double a1 = (h16 ? v5 : v1) + __shfl_xor_sync(0xffffffffu, h16 ? v1 : v5, 16);
    double a2 = (h16 ? v6 : v2) + __shfl_xor_sync(0xffffffffu, h16 ? v2 : v6, 16);
    double a3 = (h16 ? v7 : v3) + __shfl_xor_sync(0xffffffffu, h16 ? v3 : v7, 16);
    /* 8: keep a0, a1 | a2, a3 */
    double b0 = (h8 ? a2 : a0) + __shfl_xor_sync(0xffffffffu, h8 ? a0 : a2, 8);
    double b1 = (h8 ? a3 : a1) + __shfl_xor_sync(0xffffffffu, h8 ? a1 : a3, 8);
    /* 4: keep b0 | b1 */
    double c = (h4 ? b1 : b0) + __shfl_xor_sync(0xffffffffu, h4 ? b0 : b1, 4);
    c = c + __shfl_xor_sync(0xffffffffu, c, 2);
    c = c + __shfl_xor_sync(0xffffffffu, c, 1);
    /* lane 4g holds value index 4*[bit 4] + 2*[bit 3] + [bit 2] of g = lane/4 */
    const int idx = ((lane >> 4) & 1)*4 + ((lane >> 3) & 1)*2 + ((lane >> 2) & 1);
    if ((lane & 3) == 0 && idx < RT_ITEM_SUMS) dst[idx] = c;
}

/* warp-reduce the accumulators into the warp's record of (tile, slot) and reset them */
__device__ __forceinline__ void acc_flush(double *acc, double *scratch, int64_t tile, int64_t slot,
                                          int64_t slots_per_tile)
{
    const int lane = threadIdx.x & 31;
    double *dst = scratch + ((tile*slots_per_tile + slot)*RT_WARPS + (threadIdx.x >> 5))*RT_SUMMARY_DOUBLES;
#pragma unroll
    for (int k = 0; k < RT_ACC; k++) {
        double x = acc[k*RT_BLOCK + threadIdx.x];
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            double y = __shfl_down_sync(0xffffffffu, x, off);
            if (k == 10 || k == 12) x = fmin(x, y);
            else if (k == 11 || k == 13) x = fmax(x, y);
            else x = x + y;
        }
        if (lane == 0) dst[k] = x;
    }
    if (lane == 0) dst[RT_ACC] = 1.0;
    acc_init(acc);
}

/* per-chunk variant (chunk slots): the lanes' contributions are reduced straight
 * from registers; lanes without a ray contribute the identity */
__device__ __forceinline__ void warp_record_from_regs(bool have, int status, double ax, double ay,
                                                      double op, double *scratch, int64_t tile,
                                                      int64_t slot, int64_t slots_per_tile, int slice)
{
    const int lane = threadIdx.x & 31;
    double *dst = scratch + ((tile*slots_per_tile + slot)*RT_WARPS + slice)*RT_SUMMARY_DOUBLES;
    const bool ok = have && status == RT_RAY_OK;
#pragma unroll
    for (int k = 0; k < RT_ACC; k++) {
        double x;
        if (k < 5) {
            const int ck = status == RT_RAY_OK ? 0 : (status <= RT_RAY_BLOCKED ? status : 4);
            x = (have && ck == k) ? 1.0 : 0.0;
        } else if (k == 10 || k == 12) x = ok ? (k == 10 ? ax : ay) : CUDART_INF;
        else if (k == 11 || k == 13) x = ok ? (k == 11 ? ax : ay) : -CUDART_INF;
        else if (!ok) x = 0.0;
        else x = k == 5 ? ax : k == 6 ? ay : k == 7 ? ax*ax : k == 8 ? ay*ay : k == 9 ? ax*ay : op;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            double y = __shfl_down_sync(0xffffffffu, x, off);
            if (k == 10 || k == 12) x = fmin(x, y);
            else if (k == 11 || k == 13) x = fmax(x, y);
            else x = x + y;
        }
        if (lane == 0) dst[k] = x;
    }
    if (lane == 0) dst[RT_ACC] = 1.0;
}

/* chunk loop shared by the general and the lean grid kernels: start ray ->
 * trace -> per-ray results -> transverse aberration (focus_pupil_coords,
 * analyses.py:561-580) -> spot sums */
template <bool SUMMARY, bool WAVE, typename TraceFn>
__device__ __forceinline__ void grid_chunk_loop(const GridDev &G, int64_t chunk_begin, int64_t chunk_end,
                                                const rt_out &out, double *scratch, double *acc,
                                                unsigned long long *work_counter, double *item_sums,
                                                TraceFn trace)
{
    const int64_t tile0 = chunk_begin/G.chunks_per_tile;
    const int64_t ray0 = tile0*G.rays_per_tile + (chunk_begin - tile0*G.chunks_per_tile)*RT_BLOCK;
    const int64_t sl = G.chunks_per_tile < RT_MAX_GRID ? G.chunks_per_tile : RT_MAX_GRID;
    const bool chunk_slots = G.chunks_per_tile <= (int64_t)gridDim.x;
    int64_t cur_tile = -1;
    if (SUMMARY && !chunk_slots) acc_init(acc);
    const unsigned long long n_items = (unsigned long long)(chunk_end - chunk_begin)*RT_WARPS;
    for (;;) {
        /* one work item = 32 consecutive rays: every warp draws its next item from a global
         * counter, so no warp idles while rays are left (the cost of a chunk varies several-fold
         * between the pupil centre and its clipped edge) */
        unsigned long long item = 0;
        if ((threadIdx.x & 31) == 0) item = atomicAdd(work_counter, 1ull);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int64_t c = chunk_begin + (int64_t)(item/RT_WARPS);
        const int slice = (int)(item % RT_WARPS);     /* which 32 rays of the chunk this warp takes */
        const int64_t tile = c/G.chunks_per_tile;
        const int64_t lc = c - tile*G.chunks_per_tile;
        const int64_t loc = lc*RT_BLOCK + slice*32 + (threadIdx.x & 31);
        const bool have = loc < G.rays_per_tile;
        if (SUMMARY && !chunk_slots && tile != cur_tile) {
            if (cur_tile >= 0) acc_flush(acc, scratch, cur_tile, blockIdx.x, sl);
            cur_tile = tile;
        }
        int status = RT_RAY_OK;
        double ax = 0.0, ay = 0.0, op = 0.0;
        if (have) {
            const int f = (int)(tile/G.n_wvls);
            const int w = (int)(tile - (int64_t)f*G.n_wvls);
            const int64_t k = tile*G.rays_per_tile + loc - ray0;
            RayResult R;
            Vec3 d0;
            trace(f, w, loc, k, R, d0);
            store_result(out, k, R);
            status = R.status; op = R.op;
            if (WAVE)
                out.opd[k] = (R.status == RT_RAY_OK)
                                 ? wave_opd(G.wave + tile*RT_WAVE_DOUBLES, R.p1, d0, R.pk, R.dk, R.p, R.d, R.op)
                                 : CUDART_NAN;
            if (out.abr_x || SUMMARY) {
                const double rx = G.ref_img ? G.ref_img[tile*2 + 0] : 0.0;
                const double ry = G.ref_img ? G.ref_img[tile*2 + 1] : 0.0;
                double dist = div_maybe_zero(G.foc, R.d.z);
                ax = (R.p.x + dist*R.d.x) - rx;
                ay = (R.p.y + dist*R.d.y) - ry;
                if (out.abr_x) {
                    double sx = ax, sy = ay;
                    if ((out.flags & RT_OUT_ABR_NAN_STATUS) && status != RT_RAY_OK) {
                        sx = __longlong_as_double((long long)(RT_NAN_PAYLOAD_BASE | (unsigned long long)(status & 0xFFFF)));
                        sy = __longlong_as_double((long long)(RT_NAN_PAYLOAD_BASE | (unsigned long long)(R.fail_surf & 0xFFFF)));
                    }
                    out.abr_x[k] = sx; out.abr_y[k] = sy;
                }
                if (SUMMARY && !chunk_slots) acc_add(acc, status, ax, ay);
            }
        }
        /* which warp adds which rays varies from run to run, so the sums of every work item are
         * stored on their own and k_reduce_summary adds them in item order -- the summary stays
         * bit-reproducible */
        if (SUMMARY && !chunk_slots)
            item_sums_store(have && status == RT_RAY_OK, ax, ay, op, item_sums + item*RT_ITEM_SUMS);
        if (SUMMARY && chunk_slots) warp_record_from_regs(have, status, ax, ay, op, scratch, tile, lc, sl, slice);
    }
    if (SUMMARY && !chunk_slots && cur_tile >= 0) acc_flush(acc, scratch, cur_tile, blockIdx.x, sl);
}

template <bool FULL, bool SUMMARY, bool STAGE, bool WAVE>
__global__ void __launch_bounds__(RT_BLOCK)
k_trace_grid(const rt_surface_desc *__restrict__ g_surfs, const double *__restrict__ g_n,
             int n_ifc, int n_wvl, GridDev G, int64_t chunk_begin, int64_t chunk_end,
             rt_opts o, rt_out out, double *__restrict__ scratch, const double *__restrict__ g_wvl,
             int pupil_kind, unsigned long long *work_counter, double *item_sums)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const rt_surface_desc *tab;
    const double *ntab;
    double *acc = reinterpret_cast<double *>(smem);          /* [RT_ACC][RT_BLOCK] when SUMMARY */
    stage_table<STAGE>(g_surfs, g_n, n_ifc, n_wvl, smem + (SUMMARY ? RT_ACC_BYTES : 0), tab, ntab);
    grid_chunk_loop<SUMMARY, WAVE>(G, chunk_begin, chunk_end, out, scratch, acc, work_counter, item_sums,
        [&](int f, int w, int64_t loc, int64_t k, RayResult &R, Vec3 &d0) {
            Vec3 p0;
            grid_start_ray<false>(G, pupil_kind, f, loc, p0, d0);
            FullWriter fw = {FULL ? out.full + k : nullptr, out.full_stride};
            const int wi = G.wvl_idx[w];
            trace_ray<FULL, WAVE>(tab, ntab + (int64_t)wi*n_ifc, g_wvl[wi], n_ifc, o, p0, d0, fw, R);
        });
}

/* ---- lean kernels: plan built in shared memory by the CTA (rt_lean.cuh) */
template <int OUT, bool POLY>
__global__ void __launch_bounds__(RT_BLOCK, POLY ? 2 : RT_LEAN_MIN_CTAS)
k_trace_bundle_lean(const rt_surface_desc *__restrict__ g_surfs, const double *__restrict__ g_n,
                    int n_ifc, int n_wvl, int64_t n_rays,
                    const double *__restrict__ px, const double *__restrict__ py,
                    const double *__restrict__ pz, const double *__restrict__ dx,
                    const double *__restrict__ dy, const double *__restrict__ dz,
                    const int32_t *__restrict__ wvl_idx, rt_opts o, rt_out out)
{
    extern __shared__ __align__(16) unsigned char smem[];
    LeanSurf *ls = reinterpret_cast<LeanSurf *>(smem);
    LeanIdx *li = reinterpret_cast<LeanIdx *>(ls + n_ifc);
    LeanPoly *lp = reinterpret_cast<LeanPoly *>(li + (size_t)n_ifc*n_wvl);      /* POLY instances only */
    build_plan(g_surfs, g_n, n_ifc, n_wvl, o, ls, li);
    if (POLY) build_poly_plan(g_surfs, n_ifc, lp);
    __syncthreads();

    const int64_t step = (int64_t)gridDim.x*blockDim.x;
    for (int64_t r = (int64_t)blockIdx.x*blockDim.x + threadIdx.x; r < n_rays; r += step) {
        Vec3 p0 = {px[r], py[r], pz[r]};
        Vec3 d0 = {dx[r], dy[r], dz[r]};
        const int w = wvl_idx ? wvl_idx[r] : o.wvl_idx;
        FullWriter fw = {OUT == 2 ? out.full + r : nullptr, out.full_stride};
        RayResult R;
        trace_ray_lean<OUT, false, POLY>(ls, li + (int64_t)w*n_ifc, lp, g_surfs, n_ifc, o, p0, d0, fw, R);
        store_result(out, r, R);
    }
}

template <int OUT, bool SUMMARY, bool WAVE, bool POLY>
__global__ void __launch_bounds__(RT_BLOCK, POLY ? 2 : RT_LEAN_MIN_CTAS)
k_trace_grid_lean(const rt_surface_desc *__restrict__ g_surfs, const double *__restrict__ g_n,
                  int n_ifc, int n_wvl, GridDev G, int64_t chunk_begin, int64_t chunk_end,
                  rt_opts o, rt_out out, double *__restrict__ scratch, unsigned long long *work_counter,
                  double *item_sums)
{
    extern __shared__ __align__(16) unsigned char smem[];
    double *acc = reinterpret_cast<double *>(smem);          /* [RT_ACC][RT_BLOCK] when SUMMARY */
    LeanSurf *ls = reinterpret_cast<LeanSurf *>(smem + (SUMMARY ? RT_ACC_BYTES : 0));
    LeanIdx *li = reinterpret_cast<LeanIdx *>(ls + n_ifc);
    LeanPoly *lp = reinterpret_cast<LeanPoly *>(li + (size_t)n_ifc*n_wvl);      /* POLY instances only */
    build_plan(g_surfs, g_n, n_ifc, n_wvl, o, ls, li);
    if (POLY) build_poly_plan(g_surfs, n_ifc, lp);
    __syncthreads();
    grid_chunk_loop<SUMMARY, WAVE>(G, chunk_begin, chunk_end, out, scratch, acc, work_counter, item_sums,
        [&](int f, int w, int64_t loc, int64_t k, RayResult &R, Vec3 &d0) {
            Vec3 p0;
            grid_start_ray<true>(G, RT_PUPIL_EPD, f, loc, p0, d0);
            FullWriter fw = {OUT == 2 ? out.full + k : nullptr, out.full_stride};
            trace_ray_lean<OUT, WAVE, POLY>(ls, li + (int64_t)G.wvl_idx[w]*n_ifc, lp, g_surfs, n_ifc, o, p0, d0, fw, R);
        });
}

/* division self-test: div_shared/normalize3_shared against the IEEE `/` */
__global__ void k_selftest_division(uint64_t seed, int64_t n_per_thread, unsigned long long *mismatch)
{
    uint64_t x = seed + 0x9E3779B97F4A7C15ull*(uint64_t)(blockIdx.x*blockDim.x + threadIdx.x + 1);
    unsigned long long bad = 0;
    for (int64_t it = 0; it < n_per_thread; it++) {
        uint64_t r[4];
        for (int k = 0; k < 4; k++) {          /* splitmix64 */
            x += 0x9E3779B97F4A7C15ull;
            uint64_t z = x;
            z = (z ^ (z >> 30))*0xBF58476D1CE4E5B9ull;
            z = (z ^ (z >> 27))*0x94D049BB133111EBull;
            r[k] = z ^ (z >> 31);
        }
        /* operands: random mantissas, exponents spread over a window chosen by the draw:
         * mostly ordinary magnitudes, sometimes extreme (exercise the fallback) */
        const int mode = (int)(r[3] & 15);
        const int span = mode < 12 ? 40 : (mode < 15 ? 600 : 2046);
        double a[3], b;
        uint64_t bm = (r[3] >> 8) & 0xFFFFFFFFFFFFFull;
        if (((r[3] >> 4) & 15) == 0) bm = 0xFFFFFFFFFFFFFull;        /* all-ones mantissa */
        if (((r[3] >> 4) & 15) == 1) bm = 0;                          /* power of two */
        int be = 1023 + (int)((r[2] >> 40) % (uint64_t)span) - span/2;
        be = be < 0 ? 0 : (be > 2047 ? 2047 : be);
        b = __longlong_as_double((long long)(((r[2] & 1) << 63) | ((uint64_t)be << 52) | bm));
        for (int k = 0; k < 3; k++) {
            int ae = 1023 + (int)((r[k] >> 53) % (uint64_t)span) - span/2;
            ae = ae < 0 ? 0 : (ae > 2047 ? 2047 : ae);
            uint64_t am = r[k] & 0xFFFFFFFFFFFFFull;
            if (((r[k] >> 60) & 7) == 0) am = 0;
            a[k] = __longlong_as_double((long long)(((r[k] >> 52 & 1) << 63) | ((uint64_t)ae << 52) | am));
            if (mode == 7 && k == 2) a[k] = 0.0;
        }
        const double rr = rcp_refined(b);
        for (int k = 0; k < 3; k++) {
            double q1 = div_shared(a[k], b, rr), q2 = a[k]/b;
            if (__double_as_longlong(q1) != __double_as_longlong(q2) && !(isnan(q1) && isnan(q2))) bad++;
        }
        Vec3 v = {a[0], a[1], a[2]};
        if (mode < 12) {
            Vec3 n1 = normalize3_shared(v), n2 = normalize3(v);
            if (__double_as_longlong(n1.x) != __double_as_longlong(n2.x) ||
                __double_as_longlong(n1.y) != __double_as_longlong(n2.y) ||
                __double_as_longlong(n1.z) != __double_as_longlong(n2.z)) {
                if (!(isnan(n1.x) && isnan(n2.x)) ) bad++;
            }
        }
    }
    {   /* sqrt_near_one against sqrt for every bit pattern within 2048 ulps of 1 */
        long long k = (long long)((blockIdx.x*blockDim.x + threadIdx.x) % 4097) - 2048;
        double sv = __longlong_as_double(0x3FF0000000000000LL + k);
        if (__double_as_longlong(sqrt_near_one(sv)) != __double_as_longlong(sqrt(sv))) bad++;
    }
    if (bad) atomicAdd(mismatch, bad);
}

/* Fixed-order reduction of the valid records of each tile.  RT_RED_SPLIT CTAs per
 * tile each add up a contiguous range of records (thread t takes records t,
 * t+256, ... ascending, then a fixed binary tree over the 256 thread sums); the
 * CTA that finishes last (ticket) combines the RT_RED_SPLIT partials in order. */
#define RT_RED_THREADS 256
#define RT_RED_SPLIT 16
__device__ __forceinline__ double red_op(int k, double a, double y)
{
    if (k == 10 || k == 12) return fmin(a, y);
    if (k == 11 || k == 13) return fmax(a, y);
    return a + y;
}

__global__ void __launch_bounds__(RT_RED_THREADS)
k_reduce_summary(const double *__restrict__ scratch, int64_t recs_per_tile, double *partials,
                 unsigned int *tickets, double *__restrict__ summary,
                 const double *__restrict__ item_sums, int64_t chunk_begin, int64_t chunk_end,
                 int64_t chunks_per_tile)
{
    __shared__ double sh[RT_RED_THREADS][RT_SUMMARY_DOUBLES + 1];
    __shared__ bool last;
    const int64_t tile = blockIdx.x/RT_RED_SPLIT;
    const int part = blockIdx.x%RT_RED_SPLIT;
    const int64_t per = (recs_per_tile + RT_RED_SPLIT - 1)/RT_RED_SPLIT;
    int64_t r0 = part*per, r1 = r0 + per;
    if (r1 > recs_per_tile) r1 = recs_per_tile;
    double x[RT_ACC];
#pragma unroll
    for (int k = 0; k < RT_ACC; k++)
        x[k] = (k == 10 || k == 12) ? CUDART_INF : ((k == 11 || k == 13) ? -CUDART_INF : 0.0);
    for (int64_t r = r0 + threadIdx.x; r < r1; r += RT_RED_THREADS) {
        const double *p = scratch + (tile*recs_per_tile + r)*RT_SUMMARY_DOUBLES;
        if (p[RT_ACC] != 0.0) {
#pragma unroll
            for (int k = 0; k < RT_ACC; k++) x[k] = red_op(k, x[k], p[k]);
        }
    }
    if (item_sums) {
        /* the work items of this tile inside the launch's chunk range, in item order: thread t of
         * part p takes items t, t + 256, ... of the part's contiguous range */
        int64_t c0 = tile*chunks_per_tile, c1 = c0 + chunks_per_tile;
        if (c0 < chunk_begin) c0 = chunk_begin;
        if (c1 > chunk_end) c1 = chunk_end;
        if (c1 > c0) {
            const int64_t i0 = (c0 - chunk_begin)*RT_WARPS, n_it = (c1 - c0)*RT_WARPS;
            const int64_t per_it = (n_it + RT_RED_SPLIT - 1)/RT_RED_SPLIT;
            int64_t a0 = part*per_it, a1 = a0 + per_it;
            if (a1 > n_it) a1 = n_it;
            const int col[RT_ITEM_SUMS] = {5, 6, 7, 8, 9, 14};
            for (int64_t it = a0 + threadIdx.x; it < a1; it += RT_RED_THREADS) {
                const double *p = item_sums + (i0 + it)*RT_ITEM_SUMS;
#pragma unroll
                for (int k = 0; k < RT_ITEM_SUMS; k++) x[col[k]] += p[k];
            }
        }
    }
#pragma unroll
    for (int k = 0; k < RT_ACC; k++) sh[threadIdx.x][k] = x[k];
    __syncthreads();
    for (int off = RT_RED_THREADS/2; off > 0; off >>= 1) {
        if (threadIdx.x < off) {
#pragma unroll
            for (int k = 0; k < RT_ACC; k++)
                sh[threadIdx.x][k] = red_op(k, sh[threadIdx.x][k], sh[threadIdx.x + off][k]);
        }
        __syncthreads();
    }
    double *mine = partials + ((int64_t)blockIdx.x)*RT_SUMMARY_DOUBLES;
    if (threadIdx.x < RT_ACC) mine[threadIdx.x] = sh[0][threadIdx.x];
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = (atomicAdd(&tickets[tile], 1u) == RT_RED_SPLIT - 1);
    __syncthreads();
    if (last && threadIdx.x < RT_SUMMARY_DOUBLES) {
        __threadfence();
        const int k = threadIdx.x;
        double v = 0.0;
        if (k < RT_ACC) {
            const volatile double *pp = partials + tile*RT_RED_SPLIT*RT_SUMMARY_DOUBLES;
            v = pp[k];
            for (int j = 1; j < RT_RED_SPLIT; j++) v = red_op(k, v, pp[j*RT_SUMMARY_DOUBLES + k]);
        }
        summary[tile*RT_SUMMARY_DOUBLES + k] = v;
    }
}

/* summary of an empty chunk range: zero counts / sums, identities in the min / max columns */
__global__ void k_summary_identity(double *__restrict__ summary, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x*blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int k = (int)(i % RT_SUMMARY_DOUBLES);
    summary[i] = (k == 10 || k == 12) ? CUDART_INF : ((k == 11 || k == 13) ? -CUDART_INF : 0.0);
}

/* out[tile][k] = parts[0][tile][k] (+|min|max) parts[1][tile][k] ... in part order */
__global__ void k_combine_summaries(const double *__restrict__ parts, int n_parts, int64_t n,
                                    double *__restrict__ out)
{
    const int64_t i = (int64_t)blockIdx.x*blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int k = (int)(i % RT_SUMMARY_DOUBLES);
    double v = parts[i];
    for (int p = 1; p < n_parts; p++) v = red_op(k, v, parts[(int64_t)p*n + i]);
    out[i] = v;
}

/* chief rays of all fields: pupil (0, 0), no vignetting, apertures not checked, general
 * per-ray code on the global table (bit-identical to the lean loop by construction, and
 * n_fields rays do not need the specialised kernel).  One thread per field. */
__global__ void k_chief_ref(const rt_surface_desc *__restrict__ g_surfs, const double *__restrict__ g_n,
                            int n_ifc, GridDev G, int n_fields, int pupil_kind, int wi,
                            const double *__restrict__ g_wvl, rt_opts o, double *__restrict__ ref_img,
                            double *__restrict__ ref_out)
{
    const int f = blockIdx.x*blockDim.x + threadIdx.x;
    if (f >= n_fields) return;
    Vec3 p0, d0;
    grid_start_ray_at<false>(G, pupil_kind, f, 0.0, 0.0, false, p0, d0);
    FullWriter fw = {nullptr, 0};
    RayResult R;
    trace_ray<false>(g_surfs, g_n + (int64_t)wi*n_ifc, g_wvl[wi], n_ifc, o, p0, d0, fw, R);
    for (int w = 0; w < G.n_wvls; w++) {
        ref_img[((int64_t)f*G.n_wvls + w)*2 + 0] = R.p.x;
        ref_img[((int64_t)f*G.n_wvls + w)*2 + 1] = R.p.y;
    }
    if (ref_out) { ref_out[f*2 + 0] = R.p.x; ref_out[f*2 + 1] = R.p.y; }
}

/* fp64 FMA microbenchmark: 8 independent chains per thread */
__global__ void __launch_bounds__(256) k_dfma_peak(double *out, int iters, double a, double b)
{
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3;
    double x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
        x0 = __fma_rn(x0, a, b); x1 = __fma_rn(x1, a, b);
        x2 = __fma_rn(x2, a, b); x3 = __fma_rn(x3, a, b);
        x4 = __fma_rn(x4, a, b); x5 = __fma_rn(x5, a, b);
        x6 = __fma_rn(x6, a, b); x7 = __fma_rn(x7, a, b);
    }
    double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 12345.678) out[blockIdx.x*blockDim.x + threadIdx.x] = s;
}

/* dependent-issue latency of the fp64 pipe: one warp, one chain of DFMAs, clock64 around it */
__global__ void k_dfma_latency(double *out, long long *cycles, int iters, double a, double b)
{
    double x = threadIdx.x;
    long long t0 = clock64();
#pragma unroll 16
    for (int i = 0; i < iters; i++) x = __fma_rn(x, a, b);
    long long t1 = clock64();
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
    if (x == 12345.678) out[threadIdx.x] = x;
}

/* ------------------------------------------------------------ launch helpers */
/* records (16 doubles each): n_tiles x min(chunks_per_tile, RT_MAX_GRID) x RT_WARPS, then
 * the reduce kernel's partials (n_tiles x RT_RED_SPLIT records) and tickets */
static int64_t scratch_records(const rt_grid *g)
{
    const int64_t sl = g->chunks_per_tile < RT_MAX_GRID ? g->chunks_per_tile : RT_MAX_GRID;
    return g->n_tiles*sl*RT_WARPS;
}

/* doubles before the per-item sums: records, the reduce kernel's partials, tickets */
static int64_t scratch_head_doubles(const rt_grid *g)
{
    return (scratch_records(g) + g->n_tiles*RT_RED_SPLIT)*RT_SUMMARY_DOUBLES + g->n_tiles;
}

/* Launch a persistent kernel of RT_BLOCK-thread CTAs: as many CTAs as are resident at once
 * (occupancy x SMs), but no more than work items or RT_MAX_GRID.  Returns the number of CTAs,
 * or a negative rt_error code. */
template <typename K, typename... A>
static int launch(K kernel, size_t smem, int sm_count, int64_t work_items, cudaStream_t stream,
                  const A &...args)
{
    if (smem > 48*1024)
        CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, RT_BLOCK, smem));
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)sm_count*per_sm;
    if (grid > work_items) grid = work_items;
    if (grid > RT_MAX_GRID) grid = RT_MAX_GRID;
    if (grid < 1) grid = 1;
    kernel<<<(unsigned)grid, RT_BLOCK, smem, stream>>>(args...);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return (int)grid;
}

/* f(std::true_type) or f(std::false_type): a runtime flag as a kernel template argument */
template <typename F>
static int with_bool(bool b, F f)
{
    return b ? f(std::true_type{}) : f(std::false_type{});
}

static int check_opts(const rt_table *t, const rt_opts *o)
{
    if (!o) return fail(RT_ERR_INVALID, "opts is NULL");
    if (o->wvl_idx < 0 || o->wvl_idx >= t->n_wvl) return fail(RT_ERR_INVALID, "opts.wvl_idx out of range");
    return RT_OK;
}

/* work counter of one launch: a slot of the table's ring, zeroed on the stream */
static int launch_counter(const rt_table *t, cudaStream_t stream, unsigned long long **out)
{
    rt_table *tt = const_cast<rt_table *>(t);
    *out = t->d_counters + (tt->next_counter++ % RT_COUNTERS);
    CUDA_TRY(cudaMemsetAsync(*out, 0, sizeof(unsigned long long), stream));
    return RT_OK;
}

/* 0: p,d only; 1: + normal/dst; 2: whole ray */
static int out_kind(const rt_out *out)
{
    if (out->full) return 2;
    if (out->nx || out->ny || out->nz || out->dst) return 1;
    return 0;
}

/* f(std::integral_constant<int, out_kind(out)>): the lean kernels' output kind as a template argument */
template <typename F>
static int with_out_kind(const rt_out *out, F f)
{
    switch (out_kind(out)) {
    case 0: return f(std::integral_constant<int, 0>{});
    case 1: return f(std::integral_constant<int, 1>{});
    default: return f(std::integral_constant<int, 2>{});
    }
}

static GridDev grid_dev(const rt_grid *g)
{
    GridDev G;
    G.n_wvls = g->n_wvls; G.nx = g->nx; G.ny = g->ny;
    G.apply_vignetting = g->apply_vignetting; G.flip_z_dir = g->flip_z_dir; G.paired = g->paired;
    G.eprad = g->eprad; G.z_pupil = g->z_pupil; G.foc = g->foc;
    G.fields = g->d_fields; G.wvl_idx = g->d_wvl_idx;
    G.pupil_x = g->d_pupil_x; G.pupil_y = g->d_pupil_y; G.ref_img = g->d_ref_img; G.wave = g->d_wave;
    G.rays_per_tile = g->rays_per_tile; G.chunks_per_tile = g->chunks_per_tile;
    return G;
}

/* ------------------------------------------------------------------ C ABI */
extern "C" {

int rt_abi_version(void) { return RT_ABI_VERSION; }
int32_t rt_chunk_rays(void) { return RT_BLOCK; }
const char *rt_last_error(void) { return g_err.c_str(); }
int64_t rt_launch_count(void) { return g_launches.load(); }

int rt_table_create(const rt_surface_desc *surfs, int32_t n_ifc, const double *n_by_wvl,
                    int32_t n_wvl, int32_t device, rt_table **out)
{
    if (!surfs || !n_by_wvl || !out || n_ifc < 2 || n_wvl < 1)
        return fail(RT_ERR_INVALID, "rt_table_create: bad arguments");
    for (int i = 0; i < n_ifc; i++) {
        const rt_surface_desc &s = surfs[i];
        if (s.profile < RT_PROFILE_SPHERICAL || s.profile > RT_PROFILE_THINLENS)
            return fail(RT_ERR_UNSUPPORTED, "rt_table_create: unknown profile id");
        if (s.mode < RT_MODE_TRANSMIT || s.mode > RT_MODE_PHANTOM)
            return fail(RT_ERR_UNSUPPORTED, "rt_table_create: unknown interact mode");
        if (s.n_coefs < 0 || s.n_coefs > RT_MAX_COEFS || s.n_apertures < 0 ||
            s.n_apertures > RT_MAX_APERTURES)
            return fail(RT_ERR_INVALID, "rt_table_create: coefficient / aperture count out of range");
        if (s.phase_kind < RT_PHASE_NONE || s.phase_kind > RT_PHASE_RADIAL)
            return fail(RT_ERR_UNSUPPORTED, "rt_table_create: unknown phase element kind");
        if (s.n_phase_coefs < 0 || s.n_phase_coefs > RT_MAX_PHASE_COEFS)
            return fail(RT_ERR_INVALID, "rt_table_create: phase coefficient count out of range");
    }
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    rt_table *t = new (std::nothrow) rt_table();
    if (!t) return fail(RT_ERR_NOMEM, "rt_table_create: out of host memory");
    t->device = device; t->n_ifc = n_ifc; t->n_wvl = n_wvl;
    t->sm_count = prop.multiProcessorCount;
    t->d_surfs = nullptr; t->d_n = nullptr; t->d_wvl = nullptr; t->has_phase = false;
    t->stage_bytes = (size_t)n_ifc*sizeof(rt_surface_desc) + (size_t)n_ifc*n_wvl*sizeof(double);
    t->stage = t->stage_bytes <= RT_MAX_STAGE_BYTES - RT_ACC_BYTES;
    t->lean_bytes = (size_t)n_ifc*sizeof(LeanSurf) + (size_t)n_ifc*n_wvl*sizeof(LeanIdx);
    t->lean = t->lean_bytes <= RT_MAX_STAGE_BYTES - RT_ACC_BYTES;
    t->lean_poly = false;
    for (int i = 0; i < n_ifc; i++) {
        const rt_surface_desc &s = surfs[i];
        if (s.has_tfrm != 0 || s.n_apertures != 0) t->lean = false;
        if (s.phase_kind != RT_PHASE_NONE || s.profile == RT_PROFILE_THINLENS) { t->lean = false; t->has_phase = true; }
        if (s.profile > RT_PROFILE_CONIC) t->lean_poly = true;
    }
    if (t->lean_poly) {
        t->lean_bytes += (size_t)n_ifc*sizeof(LeanPoly);
        if (t->lean_bytes > RT_MAX_STAGE_BYTES - RT_ACC_BYTES) t->lean = false;
    }
    if (getenv("B200RT_NO_LEAN")) t->lean = false;
    t->d_counters = nullptr; t->next_counter = 0;
    {
        const rt_surface_desc &k = surfs[n_ifc >= 2 ? n_ifc - 2 : 0];
        t->wave_ok = n_ifc >= 3 && k.has_tfrm == 0 && k.t[0] == 0.0 && k.t[1] == 0.0;
    }
    cudaError_t e = cudaMalloc(&t->d_surfs, (size_t)n_ifc*sizeof(rt_surface_desc));
    if (e == cudaSuccess) e = cudaMalloc(&t->d_n, (size_t)n_ifc*n_wvl*sizeof(double));
    if (e == cudaSuccess)
        e = cudaMemcpy(t->d_surfs, surfs, (size_t)n_ifc*sizeof(rt_surface_desc), cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
        e = cudaMemcpy(t->d_n, n_by_wvl, (size_t)n_ifc*n_wvl*sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&t->d_wvl, (size_t)n_wvl*sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&t->d_counters, RT_COUNTERS*sizeof(unsigned long long));
    if (e == cudaSuccess) {
        std::vector<double> nanv((size_t)n_wvl, (double)NAN);
        e = cudaMemcpy(t->d_wvl, nanv.data(), (size_t)n_wvl*sizeof(double), cudaMemcpyHostToDevice);
    }
    /* pageable copies: see rt_grid_create */
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
    if (e != cudaSuccess) {
        cudaFree(t->d_surfs); cudaFree(t->d_n); cudaFree(t->d_wvl); cudaFree(t->d_counters); delete t;
        return fail(RT_ERR_CUDA, "rt_table_create: %s", cudaGetErrorString(e));
    }
    *out = t;
    return RT_OK;
}

int rt_table_destroy(rt_table *t)
{
    if (!t) return RT_OK;
    DeviceGuard guard(t->device);
    cudaFree(t->d_surfs);
    cudaFree(t->d_n);
    cudaFree(t->d_wvl);
    cudaFree(t->d_counters);
    delete t;
    return RT_OK;
}

int rt_table_set_wavelengths(rt_table *t, const double *wvl_nm)
{
    if (!t || !wvl_nm) return fail(RT_ERR_INVALID, "rt_table_set_wavelengths: bad arguments");
    DeviceGuard guard(t->device);
    CUDA_TRY(cudaMemcpy(t->d_wvl, wvl_nm, (size_t)t->n_wvl*sizeof(double), cudaMemcpyHostToDevice));
    CUDA_TRY(cudaStreamSynchronize(cudaStreamLegacy));
    return RT_OK;
}

int rt_table_dims(const rt_table *t, int32_t *n_ifc, int32_t *n_wvl, int32_t *device)
{
    if (!t) return fail(RT_ERR_INVALID, "rt_table_dims: NULL table");
    if (n_ifc) *n_ifc = t->n_ifc;
    if (n_wvl) *n_wvl = t->n_wvl;
    if (device) *device = t->device;
    return RT_OK;
}

int rt_trace_bundle(const rt_table *t, int64_t n_rays, const double *px, const double *py,
                    const double *pz, const double *dx, const double *dy, const double *dz,
                    const int32_t *wvl_idx, const rt_opts *o, const rt_out *out, void *stream)
{
    if (!t || !out || n_rays < 0 || !px || !py || !pz || !dx || !dy || !dz)
        return fail(RT_ERR_INVALID, "rt_trace_bundle: bad arguments");
    int rc = check_opts(t, o);
    if (rc) return rc;
    if (n_rays == 0) return RT_OK;
    if (out->full && out->full_stride < n_rays)
        return fail(RT_ERR_INVALID, "rt_trace_bundle: full_stride < n_rays");
    DeviceGuard guard(t->device);
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t chunks = (n_rays + RT_BLOCK - 1)/RT_BLOCK;
    int grid;
    if (t->lean) {                  /* (lean kernels: no phase elements, no wavelengths) */
        grid = with_out_kind(out, [&](auto kind) {
            return with_bool(t->lean_poly, [&](auto poly) {
                return launch(k_trace_bundle_lean<kind, poly>, t->lean_bytes, t->sm_count, chunks, s,
                              t->d_surfs, t->d_n, t->n_ifc, t->n_wvl, n_rays, px, py, pz, dx, dy, dz,
                              wvl_idx, *o, *out);
            });
        });
    } else {
        grid = with_bool(out->full != nullptr, [&](auto full) {
            return with_bool(t->stage, [&](auto stage) {
                return launch(k_trace_bundle<full, stage>, stage ? t->stage_bytes : 0, t->sm_count, chunks, s,
                              t->d_surfs, t->d_n, t->n_ifc, t->n_wvl, n_rays, px, py, pz, dx, dy, dz,
                              wvl_idx, *o, *out, t->d_wvl);
            });
        });
    }
    return grid < 0 ? grid : RT_OK;
}

int rt_grid_destroy(rt_grid *g)
{
    if (!g) return RT_OK;
    DeviceGuard guard(g->device);
    if (g->uploaded) { cudaEventSynchronize(g->uploaded); cudaEventDestroy(g->uploaded); }
    if (g->side_ok) {
        for (int k = 0; k < 2; k++) {
            cudaStreamSynchronize(g->side[k]); cudaStreamDestroy(g->side[k]); cudaEventDestroy(g->ev_side[k]);
        }
        cudaEventDestroy(g->ev_in);
    }
    cudaFree(g->d_block);
    cudaFreeHost(g->h_stage);
    delete g;
    return RT_OK;
}

static bool grid_spec_ok(const rt_grid_spec *spec)
{
    return spec && spec->n_fields >= 1 && spec->n_wvls >= 1 && spec->nx >= 1 && spec->ny >= 1 &&
           spec->fields && spec->wvl_idx && spec->pupil_x && spec->pupil_y &&
           !(spec->paired && spec->ny != 1) && spec->pupil_kind >= RT_PUPIL_EPD &&
           spec->pupil_kind <= RT_PUPIL_WIDE;
}

/* scalars of the description + the arrays into the pinned staging block (layout fixed at create) */
static void grid_fill(rt_grid *g, const rt_grid_spec *spec)
{
    g->apply_vignetting = spec->apply_vignetting; g->flip_z_dir = spec->flip_z_dir;
    g->pupil_kind = spec->pupil_kind;
    g->eprad = spec->eprad; g->z_pupil = spec->z_pupil; g->foc = spec->foc;
    unsigned char *st = g->h_stage;
    memcpy(st + g->o_fields, spec->fields, g->b_fields);
    memcpy(st + g->o_px, spec->pupil_x, g->b_px);
    memcpy(st + g->o_py, spec->pupil_y, g->b_py);
    if (spec->ref_img) memcpy(st + g->o_ref, spec->ref_img, g->b_ref);
    else memset(st + g->o_ref, 0, g->b_ref);
    if (g->b_wave) memcpy(st + g->o_wave, spec->wave, g->b_wave);
    memcpy(st + g->o_wvl, spec->wvl_idx, (size_t)g->n_wvls*sizeof(int32_t));
    g->h_wvl_idx.assign(spec->wvl_idx, spec->wvl_idx + g->n_wvls);
}

/* All arrays of the description live in ONE device allocation and travel as ONE copy from a
 * pinned staging block owned by the handle; rt_grid_update() re-uses both, so an analysis that
 * is called repeatedly pays one small asynchronous copy per call and no allocation. */
int rt_grid_create(const rt_grid_spec *spec, int32_t device, rt_grid **out)
{
    if (!grid_spec_ok(spec) || !out) return fail(RT_ERR_INVALID, "rt_grid_create: bad arguments");
    DeviceGuard guard(device);
    rt_grid *g = new (std::nothrow) rt_grid();
    if (!g) return fail(RT_ERR_NOMEM, "rt_grid_create: out of host memory");
    g->device = device;
    g->n_fields = spec->n_fields; g->n_wvls = spec->n_wvls; g->nx = spec->nx; g->ny = spec->ny;
    g->paired = spec->paired;
    g->rays_per_tile = (int64_t)spec->nx*spec->ny;
    g->chunks_per_tile = (g->rays_per_tile + RT_BLOCK - 1)/RT_BLOCK;
    g->n_tiles = (int64_t)spec->n_fields*spec->n_wvls;
    g->n_chunks = g->n_tiles*g->chunks_per_tile;
    g->n_rays = g->n_tiles*g->rays_per_tile;

    const size_t nf = (size_t)spec->n_fields, nw = (size_t)spec->n_wvls;
    g->b_fields = nf*sizeof(rt_field_desc);
    g->b_px = nf*spec->nx*sizeof(double);
    g->b_py = nf*(spec->paired ? spec->nx : spec->ny)*sizeof(double);
    g->b_ref = (size_t)g->n_tiles*2*sizeof(double);          /* zeros when spec->ref_img is NULL */
    g->b_wave = spec->wave ? (size_t)g->n_tiles*RT_WAVE_DOUBLES*sizeof(double) : 0;
    const size_t b_wvl = (nw*sizeof(int32_t) + 7)/8*8;
    g->o_fields = 0; g->o_px = g->o_fields + g->b_fields; g->o_py = g->o_px + g->b_px;
    g->o_ref = g->o_py + g->b_py; g->o_wave = g->o_ref + g->b_ref; g->o_wvl = g->o_wave + g->b_wave;
    g->total = g->o_wvl + b_wvl;
    g->d_block = nullptr; g->h_stage = nullptr; g->uploaded = nullptr; g->side_ok = false;
    cudaError_t e = cudaMallocHost((void **)&g->h_stage, g->total);
    if (e == cudaSuccess) e = cudaMalloc(&g->d_block, g->total);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->uploaded, cudaEventDisableTiming);
    if (e == cudaSuccess) {
        grid_fill(g, spec);
        e = cudaMemcpy(g->d_block, g->h_stage, g->total, cudaMemcpyHostToDevice);
    }
    /* callers launch on non-blocking streams: make the block visible to every stream */
    if (e == cudaSuccess) e = cudaStreamSynchronize(cudaStreamLegacy);
    if (e != cudaSuccess) {
        if (g->uploaded) cudaEventDestroy(g->uploaded);
        cudaFree(g->d_block);
        cudaFreeHost(g->h_stage);
        delete g;
        return fail(RT_ERR_CUDA, "rt_grid_create: %s", cudaGetErrorString(e));
    }
    unsigned char *base = (unsigned char *)g->d_block;
    g->d_fields = (rt_field_desc *)(base + g->o_fields);
    g->d_pupil_x = (double *)(base + g->o_px);
    g->d_pupil_y = (double *)(base + g->o_py);
    g->d_ref_img = (double *)(base + g->o_ref);
    g->d_wave = g->b_wave ? (double *)(base + g->o_wave) : nullptr;
    g->d_wvl_idx = (int32_t *)(base + g->o_wvl);
    *out = g;
    return RT_OK;
}

int rt_grid_update(rt_grid *g, const rt_grid_spec *spec, void *stream)
{
    if (!g || !grid_spec_ok(spec)) return fail(RT_ERR_INVALID, "rt_grid_update: bad arguments");
    if (spec->n_fields != g->n_fields || spec->n_wvls != g->n_wvls || spec->nx != g->nx ||
        spec->ny != g->ny || spec->paired != g->paired || (spec->wave != nullptr) != (g->b_wave != 0))
        return fail(RT_ERR_INVALID, "rt_grid_update: the new description has a different shape");
    DeviceGuard guard(g->device);
    CUDA_TRY(cudaEventSynchronize(g->uploaded));     /* the previous copy has left the staging block */
    grid_fill(g, spec);
    CUDA_TRY(cudaMemcpyAsync(g->d_block, g->h_stage, g->total, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    CUDA_TRY(cudaEventRecord(g->uploaded, (cudaStream_t)stream));
    return RT_OK;
}

int rt_grid_dims(const rt_grid *g, int64_t *n_rays, int64_t *n_chunks, int32_t *chunk_rays)
{
    if (!g) return fail(RT_ERR_INVALID, "rt_grid_dims: NULL grid");
    if (n_rays) *n_rays = g->n_rays;
    if (n_chunks) *n_chunks = g->n_chunks;
    if (chunk_rays) *chunk_rays = RT_BLOCK;
    return RT_OK;
}

int64_t rt_grid_scratch_bytes(const rt_grid *g, int64_t chunk_begin, int64_t chunk_end)
{
    if (!g || chunk_end < chunk_begin) return 0;
    return (scratch_head_doubles(g) + (chunk_end - chunk_begin)*RT_WARPS*RT_ITEM_SUMS)*(int64_t)sizeof(double);
}

int rt_trace_grid(const rt_table *t, const rt_grid *g, int64_t chunk_begin, int64_t chunk_end,
                  const rt_opts *o, const rt_out *out, double *summary, void *scratch, void *stream)
{
    if (!t || !g || !out) return fail(RT_ERR_INVALID, "rt_trace_grid: bad arguments");
    if (t->device != g->device) return fail(RT_ERR_INVALID, "rt_trace_grid: table and grid on different devices");
    if (chunk_begin < 0 || chunk_end > g->n_chunks || chunk_end < chunk_begin)
        return fail(RT_ERR_INVALID, "rt_trace_grid: chunk range out of bounds");
    if (summary && !scratch) return fail(RT_ERR_INVALID, "rt_trace_grid: summary needs scratch");
    int rc = check_opts(t, o);
    if (rc) return rc;
    DeviceGuard guard(t->device);
    cudaStream_t s = (cudaStream_t)stream;
    for (int32_t wi : g->h_wvl_idx)
        if (wi < 0 || wi >= t->n_wvl)
            return fail(RT_ERR_INVALID, "rt_trace_grid: the grid's wvl_idx is out of range for this table");
    if (summary && chunk_begin == chunk_end) {
        /* an empty shard contributes the identity of every column (min / max: +-inf) */
        const int64_t n = g->n_tiles*RT_SUMMARY_DOUBLES;
        k_summary_identity<<<(unsigned)((n + 255)/256), 256, 0, s>>>(summary, n);
        g_launches++;
        CUDA_TRY(cudaGetLastError());
    }
    if (chunk_begin == chunk_end) return RT_OK;
    const GridDev G = grid_dev(g);
    double *scr = (double *)scratch;
    if (summary)
        CUDA_TRY(cudaMemsetAsync(scr, 0, (size_t)rt_grid_scratch_bytes(g, chunk_begin, chunk_end), s));
    const bool summ = summary != nullptr;
    const bool wave = out->opd != nullptr;
    /* angular pupil specifications are generated by the general kernels only (rt_grid.cuh) */
    const bool lean = t->lean && g->pupil_kind == RT_PUPIL_EPD;
    if (wave) {
        if (!g->d_wave) return fail(RT_ERR_INVALID, "rt_trace_grid: out.opd needs rt_grid_spec.wave");
        if (out_kind(out) != 0) return fail(RT_ERR_UNSUPPORTED, "rt_trace_grid: opd cannot be combined with normals / whole rays");
        if (!t->wave_ok)
            return fail(RT_ERR_UNSUPPORTED, "rt_trace_grid: opd needs >= 3 interfaces and no decenter on the last one before the image");
    }
    unsigned long long *wc;
    rc = launch_counter(t, s, &wc);
    if (rc) return rc;
    double *item_sums = summ ? scr + scratch_head_doubles(g) : nullptr;
    const int64_t cb = chunk_begin, ce = chunk_end;
    auto launch_lean = [&](auto kind, auto wave_c) {
        return with_bool(summ, [&](auto summ_c) {
            return with_bool(t->lean_poly, [&](auto poly) {
                return launch(k_trace_grid_lean<kind, summ_c, wave_c, poly>,
                              t->lean_bytes + (summ_c ? RT_ACC_BYTES : 0), t->sm_count, ce - cb, s,
                              t->d_surfs, t->d_n, t->n_ifc, t->n_wvl, G, cb, ce, *o, *out, scr, wc, item_sums);
            });
        });
    };
    auto launch_general = [&](auto full, auto wave_c) {
        return with_bool(summ, [&](auto summ_c) {
            return with_bool(t->stage, [&](auto stage) {
                return launch(k_trace_grid<full, summ_c, stage, wave_c>,
                              (stage ? t->stage_bytes : 0) + (summ_c ? RT_ACC_BYTES : 0), t->sm_count, ce - cb, s,
                              t->d_surfs, t->d_n, t->n_ifc, t->n_wvl, G, cb, ce, *o, *out, scr, t->d_wvl,
                              g->pupil_kind, wc, item_sums);
            });
        });
    };
    int grid;
    if (wave)
        grid = lean ? launch_lean(std::integral_constant<int, 0>{}, std::true_type{})
                    : launch_general(std::false_type{}, std::true_type{});
    else if (lean)
        grid = with_out_kind(out, [&](auto kind) { return launch_lean(kind, std::false_type{}); });
    else
        grid = with_bool(out->full != nullptr, [&](auto full) { return launch_general(full, std::false_type{}); });
    if (grid < 0) return grid;
    if (summ) {
        const int64_t recs = scratch_records(g);
        double *partials = scr + recs*RT_SUMMARY_DOUBLES;
        unsigned int *tickets = (unsigned int *)(partials + g->n_tiles*RT_RED_SPLIT*RT_SUMMARY_DOUBLES);
        /* with chunk slots the trace kernel wrote the sums into the records (grid_chunk_loop) */
        const bool chunk_slots = g->chunks_per_tile <= grid;
        k_reduce_summary<<<(unsigned)(g->n_tiles*RT_RED_SPLIT), RT_RED_THREADS, 0, s>>>(
            scr, recs/g->n_tiles, partials, tickets, summary, chunk_slots ? nullptr : item_sums,
            chunk_begin, chunk_end, g->chunks_per_tile);
        g_launches++;
        CUDA_TRY(cudaGetLastError());
    }
    return RT_OK;
}

static int64_t first_ray_of_chunk(const rt_grid *g, int64_t c)
{
    const int64_t tile = c/g->chunks_per_tile, lc = c - tile*g->chunks_per_tile;
    const int64_t in_tile = lc*RT_BLOCK < g->rays_per_tile ? lc*RT_BLOCK : g->rays_per_tile;
    return tile*g->rays_per_tile + in_tile;
}

int64_t rt_trace_grid_to_host_scratch_bytes(const rt_grid *g, int32_t n_pieces)
{
    if (!g || n_pieces < 1) return 0;
    return 2*rt_grid_scratch_bytes(g, 0, g->n_chunks) +
           (int64_t)n_pieces*g->n_tiles*RT_SUMMARY_DOUBLES*(int64_t)sizeof(double);
}

/* The grid analyses' data path in one call: the chunk range is traced in n_pieces launches
 * alternating between two internal streams, and each piece's aberrations (NaN-coded status) go
 * device -> host right behind its trace, so the copy of one piece overlaps the trace of the
 * next without the caller issuing anything per piece. */
int rt_trace_grid_to_host(const rt_table *t, rt_grid *g, int64_t chunk_begin, int64_t chunk_end,
                          const rt_opts *o, double *d_abr_x, double *d_abr_y, double *h_abr_x,
                          double *h_abr_y, double *summary, void *scratch, int32_t n_pieces, void *stream)
{
    if (!t || !g || !d_abr_x || !d_abr_y || !h_abr_x || !h_abr_y || !scratch || n_pieces < 1)
        return fail(RT_ERR_INVALID, "rt_trace_grid_to_host: bad arguments");
    if (chunk_begin < 0 || chunk_end > g->n_chunks || chunk_end < chunk_begin)
        return fail(RT_ERR_INVALID, "rt_trace_grid_to_host: chunk range out of bounds");
    DeviceGuard guard(t->device);
    cudaStream_t s = (cudaStream_t)stream;
    if (!g->side_ok) {
        for (int k = 0; k < 2; k++) {
            CUDA_TRY(cudaStreamCreateWithFlags(&g->side[k], cudaStreamNonBlocking));
            CUDA_TRY(cudaEventCreateWithFlags(&g->ev_side[k], cudaEventDisableTiming));
        }
        CUDA_TRY(cudaEventCreateWithFlags(&g->ev_in, cudaEventDisableTiming));
        g->side_ok = true;
    }
    if (n_pieces > chunk_end - chunk_begin) n_pieces = (int32_t)(chunk_end - chunk_begin);
    if (n_pieces < 1) n_pieces = 1;
    const int64_t sb = rt_grid_scratch_bytes(g, 0, g->n_chunks);
    unsigned char *scr = (unsigned char *)scratch;
    double *partials = (double *)(scr + 2*sb);
    const int64_t tile_doubles = g->n_tiles*RT_SUMMARY_DOUBLES;
    const int64_t base = first_ray_of_chunk(g, chunk_begin);
    CUDA_TRY(cudaEventRecord(g->ev_in, s));                  /* grid upload, chief rays ... */
    for (int k = 0; k < 2; k++) CUDA_TRY(cudaStreamWaitEvent(g->side[k], g->ev_in, 0));
    for (int i = 0; i < n_pieces; i++) {
        const int64_t cb = chunk_begin + (chunk_end - chunk_begin)*i/n_pieces;
        const int64_t ce = chunk_begin + (chunk_end - chunk_begin)*(i + 1)/n_pieces;
        const int64_t a = first_ray_of_chunk(g, cb) - base, n = first_ray_of_chunk(g, ce) - first_ray_of_chunk(g, cb);
        cudaStream_t ss = g->side[i & 1];
        rt_out out;
        memset(&out, 0, sizeof out);
        out.abr_x = d_abr_x + a; out.abr_y = d_abr_y + a;
        out.flags = RT_OUT_ABR_NAN_STATUS;
        int rc = rt_trace_grid(t, g, cb, ce, o, &out, summary ? partials + i*tile_doubles : nullptr,
                               scr + (i & 1)*sb, ss);
        if (rc) return rc;
        CUDA_TRY(cudaMemcpyAsync(h_abr_x + a, d_abr_x + a, (size_t)n*sizeof(double), cudaMemcpyDeviceToHost, ss));
        CUDA_TRY(cudaMemcpyAsync(h_abr_y + a, d_abr_y + a, (size_t)n*sizeof(double), cudaMemcpyDeviceToHost, ss));
    }
    for (int k = 0; k < 2; k++) {
        CUDA_TRY(cudaEventRecord(g->ev_side[k], g->side[k]));
        CUDA_TRY(cudaStreamWaitEvent(s, g->ev_side[k], 0));
    }
    if (summary) return rt_combine_summaries(partials, n_pieces, g->n_tiles, summary, stream);
    return RT_OK;
}

int rt_grid_chief_ref(const rt_table *t, rt_grid *g, int32_t wvl_idx, double *ref_out, void *stream)
{
    if (!t || !g) return fail(RT_ERR_INVALID, "rt_grid_chief_ref: bad arguments");
    if (t->device != g->device) return fail(RT_ERR_INVALID, "rt_grid_chief_ref: table and grid on different devices");
    if (wvl_idx < 0 || wvl_idx >= t->n_wvl) return fail(RT_ERR_INVALID, "rt_grid_chief_ref: wvl_idx out of range");
    DeviceGuard guard(t->device);
    rt_opts o;
    o.eps = 1.0e-12; o.pt_inside_fuzz = -1.0; o.check_apertures = 0; o.intersect_obj = 1;
    o.filter_out_phantoms = 0; o.first_surf = 1; o.last_surf = t->n_ifc - 2; o.wvl_idx = wvl_idx;
    const int threads = 32, blocks = (g->n_fields + threads - 1)/threads;
    k_chief_ref<<<blocks, threads, 0, (cudaStream_t)stream>>>(t->d_surfs, t->d_n, t->n_ifc, grid_dev(g),
                                                              g->n_fields, g->pupil_kind, wvl_idx, t->d_wvl,
                                                              o, g->d_ref_img, ref_out);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

int rt_combine_summaries(const double *parts, int32_t n_parts, int64_t n_tiles, double *out, void *stream)
{
    if (!parts || !out || n_parts < 1 || n_tiles < 0)
        return fail(RT_ERR_INVALID, "rt_combine_summaries: bad arguments");
    if (n_tiles == 0) return RT_OK;
    const int64_t n = n_tiles*RT_SUMMARY_DOUBLES;
    k_combine_summaries<<<(unsigned)((n + 255)/256), 256, 0, (cudaStream_t)stream>>>(parts, n_parts, n, out);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RT_OK;
}

/* fp64 vector-pipe peak, measured with a DFMA chain kernel: the roofline
 * denominator for the register-resident trace (DESIGN.md "roofline"). */
int rt_measure_fp64_peak(int32_t device, double *tflops)
{
    if (!tflops) return fail(RT_ERR_INVALID, "rt_measure_fp64_peak: NULL output");
    DeviceGuard guard(device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount*8, iters = 1 << 14;
    double *d_out;
    CUDA_TRY(cudaMalloc(&d_out, (size_t)blocks*256*sizeof(double)));
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        CUDA_TRY(cudaEventRecord(e0));
        k_dfma_peak<<<blocks, 256>>>(d_out, iters, 0.999999, 1e-9);
        g_launches++;
        CUDA_TRY(cudaEventRecord(e1));
        CUDA_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        double fl = 2.0*8.0*(double)iters*256.0*blocks;
        double tf = fl/(ms*1e-3)/1e12;
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d_out);
    *tflops = best;
    return RT_OK;
}

/* Cycles between two DEPENDENT fp64 FMAs of one warp (the latency that the per-ray chains of
 * the trace kernels expose; DESIGN.md "what bounds the kernel"). */
int rt_measure_fp64_latency(int32_t device, double *cycles_per_dependent_dfma)
{
    if (!cycles_per_dependent_dfma) return fail(RT_ERR_INVALID, "rt_measure_fp64_latency: NULL output");
    DeviceGuard guard(device);
    double *d_out; long long *d_cyc;
    CUDA_TRY(cudaMalloc(&d_out, 32*sizeof(double)));
    CUDA_TRY(cudaMalloc(&d_cyc, sizeof(long long)));
    const int iters = 1 << 14;
    long long best = -1;
    for (int rep = 0; rep < 3; rep++) {
        k_dfma_latency<<<1, 32>>>(d_out, d_cyc, iters, 0.999999, 1e-9);
        g_launches++;
        long long c = 0;
        CUDA_TRY(cudaMemcpy(&c, d_cyc, sizeof c, cudaMemcpyDeviceToHost));
        if (best < 0 || c < best) best = c;
    }
    cudaFree(d_out); cudaFree(d_cyc);
    *cycles_per_dependent_dfma = (double)best/iters;
    return RT_OK;
}

/* Self-test of the shared-reciprocal division used by the lean kernels:
 * n_blocks x 256 threads x n_per_thread random operand sets (3 quotients + one
 * normalisation each) compared bit-for-bit with the IEEE `/`.  *mismatches
 * must come back 0. */
int rt_selftest_division(int32_t device, int32_t n_blocks, int64_t n_per_thread, uint64_t seed,
                         uint64_t *mismatches)
{
    if (!mismatches || n_blocks < 1 || n_per_thread < 1)
        return fail(RT_ERR_INVALID, "rt_selftest_division: bad arguments");
    DeviceGuard guard(device);
    unsigned long long *d_bad;
    CUDA_TRY(cudaMalloc(&d_bad, sizeof(unsigned long long)));
    CUDA_TRY(cudaMemset(d_bad, 0, sizeof(unsigned long long)));
    k_selftest_division<<<n_blocks, 256>>>(seed, n_per_thread, d_bad);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    unsigned long long bad = 0;
    CUDA_TRY(cudaMemcpy(&bad, d_bad, sizeof bad, cudaMemcpyDeviceToHost));
    cudaFree(d_bad);
    *mismatches = bad;
    return RT_OK;
}

}  /* extern "C" */
