// warp_tma.cu - K1s: the CPN.align tail (affine grid -> bilinear warp of RGB + bilinear
// visibility > 0.5 + v_map) as a PERSISTENT kernel whose reference tiles are staged in shared
// memory by TMA.
//
// Replaces CPN.align tail, master_thesis/model_cpn.py:75-89 (a3): F.affine_grid (:75-77),
// F.grid_sample of the frames (:79-83) and of 1 - masks (:84-88), v_maps (:89).
//
// Why (evidence in profiles/r1_experiments.md): the direct-gather kernel (warp.cu) peaks near
// 46 % of HBM peak.  Its CTAs live for one 128 x 2 pixel strip: every CTA pays a dependent
// chain "theta load -> coordinates -> gathers -> stores" with nothing in flight during the first
// and last links, all CTAs of a wave are in the same phase, and more loads in flight per thread
// (ptxas scheduling sweep) or fewer instructions per pixel (row loops) changed nothing.  Here the
// memory pipeline is decoupled from the arithmetic:
//   * one CTA per SM, persistent over 32 x 32 output tiles (static round-robin);
//   * warp 16 = producer: for the tile kStages ahead it evaluates the affine map at the four
//     corner pixels with EXACTLY the consumers' arithmetic (every step is monotone in the column
//     and in the row index, so the corners bound the tile's taps), and issues two TMA box loads
//     (RGB planes: 5-D map, one instruction; mask plane: 4-D map) of kBox x kBox source pixels
//     into the stage, plus the 32 x 32 tile of the target mask (v_map needs it; as a per-thread
//     global load its DRAM latency bounded every warp's time per tile: 24.8 us, no better than
//     the strip kernel); TMA zero-fills outside the frame = grid_sample's zero padding;
//   * warps 0..15 = consumers: 2 rows x 32 columns each; coordinates from per-CTA tables of the
//     linspace base grid (the IEEE division of align_corners=False is paid once per CTA, not per
//     thread), 16 LDS with immediate offsets per pixel, interpolation in the pinned order,
//     128 B-coalesced streaming stores.  Full/empty mbarriers per stage; no CTA-wide barrier in
//     the loop, so the 16 warps drift apart and overlap each other's phases.
// A tile whose footprint does not fit the box (|theta| far from identity, NaN) is flagged by the
// producer and its pixels take the direct-gather path of warp.cu inside the same kernel.
// Results are bit-identical to warp_fwd_kernel: same operations in the same order on the same
// values (tests/test_gpu_parity.py compares the two paths as well as the oracle).
#include "mt_common.cuh"
#include "mt_tma.cuh"
#include "warp_common.cuh"

namespace mt {
namespace {

constexpr int kTileW = 32, kTileH = 32;  // output tile
constexpr int kBox = 48;                 // staged source box: kBox x kBox pixels per plane
constexpr int kStages = 5;               // ring of 40 KB stages
constexpr int kConsWarps = kTileW / 2;   // consumer warps of 16 x 4 pixels each, + one producer warp
constexpr int kStagedThreads = (kConsWarps + 1) * 32;
constexpr int kMaxTable = 1024;          // W, H <= 1024 (tables of the base grid in shared memory)

struct TileDesc {  // written by the producer, read by the consumers after the full barrier
    int flags;     // bit 0: staged in smem; bit 1: every tap of the tile is inside the frame
    int bx0, by0;  // frame coordinates of the box origin
    int b, f, n;   // sample, reference frame, n = b * F + f
    int tx, ty;
    float th[6];
    int pad[2];
};
static_assert(sizeof(TileDesc) == 64, "TileDesc is read as four 16 B words");

struct WarpStagedArgs {
    const float *x, *vis, *theta, *m_target;
    float *x_al, *v_al, *v_map;
    int x_sb, x_sc, x_sf, vis_sb, vis_sf, mt_sb, xa_sb, xa_sc, xa_sf;
    int F, P, tiles_x, tiles_per_frame, n_tiles;
    Sampler sp;
};

constexpr int kStagedSmem = kStages * (4 * kBox * kBox + kTileW * kTileH) * 4 + 2 * kMaxTable * 4 +
                            kStages * (int)sizeof(TileDesc) + 2 * kStages * 8 + 128;
static_assert(kStagedSmem <= 227 * 1024, "stage ring exceeds the shared memory of an SM");

__device__ __forceinline__ float unnorm_t(float g, float sf, bool ac) { return unnormalize(g, sf, ac); }

// AC: align_corners; FM: `vis` holds masks (v = 1 - m inside the frame, 0 outside)
template <bool AC, bool FM>
__global__ void __launch_bounds__(kStagedThreads, 1)
warp_staged_kernel(const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_v,
                   const __grid_constant__ CUtensorMap map_t, const WarpStagedArgs a) {
    static_assert(kBox % 32 == 16, "a source row must start 16 banks after the previous one (see the lane mapping)");
    constexpr int kPlane = kBox * kBox;
    constexpr int kStageFloats = 4 * kPlane + kTileW * kTileH;  // RGB + mask boxes, target-mask tile
    constexpr uint32_t kMtBytes = kTileW * kTileH * 4u;
    // 128 B alignment (TMA destination) comes from the declaration: a manual round-up through
    // uintptr_t makes the compiler lose the shared address space (generic LD/ST instead of LDS/STS)
    extern __shared__ __align__(128) uint8_t smem_raw[];
    float *stage0 = reinterpret_cast<float *>(smem_raw);
    float *s_bx = stage0 + kStages * kStageFloats;
    float *s_by = s_bx + kMaxTable;
    TileDesc *desc = reinterpret_cast<TileDesc *>(s_by + kMaxTable);
    uint64_t *full = reinterpret_cast<uint64_t *>(desc + kStages), *empty = full + kStages;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int W = a.sp.W, H = a.sp.H;

    // ---- on-chip setup: overlaps the tail of the previous kernel (PDL) ----
    for (int i = threadIdx.x; i < W; i += kStagedThreads) s_bx[i] = base_coord(i, W, a.sp.stepx, AC);
    for (int i = threadIdx.x; i < H; i += kStagedThreads) s_by[i] = base_coord(i, H, a.sp.stepy, AC);
    if (threadIdx.x == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_x) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_v) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_t) : "memory");
        for (int s = 0; s < kStages; ++s) {
            mbar_init(smem_u32(full + s), 1);
            mbar_init(smem_u32(empty + s), kConsWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // no launch_dependents: this kernel holds ~200 KB of shared memory per SM and leaves the trigger to its exit
    // (see pdl_sync; cfg5 step 121.8 -> 109.8 us: the streaming kernels behind it get their L1 back)
    pdl_wait();

    const float wmax = a.sp.wmax, hmax = a.sp.hmax;

    // ---- producer duty (lane 0 of the producer warp) ----
    // The descriptor of a tile: theta load, two integer divisions, four corner evaluations.
    auto prepare = [&](int t) {
        TileDesc d;
        const int n = t / a.tiles_per_frame, r = t - n * a.tiles_per_frame;
        const int ty = r / a.tiles_x, tx = r - ty * a.tiles_x;
#pragma unroll
        for (int j = 0; j < 6; ++j) d.th[j] = __ldg(a.theta + n * 6 + j);
        const int b = n / a.F, f = n - b * a.F;
        const int xs[2] = {tx * kTileW, min(tx * kTileW + kTileW - 1, W - 1)};
        const int ys[2] = {ty * kTileH, min(ty * kTileH + kTileH - 1, H - 1)};
        float xlo = 3.0e38f, xhi = -3.0e38f, ylo = 3.0e38f, yhi = -3.0e38f;
        bool finite = true;
#pragma unroll
        for (int cy = 0; cy < 2; ++cy) {
#pragma unroll
            for (int cx = 0; cx < 2; ++cx) {
                const float bx = s_bx[xs[cx]], by = s_by[ys[cy]];
                // identical to the consumers' arithmetic below
                const float gx = __fadd_rn(__fmaf_rn(by, d.th[1], __fmul_rn(bx, d.th[0])), d.th[2]);
                const float gy = __fadd_rn(__fmaf_rn(by, d.th[4], __fmul_rn(bx, d.th[3])), d.th[5]);
                const float xw = floorf(unnorm_t(gx, a.sp.sfx, AC)), yn = floorf(unnorm_t(gy, a.sp.sfy, AC));
                finite = finite && (fabsf(xw) <= 1.0e6f) && (fabsf(yn) <= 1.0e6f);  // false for NaN / inf
                xlo = fminf(xlo, xw); xhi = fmaxf(xhi, xw);
                ylo = fminf(ylo, yn); yhi = fmaxf(yhi, yn);
            }
        }
        // taps span [xlo, xhi + 1] x [ylo, yhi + 1].  TMA needs the innermost start coordinate on a
        // 16 B boundary (an unaligned one faults with "illegal instruction", tools/tma_probe.cu), so
        // the box origin is xlo rounded down to a multiple of 4 pixels (two's complement: also for
        // negative coordinates)
        const int bx0 = finite ? ((int)xlo & ~3) : 0, by0 = finite ? (int)ylo : 0;
        const bool fits = finite && ((int)xhi + 2 - bx0 <= kBox) && ((int)yhi + 2 - by0 <= kBox);
        const bool inside = fits && xlo >= 0.0f && xhi + 1.0f <= wmax && ylo >= 0.0f && yhi + 1.0f <= hmax;
        d.flags = (fits ? 1 : 0) | (inside ? 2 : 0);
        d.bx0 = bx0; d.by0 = by0;
        d.b = b; d.f = f; d.n = n; d.tx = tx; d.ty = ty;
        d.pad[0] = d.pad[1] = 0;
        return d;
    };
    // i-th tile of this CTA -> stage i % kStages (waits until the consumers have released it)
    auto issue = [&](int i, const TileDesc &d) {
        const int s = i % kStages;
        const uint32_t ph = (uint32_t)(i / kStages) & 1u;
        mbar_wait(smem_u32(empty + s), ph ^ 1u);
        desc[s] = d;
        const bool fits = (d.flags & 1) != 0;
        float *dst = stage0 + s * kStageFloats;
        mbar_expect_tx(smem_u32(full + s), fits ? 4u * kPlane * 4u + kMtBytes : kMtBytes);
        if (fits) {
            // x as (W, H, C, F, B): box (kBox, kBox, 3, 1, 1); masks as (W, H, F, B): box (kBox, kBox, 1, 1)
            tma_load_5d(smem_u32(dst), &map_x, smem_u32(full + s), d.bx0, d.by0, 0, d.f, d.b);
            tma_load_4d(smem_u32(dst + 3 * kPlane), &map_v, smem_u32(full + s), d.bx0, d.by0, d.f, d.b);
        }
        // target mask as (W, H, B): the tile itself
        tma_load_3d(smem_u32(dst + 4 * kPlane), &map_t, smem_u32(full + s), d.tx * kTileW, d.ty * kTileH, d.b);
    };

    if (warp == kConsWarps) {
        // ===================== producer warp =====================
        // The descriptor of the next tile is prepared while its stage is still in use: between
        // "stage released" and "TMA issued" there is only the descriptor store (ncu: consumers
        // polled the full barrier 2.9 times per tile while this chain sat behind the empty wait).
        if (lane == 0) {
            int t = blockIdx.x;
            TileDesc d;
            if (t < a.n_tiles) d = prepare(t);
            for (int i = 0; t < a.n_tiles; ++i) {
                issue(i, d);
                t += gridDim.x;
                if (t < a.n_tiles) d = prepare(t);
            }
        }
        return;
    }

    // ===================== consumers =====================
    const float wm2 = wmax - 1.0f, hm2 = hmax - 1.0f;
    int i = 0;
    for (int t = blockIdx.x; t < a.n_tiles; t += gridDim.x, ++i) {
        const int s = i % kStages;
        const uint32_t ph = (uint32_t)(i / kStages) & 1u;
        mbar_wait(smem_u32(full + s), ph);
        const int4 d0 = reinterpret_cast<const int4 *>(desc + s)[0];      // flags, bx0, by0, b
        const int4 d1 = reinterpret_cast<const int4 *>(desc + s)[1];      // f, n, tx, ty
        const float4 d2 = reinterpret_cast<const float4 *>(desc + s)[2];  // th0..3
        const float4 d3 = reinterpret_cast<const float4 *>(desc + s)[3];  // th4, th5
        const int flags = d0.x, bx0 = d0.y, by0 = d0.z, b = d0.w, f = d1.x, n = d1.y;
        // lane -> pixel: a warp instruction covers 16 columns x 2 adjacent rows (and the thread's second
        // pixel lies 2 rows below).  With the box pitch of 48 words a source row starts 16 banks after
        // the previous one, so the two half-warps read disjoint bank ranges and a tap instruction is
        // one shared-memory wavefront; the 32 x 1 mapping had 2-way conflicts wherever the footprint
        // of the 32 lanes stepped to the next source row (ncu: 44 % of the LDS wavefronts).
        constexpr int kColGroups = kTileW / 16, kRowStep = 2;
        const int tcol = (warp % kColGroups) * 16 + (lane & 15), trow = (warp / kColGroups) * 4 + (lane >> 4);
        const int xg = d1.z * kTileW + tcol, y0 = d1.w * kTileH + trow;
        const bool live = xg < W;
        const int x = min(xg, W - 1);
        const int p0 = y0 * W + x;
        const float *st = stage0 + s * kStageFloats;
        float mtv[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) mtv[k] = st[4 * kPlane + (trow + k * kRowStep) * kTileW + tcol];
        const float bx = s_bx[x];
        const float bxt0 = __fmul_rn(bx, d2.x), bxt3 = __fmul_rn(bx, d2.w);
        float ix[2], iy[2], xw[2], yn[2], wnw[2], wne[2], wsw[2], wse[2];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float by = s_by[min(y0 + k * kRowStep, H - 1)];
            const float gx = __fadd_rn(__fmaf_rn(by, d2.y, bxt0), d2.z);  // fma(by, t1, bx*t0) + t2 (pinned order)
            const float gy = __fadd_rn(__fmaf_rn(by, d3.x, bxt3), d3.y);
            ix[k] = unnorm_t(gx, a.sp.sfx, AC);
            iy[k] = unnorm_t(gy, a.sp.sfy, AC);
            xw[k] = floorf(ix[k]);
            yn[k] = floorf(iy[k]);
            const float w = __fsub_rn(ix[k], xw[k]), e = __fsub_rn(1.0f, w);
            const float nn = __fsub_rn(iy[k], yn[k]), ss = __fsub_rn(1.0f, nn);
            wnw[k] = __fmul_rn(ss, e); wne[k] = __fmul_rn(ss, w);
            wsw[k] = __fmul_rn(nn, e); wse[k] = __fmul_rn(nn, w);
        }
        float xa[3][2], va[2];
        if (flags & 1) {
            // ---------------- taps from the staged box ----------------
            float q[4][2][4];
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const float *p = st + (((int)yn[k] - by0) * kBox + ((int)xw[k] - bx0));
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    q[c][k][0] = p[c * kPlane]; q[c][k][1] = p[c * kPlane + 1];
                    q[c][k][2] = p[c * kPlane + kBox]; q[c][k][3] = p[c * kPlane + kBox + 1];
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(empty + s));
#pragma unroll
            for (int k = 0; k < 2; ++k) {
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    xa[c][k] = __fmaf_rn(q[c][k][3], wse[k], __fmaf_rn(q[c][k][2], wsw[k],
                               __fmaf_rn(q[c][k][1], wne[k], __fmul_rn(q[c][k][0], wnw[k]))));
                float v00 = q[3][k][0], v01 = q[3][k][1], v10 = q[3][k][2], v11 = q[3][k][3];
                if (FM) {
                    v00 = __fsub_rn(1.0f, v00); v01 = __fsub_rn(1.0f, v01);
                    v10 = __fsub_rn(1.0f, v10); v11 = __fsub_rn(1.0f, v11);
                    if (!(flags & 2)) {  // border tile: v is zero-padded, not 1 - 0
                        const float xe = xw[k] + 1.0f, ys = yn[k] + 1.0f;
                        const bool bx0i = (xw[k] >= 0.0f) && (xw[k] <= wmax), bx1i = (xe >= 0.0f) && (xe <= wmax);
                        const bool by0i = (yn[k] >= 0.0f) && (yn[k] <= hmax), by1i = (ys >= 0.0f) && (ys <= hmax);
                        v00 = (by0i && bx0i) ? v00 : 0.0f; v01 = (by0i && bx1i) ? v01 : 0.0f;
                        v10 = (by1i && bx0i) ? v10 : 0.0f; v11 = (by1i && bx1i) ? v11 : 0.0f;
                    }
                }
                const float vs = __fmaf_rn(v11, wse[k], __fmaf_rn(v10, wsw[k],
                                 __fmaf_rn(v01, wne[k], __fmul_rn(v00, wnw[k]))));
                va[k] = vs > 0.5f ? 1.0f : 0.0f;  // strict, model_cpn.py:88
            }
        } else {
            // ---------------- direct gathers (footprint larger than the box) ----------------
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(empty + s));
            const float *xp = a.x + (b * a.x_sb + f * a.x_sf);
            const float *vp = a.vis + (b * a.vis_sb + f * a.vis_sf);
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const Bil bl = bil_params(ix[k], iy[k], a.sp);
#pragma unroll
                for (int c = 0; c < 3; ++c) xa[c][k] = interp(gather(xp + c * a.x_sc, bl, W), bl);
                Corners cv = gather(vp, bl, W);
                if (FM) {
                    cv.nw = (bl.y0 && bl.x0) ? __fsub_rn(1.0f, cv.nw) : 0.0f;
                    cv.ne = (bl.y0 && bl.x1) ? __fsub_rn(1.0f, cv.ne) : 0.0f;
                    cv.sw = (bl.y1 && bl.x0) ? __fsub_rn(1.0f, cv.sw) : 0.0f;
                    cv.se = (bl.y1 && bl.x1) ? __fsub_rn(1.0f, cv.se) : 0.0f;
                }
                va[k] = interp(cv, bl) > 0.5f ? 1.0f : 0.0f;
            }
        }
        (void)wm2; (void)hm2;
        // ---------------- stores (coalesced, streaming) ----------------
        if (live) {
            const int xao = b * a.xa_sb + f * a.xa_sf + p0, np0 = n * a.P + p0;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                if (y0 + k * kRowStep >= H) break;
                const int ro = k * kRowStep * W;
#pragma unroll
                for (int c = 0; c < 3; ++c) st_stream1(a.x_al + (xao + c * a.xa_sc + ro), xa[c][k]);
                st_stream1(a.v_al + (np0 + ro), va[k]);
                st_stream1(a.v_map + (np0 + ro), clamp01(__fsub_rn(va[k], __fsub_rn(1.0f, mtv[k]))));
            }
        }
    }
}

}  // namespace

// 1 = launched, 0 = not applicable (caller uses the direct-gather kernel), < 0 = error.
int warp_staged_launch(const float *x, int64_t x_sb, int64_t x_sc, int64_t x_sf, const float *vis,
                       int64_t vis_sb, int64_t vis_sf, const float *theta, const float *m_target,
                       int64_t mt_sb, float *x_aligned, int64_t xa_sb, int64_t xa_sc, int64_t xa_sf,
                       float *v_aligned, float *v_map, int B, int F, int H, int W, bool ac, bool from_mask,
                       cudaStream_t st) {
    if (!tuning("MT_WARP_STAGED", 1)) return 0;
    if (!(x_aligned && v_aligned && v_map && m_target)) return 0;
    if (W > kMaxTable || H > kMaxTable) return 0;
    // TMA: 16 B aligned base, every stride a multiple of 16 B
    if ((W & 3) || (x_sb & 3) || (x_sc & 3) || (x_sf & 3) || (vis_sb & 3) || (vis_sf & 3)) return 0;
    if (!aligned16(x) || !aligned16(vis) || !aligned16(m_target) || (mt_sb & 3)) return 0;
    // a stride of 0 with an extent > 1 (expanded views such as m_target.expand(B, ...)) cannot be encoded in a
    // tensor map (the encoders below substitute 16 B, which is only harmless for extent 1): direct-gather kernel
    if ((B > 1 && (x_sb == 0 || vis_sb == 0 || mt_sb == 0)) || (F > 1 && (x_sf == 0 || vis_sf == 0)) || x_sc == 0)
        return 0;
    EncodeTiledFn enc = encode_fn();
    if (!enc) return 0;
    const int tiles_x = (W + kTileW - 1) / kTileW, tiles_y = (H + kTileH - 1) / kTileH;
    const int64_t n_tiles = (int64_t)B * F * tiles_x * tiles_y;
    // tiny problems cannot fill a persistent grid of one CTA per SM: keep the strip kernel
    if (n_tiles < 2 * (int64_t)sm_count() || n_tiles > (1ll << 30)) return 0;
    CUtensorMap map_x, map_v, map_t;
    {
        cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
        cuuint64_t strides[2] = {(cuuint64_t)W * 4, mt_sb ? (cuuint64_t)mt_sb * 4 : 16};
        cuuint32_t bx[3] = {(cuuint32_t)kTileW, (cuuint32_t)kTileH, 1};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&map_t, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(m_target), dims, strides,
                         bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return 0;
    }
    {
        cuuint64_t dims[5] = {(cuuint64_t)W, (cuuint64_t)H, 3, (cuuint64_t)F, (cuuint64_t)B};
        cuuint64_t strides[4] = {(cuuint64_t)W * 4, (cuuint64_t)x_sc * 4, (cuuint64_t)x_sf * 4, (cuuint64_t)x_sb * 4};
        // a stride of 0 bytes (B or F of extent 1 sliced out of a view) is not encodable: any multiple of 16 is fine there
        for (int i = 1; i < 4; ++i) if (strides[i] == 0) strides[i] = 16;
        cuuint32_t bx[5] = {(cuuint32_t)kBox, (cuuint32_t)kBox, 3, 1, 1};
        cuuint32_t estr[5] = {1, 1, 1, 1, 1};
        CUresult r = enc(&map_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float *>(x), dims, strides, bx, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return 0;  // e.g. strides beyond the encodable range: direct kernel
    }
    {
        cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)F, (cuuint64_t)B};
        cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)vis_sf * 4, (cuuint64_t)vis_sb * 4};
        for (int i = 1; i < 3; ++i) if (strides[i] == 0) strides[i] = 16;
        cuuint32_t bx[4] = {(cuuint32_t)kBox, (cuuint32_t)kBox, 1, 1};
        cuuint32_t estr[4] = {1, 1, 1, 1};
        CUresult r = enc(&map_v, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float *>(vis), dims, strides, bx,
                         estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return 0;
    }
    WarpStagedArgs a;
    a.x = x; a.vis = vis; a.theta = theta; a.m_target = m_target;
    a.x_al = x_aligned; a.v_al = v_aligned; a.v_map = v_map;
    a.x_sb = (int)x_sb; a.x_sc = (int)x_sc; a.x_sf = (int)x_sf;
    a.vis_sb = (int)vis_sb; a.vis_sf = (int)vis_sf; a.mt_sb = (int)mt_sb;
    a.xa_sb = (int)xa_sb; a.xa_sc = (int)xa_sc; a.xa_sf = (int)xa_sf;
    a.F = F; a.P = H * W; a.tiles_x = tiles_x; a.tiles_per_frame = tiles_x * tiles_y; a.n_tiles = (int)n_tiles;
    a.sp = make_sampler(H, W, ac);
    int ctas = sm_count();
    if (ctas > n_tiles) ctas = (int)n_tiles;
    auto kern = ac ? (from_mask ? warp_staged_kernel<true, true> : warp_staged_kernel<true, false>)
                   : (from_mask ? warp_staged_kernel<false, true> : warp_staged_kernel<false, false>);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kStagedSmem);
    if (e != cudaSuccess) {
        set_error("mt_warp_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        return MT_ERR_CUDA;
    }
    launch(kern, dim3(ctas), dim3(kStagedThreads), (size_t)kStagedSmem, st, map_x, map_v, map_t, a);
    return 1;
}

}  // namespace mt
