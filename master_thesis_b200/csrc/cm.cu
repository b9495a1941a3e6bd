// cm.cu - K3: CPN context matching.
//
// Replaces CM_Module.forward + CM_Module.masked_softmax
//   master_thesis/model_cpn.py:206-254                                   (a8)
//
// The reference's "correlation" here is ONE masked global dot product per
// (sample, reference) - K = C*h*w = 524 288 terms, M = N = 1 - followed by a
// per-pixel softmax over the references and a weighted copy.  It is HBM-bound
// (AI ~ 0.6 flop/B), not a GEMM, so it stays on the SIMT pipes.  Default: two launches
//   pass 0  cm_masks:  v' = bilinear_resize(v, (h,w)) > 0.5 for target + refs, as floats and as
//                      one byte per pixel (bit 0 target, bit r+1 reference r); re-arms the counters of pass 1+2
//   pass 1+2 cm_group: the resident grid is split into groups of CTAs, one sample per group at a time;
//                      a group streams c_feats ONCE from HBM for the R similarities (and copies c_t through),
//                      hands off among its own CTAs only, folds the per-CTA partials into gs (fixed
//                      order, double), evaluates the masked softmax once per MASK PATTERN (2^R entries) and
//                      produces sum_r w_r c_r and c_mask from registers / shared memory / L2 (see the kernel).
// Kept for comparison and for 8 references (the mask byte holds 7): cm_sim | cm_copy2 (MT_CM_TABLE=1: two
// passes over c_feats from HBM, 1.64x the algorithmic traffic) and cm_sim | cm_weights | cm_copy (MT_CM_TABLE=0).
// Reductions are fixed-order (deterministic).  History (profiles/r1_experiments.md, r2_experiments.md):
// a single-CTA-per-sample reduction kernel cost 14 us (latency chain); a per-sample ticket tail in pass 1
// doubled pass 1; per-group launches and a persistent software-pipelined single launch with GLOBAL hand-offs
// ("K3p", round 1, removed) were 1.3-2x slower; the grouped form synchronises per group of CTAs instead.
#include <math.h>

#include "mt_common.cuh"

namespace mt {
namespace {

constexpr int kSimChannels = 4;   // default channels per CTA slab in pass 1 (swept on B200: profiles/)
constexpr int kCopyChannels = 4;  // default channels per CTA slab in pass 2 (template CC)
constexpr int kMaxRefs = 8;
constexpr int kMaxGroupCtas = 512;  // CTAs per group of cm_group_kernel (rows of per-CTA partials per sample)

struct CmArgs {
    const float *c_feats, *v_t, *v_al;
    float *out, *c_mask;
    float *masks;     // workspace: (B, f, P)   index 0 = target
    float *partials;  // workspace: (B, nparts, 2R): [dot_r ..., vsum_r ...]
    float *gs;        // workspace: (B, R)  (exported for tests)
    float *weights;   // workspace: (B, R, P) softmax weights over references
    int B, C, f, h, w, H, W, P, R, nparts, chunks, sim_ch, b_off;
    unsigned char *pmask;        // (B, P) bit 0: vt', bit r + 1: vr' of reference r
    int copy_reverse;
    // grouped single-launch variant (cm_group_kernel)
    unsigned int *counters;      // (B) arrivals per sample, zeroed by cm_masks
    float *gpart;                // (B, S, 2R) per-CTA partials
    int G, S;                    // samples in flight (groups of S CTAs)
};

// F.interpolate(bilinear, align_corners=False) source index (UpSample.h)
__device__ __forceinline__ void src_index(int dst, float scale, int in_size, int &i0, int &i1, float &l0,
                                          float &l1) {
    float s = __fsub_rn(__fmul_rn(scale, __fadd_rn((float)dst, 0.5f)), 0.5f);
    s = s < 0.0f ? 0.0f : s;
    i0 = (int)s;
    i1 = i0 + (i0 < in_size - 1 ? 1 : 0);
    l1 = __fsub_rn(s, (float)i0);
    l0 = __fsub_rn(1.0f, l1);
}

// pass 0: grid (ceil(P / 256), B); thread = one low-resolution pixel, all f masks.
__global__ void __launch_bounds__(256) cm_masks_kernel(const CmArgs a) {
    pdl_sync();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    const int b = blockIdx.y;
    if (p == 0) a.counters[b] = 0u;  // arrival counter of cm_group_kernel (this kernel precedes it in the stream)
    if (p >= a.P) return;
    const int y = p / a.w, x = p - y * a.w;
    int y0, y1, x0, x1;
    float ly0, ly1, lx0, lx1;
    src_index(y, __fdiv_rn((float)a.H, (float)a.h), a.H, y0, y1, ly0, ly1);
    src_index(x, __fdiv_rn((float)a.W, (float)a.w), a.W, x0, x1, lx0, lx1);
    unsigned int bits = 0u;
    // all 4 * f taps are requested before the first use: one DRAM round trip instead of f
    float v00[kMaxRefs + 1], v01[kMaxRefs + 1], v10[kMaxRefs + 1], v11[kMaxRefs + 1];
#pragma unroll
    for (int j = 0; j <= kMaxRefs; ++j) {  // j = 0: target, j >= 1: reference j - 1
        if (j < a.f) {
            const float *src = (j == 0) ? a.v_t + (int64_t)b * a.H * a.W
                                        : a.v_al + ((int64_t)b * a.R + (j - 1)) * a.H * a.W;
            v00[j] = __ldg(src + y0 * a.W + x0); v01[j] = __ldg(src + y0 * a.W + x1);
            v10[j] = __ldg(src + y1 * a.W + x0); v11[j] = __ldg(src + y1 * a.W + x1);
        }
    }
#pragma unroll
    for (int j = 0; j <= kMaxRefs; ++j) {
        if (j < a.f) {
            const float top = __fadd_rn(__fmul_rn(lx0, v00[j]), __fmul_rn(lx1, v01[j]));
            const float bot = __fadd_rn(__fmul_rn(lx0, v10[j]), __fmul_rn(lx1, v11[j]));
            const float val = __fadd_rn(__fmul_rn(ly0, top), __fmul_rn(ly1, bot));
            const bool on = val > 0.5f;                                            // model_cpn.py:208-217
            a.masks[((int64_t)b * a.f + j) * a.P + p] = on ? 1.0f : 0.0f;
            bits |= on ? (1u << j) : 0u;
        }
    }
    a.pmask[(int64_t)b * a.P + p] = (unsigned char)bits;
}

// masked_softmax over the references, once per mask pattern t                         :245-254
// (same operations in the same order as the per-pixel code of cm_weights_kernel)
template <int R>
__device__ __forceinline__ void softmax_table(const float *gs_smem, float *tab) {
    for (int t = threadIdx.x; t < (1 << R); t += blockDim.x) {
        float vr[R], wv[R];
#pragma unroll
        for (int r = 0; r < R; ++r) vr[r] = ((t >> r) & 1) ? 1.0f : 0.0f;
        float mx = -INFINITY;
#pragma unroll
        for (int r = 0; r < R; ++r) mx = fmaxf(mx, __fmul_rn(gs_smem[r], vr[r]));
        float sum = 0.0f;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            wv[r] = __fmul_rn(expf(__fsub_rn(__fmul_rn(gs_smem[r], vr[r]), mx)), vr[r]);
            sum = __fadd_rn(sum, wv[r]);
        }
        if (sum < 1e-4f) sum = __fadd_rn(sum, 1.0f);
        float cm = 0.0f;
#pragma unroll
        for (int r = 0; r < R; ++r) {
            wv[r] = __fdiv_rn(wv[r], sum);
            cm = __fadd_rn(cm, __fmul_rn(wv[r], vr[r]));                          // :240
            tab[t * (R + 1) + r] = wv[r];
        }
        tab[t * (R + 1) + R] = __fsub_rn(1.0f, cm);                               // :241
    }
}

// gs[b, :] from the partials of sample b (fixed order, double).  Result in smem gs[R].
template <int R>
__device__ __forceinline__ void fold_gs(const CmArgs &a, int b, float *gs_smem) {
    __shared__ double dred[2 * R * 8];
    double v[2 * R];
#pragma unroll
    for (int r = 0; r < 2 * R; ++r) v[r] = 0.0;
    for (int i = threadIdx.x; i < a.nparts; i += blockDim.x) {
        const float *o = a.partials + ((int64_t)b * a.nparts + i) * (2 * R);
#pragma unroll
        for (int r = 0; r < 2 * R; ++r) v[r] += (double)__ldcg(o + r);
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int r = 0; r < 2 * R; ++r) {
        v[r] = warp_sum(v[r]);
        if (lane == 0) dred[r * 8 + wid] = v[r];
    }
    __syncthreads();
    if (threadIdx.x < R) {
        const int r = threadIdx.x;
        double d = 0.0, vs = 0.0;
        for (int w = 0; w < nw; ++w) { d += dred[r * 8 + w]; vs += dred[(R + r) * 8 + w]; }
        const bool zero = vs < 1e-4;                                       // :222
        const float v_sum = (float)vs + (zero ? 1.0f : 0.0f);              // :223
        const float g = (float)d / (v_sum * (float)a.C);                   // :225-227
        gs_smem[r] = zero ? 0.0f : g;                                      // :228
    }
    __syncthreads();
}

// pass 1 for one (1024-pixel chunk, SC-channel slab, sample): thread = 4 pixels x SC channels
template <int R, int SC, bool WAIT>
__device__ __forceinline__ void cm_sim_body(const CmArgs &a, int slab, int b, float *red) {
    const int p0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    float acc[2 * R];  // [0, R): dot products, [R, 2R): sum of vt'*vr' (slab 0 only)
#pragma unroll
    for (int r = 0; r < 2 * R; ++r) acc[r] = 0.0f;
    const int c0 = slab * SC;
    float4 ct[SC], cr[SC][R];
    if (p0 < a.P) {
#pragma unroll
        for (int k = 0; k < SC; ++k) {
            const int c = c0 + k;
            if (c < a.C) {
                const float *base = a.c_feats + ((int64_t)b * a.C + c) * a.f * a.P + p0;
                // default L2 policy (NOT evict-first): pass 2 re-reads these from L2
                ct[k] = __ldg(reinterpret_cast<const float4 *>(base));
#pragma unroll
                for (int r = 0; r < R; ++r)
                    cr[k][r] = __ldg(reinterpret_cast<const float4 *>(base + (int64_t)(r + 1) * a.P));
            }
        }
    }
    // WAIT: the features above were requested while the previous kernel of the stream (cm_masks) was
    // still running - they do not depend on it; the masks below do (pdl_wait)
    if (WAIT) pdl_wait();
    if (p0 < a.P) {
        float4 vm[R];
        if (R <= 7) {
            // the masks of 4 pixels as 4 bytes (bit 0 target, bit r + 1 reference r) instead of R + 1 float4
            const uint32_t mw = __ldcg(reinterpret_cast<const uint32_t *>(a.pmask + (int64_t)b * a.P + p0));
#pragma unroll
            for (int r = 0; r < R; ++r) {  // vt' * vr'                  :220
                const uint32_t m = mw & (mw >> (r + 1)) & 0x01010101u;
                vm[r] = make_float4((float)(m & 1u), (float)((m >> 8) & 1u), (float)((m >> 16) & 1u),
                                    (float)((m >> 24) & 1u));
            }
        } else {
            const float *mk = a.masks + (int64_t)b * a.f * a.P + p0;
            const float4 vt = __ldcg(reinterpret_cast<const float4 *>(mk));
#pragma unroll
            for (int r = 0; r < R; ++r) {
                const float4 vr = __ldcg(reinterpret_cast<const float4 *>(mk + (int64_t)(r + 1) * a.P));
                vm[r] = make_float4(vt.x * vr.x, vt.y * vr.y, vt.z * vr.z, vt.w * vr.w);  // :220
            }
        }
#pragma unroll
        for (int r = 0; r < R; ++r)
            if (slab == 0) acc[R + r] = (vm[r].x + vm[r].y) + (vm[r].z + vm[r].w);     // :221
#pragma unroll
        for (int k = 0; k < SC; ++k) {
            if (c0 + k < a.C) {
#pragma unroll
                for (int r = 0; r < R; ++r) {  // vmap * c_t * c_r            :226
                    acc[r] += vm[r].x * ct[k].x * cr[k][r].x;
                    acc[r] += vm[r].y * ct[k].y * cr[k][r].y;
                    acc[r] += vm[r].z * ct[k].z * cr[k][r].z;
                    acc[r] += vm[r].w * ct[k].w * cr[k][r].w;
                }
            }
        }
    }
    block_sum<2 * R>(acc, red);
    if (threadIdx.x == 0) {
        float *o = a.partials + ((int64_t)b * a.nparts + slab * a.chunks + blockIdx.x) * (2 * R);
#pragma unroll
        for (int r = 0; r < 2 * R; ++r) o[r] = acc[r];
    }
}

// pass 1: grid (chunks, C / SC, B)
template <int R, int SC>
__global__ void __launch_bounds__(256) cm_sim_kernel(const CmArgs a) {
    // Scheduled while cm_masks_kernel is still running (that kernel waited for ITS predecessor before it
    // let this one start, so c_feats is complete): the feature loads overlap it, the wait sits in the body.
    pdl_launch();
    __shared__ float red[2 * R * 32];
    cm_sim_body<R, SC, true>(a, (int)blockIdx.y, (int)blockIdx.z + a.b_off, red);
}

// pass 1b: similarities -> per-pixel softmax weights, computed ONCE per pixel.
// grid (ceil(P / 1024), B), 256 threads, one 4-pixel group per thread.
template <int R>
__global__ void __launch_bounds__(256) cm_weights_kernel(const CmArgs a) {
    // launch_dependents BEFORE the wait: the CTAs of cm_copy_kernel are scheduled into the slots that the
    // last wave of pass 1 frees and request their features (old data: c_feats) while pass 1 drains and
    // this kernel runs; they wait for this kernel before they touch the weights.
    pdl_launch();
    pdl_wait();
    __shared__ float gs_smem[R];
    const int b = blockIdx.y + a.b_off;
    fold_gs<R>(a, b, gs_smem);
    if (blockIdx.x == 0 && threadIdx.x < R) a.gs[(int64_t)b * R + threadIdx.x] = gs_smem[threadIdx.x];
    float gsr[R];
#pragma unroll
    for (int r = 0; r < R; ++r) gsr[r] = gs_smem[r];
    const float *mk = a.masks + (int64_t)b * a.f * a.P;
    float *wout = a.weights + (int64_t)b * R * a.P;
    float *ocm = a.out + ((int64_t)b * (2 * a.C + 1) + 2 * a.C) * a.P;
    float *ocm2 = a.c_mask + (int64_t)b * a.P;
    // one 16 B group (4 pixels) per thread
    constexpr int kTail = 1;
    const int ngroups = a.P >> 2;
    for (int g0 = blockIdx.x * blockDim.x + threadIdx.x; g0 < ngroups; g0 += ngroups) {
        float4 vr4[kTail][R];
#pragma unroll
        for (int t = 0; t < kTail; ++t) {
            const int g = g0 + t * blockDim.x;
#pragma unroll
            for (int r = 0; r < R; ++r)
                vr4[t][r] = g < ngroups ? __ldcg(reinterpret_cast<const float4 *>(mk + (int64_t)(r + 1) * a.P) + g)
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int t = 0; t < kTail; ++t) {
            const int g = g0 + t * blockDim.x;
            if (g >= ngroups) break;
            float w4[R][4], cm4[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float vr[R];
#pragma unroll
                for (int r = 0; r < R; ++r)
                    vr[r] = i == 0 ? vr4[t][r].x : (i == 1 ? vr4[t][r].y : (i == 2 ? vr4[t][r].z : vr4[t][r].w));
                float mx = -INFINITY;  // masked_softmax over refs               :245-254
#pragma unroll
                for (int r = 0; r < R; ++r) mx = fmaxf(mx, __fmul_rn(gsr[r], vr[r]));
                float sum = 0.0f;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    w4[r][i] = __fmul_rn(expf(__fsub_rn(__fmul_rn(gsr[r], vr[r]), mx)), vr[r]);
                    sum = __fadd_rn(sum, w4[r][i]);
                }
                if (sum < 1e-4f) sum = __fadd_rn(sum, 1.0f);
                float cm = 0.0f;
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    w4[r][i] = __fdiv_rn(w4[r][i], sum);
                    cm = __fadd_rn(cm, __fmul_rn(w4[r][i], vr[r]));              // :240
                }
                cm4[i] = __fsub_rn(1.0f, cm);                                    // :241
            }
#pragma unroll
            for (int r = 0; r < R; ++r)
                reinterpret_cast<float4 *>(wout + (int64_t)r * a.P)[g] = make_float4(w4[r][0], w4[r][1], w4[r][2], w4[r][3]);
            const float4 c4 = make_float4(cm4[0], cm4[1], cm4[2], cm4[3]);
            reinterpret_cast<float4 *>(ocm)[g] = c4;
            reinterpret_cast<float4 *>(ocm2)[g] = c4;
        }
    }
}

// pass 2 for one (1024-pixel chunk, CC-channel slab, sample): thread = 4 pixels x CC channels
template <int R, int CC, bool WAIT>
__device__ __forceinline__ void cm_copy_body(const CmArgs &a, int slab, int b) {
    const int p0 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (p0 >= a.P) {
        if (WAIT) pdl_wait();
        return;
    }
    const int c0 = slab * CC;
    float4 ct[CC], cr[CC][R];
#pragma unroll
    for (int k = 0; k < CC; ++k) {
        if (c0 + k < a.C) {
            const float *base = a.c_feats + ((int64_t)b * a.C + c0 + k) * a.f * a.P + p0;
            ct[k] = ld_stream4(base);
#pragma unroll
            for (int r = 0; r < R; ++r) cr[k][r] = ld_stream4(base + (int64_t)(r + 1) * a.P);
        }
    }
    // WAIT: the features above were requested while cm_weights_kernel was still running
    if (WAIT) pdl_wait();
    float4 wg[R];
    const float *wp = a.weights + (int64_t)b * R * a.P + p0;
#pragma unroll
    for (int r = 0; r < R; ++r) wg[r] = __ldcg(reinterpret_cast<const float4 *>(wp + (int64_t)r * a.P));
    float *ob = a.out + (int64_t)b * (2 * a.C + 1) * a.P + p0;
#pragma unroll
    for (int k = 0; k < CC; ++k) {
        const int c = c0 + k;
        if (c >= a.C) break;
        float4 o = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
        for (int r = 0; r < R; ++r) {  // sum_r c_r * w_r, sequential over r    :238
            o.x = __fadd_rn(o.x, __fmul_rn(cr[k][r].x, wg[r].x));
            o.y = __fadd_rn(o.y, __fmul_rn(cr[k][r].y, wg[r].y));
            o.z = __fadd_rn(o.z, __fmul_rn(cr[k][r].z, wg[r].z));
            o.w = __fadd_rn(o.w, __fmul_rn(cr[k][r].w, wg[r].w));
        }
        st_stream4(ob + (int64_t)c * a.P, ct[k]);                             // cat[c_t, ...]  :243
        st_stream4(ob + (int64_t)(a.C + c) * a.P, o);
    }
}

// pass 2: grid (chunks, ceil(C / CC), B)
template <int R, int CC>
__global__ void __launch_bounds__(256) cm_copy_kernel(const CmArgs a) {
    pdl_launch();
    // samples in REVERSE order: pass 1 streamed them 0 .. B-1, so the tail of the batch is what is
    // still in L2 (126 MB); walking forwards again evicts it just before it is needed (LRU: ncu
    // 4.6 % hit rate at B=8)
    const int b = (a.copy_reverse ? (int)gridDim.z - 1 - (int)blockIdx.z : (int)blockIdx.z) + a.b_off;
    cm_copy_body<R, CC, true>(a, (int)blockIdx.y, b);
}

// pass 1b + 2 in one launch (the default): every CTA folds the partials of its sample itself (4 KB from
// L2, one double per thread, fixed order) and evaluates the masked softmax once per MASK PATTERN - vr' is
// 0/1, so a sample has only 2^R distinct weight vectors; same operations in the same order as
// cm_weights_kernel, hence the same bits - while its feature loads, issued before the wait, are still in
// flight.  Per pixel the weights are a table lookup by the mask byte.  This removes cm_weights_kernel
// from the chain (7 us as a launch of 32 latency-bound CTAs), the weights array (B,R,P) and its reads.
template <int R, int CC>
__global__ void __launch_bounds__(256, 2) cm_copy2_kernel(const CmArgs a) {
    constexpr int G2 = 2 * R, TABF = (1 << R) * (R + 1);
    __shared__ double dred[256];
    __shared__ float gs_smem[R];
    __shared__ float tab[TABF];
    pdl_launch();
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int p0 = (blockIdx.x * blockDim.x + tid) * 4;
    const bool live = p0 < a.P;
    const int slab = blockIdx.y, b = (a.copy_reverse ? (int)gridDim.z - 1 - (int)blockIdx.z : (int)blockIdx.z) + a.b_off;
    const int c0 = slab * CC;
    float4 ct[CC], cr[CC][R];
    if (live) {
#pragma unroll
        for (int k = 0; k < CC; ++k) {
            if (c0 + k < a.C) {
                const float *base = a.c_feats + ((int64_t)b * a.C + c0 + k) * a.f * a.P + p0;
                ct[k] = ld_stream4(base);
#pragma unroll
                for (int r = 0; r < R; ++r) cr[k][r] = ld_stream4(base + (int64_t)(r + 1) * a.P);
            }
        }
    }
    pdl_wait();  // pass 1 (and cm_masks before it) complete: partials and mask bytes are valid
    const uint32_t mw = live ? __ldcg(reinterpret_cast<const uint32_t *>(a.pmask + (int64_t)b * a.P + p0)) : 0u;
    // ---- gs[b, :]: thread t adds element t % 2R of rows t / 2R, t / 2R + kSlots, ... in increasing order ----
    constexpr int kSlots = 256 / G2;
    double v = 0.0;
    if (tid < kSlots * G2) {
        const int r = tid % G2, i0 = tid / G2;
        const float *o = a.partials + (int64_t)b * a.nparts * G2 + r;
#pragma unroll 4
        for (int i = i0; i < a.nparts; i += kSlots) v += (double)__ldcg(o + (int64_t)i * G2);
    }
    if constexpr ((G2 & (G2 - 1)) == 0 && G2 <= 16) {
        // the lanes l, l + 2R, l + 4R, ... of a warp hold the same element: xor tree, then 8 warps
#pragma unroll
        for (int o = G2; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane < G2) dred[wid * G2 + lane] = v;
        __syncthreads();
        if (tid < R) {
            double d = 0.0, vs = 0.0;
#pragma unroll
            for (int w8 = 0; w8 < 8; ++w8) { d += dred[w8 * G2 + tid]; vs += dred[w8 * G2 + R + tid]; }
            const bool zero = vs < 1e-4;                                       // :222
            const float v_sum = (float)vs + (zero ? 1.0f : 0.0f);              // :223
            const float g = (float)d / (v_sum * (float)a.C);                   // :225-227
            gs_smem[tid] = zero ? 0.0f : g;                                    // :228
        }
    } else {
        dred[tid] = v;
        __syncthreads();
        if (tid < R) {
            double d = 0.0, vs = 0.0;
            for (int sl = 0; sl < kSlots; ++sl) { d += dred[sl * G2 + tid]; vs += dred[sl * G2 + R + tid]; }
            const bool zero = vs < 1e-4;
            const float v_sum = (float)vs + (zero ? 1.0f : 0.0f);
            const float g = (float)d / (v_sum * (float)a.C);
            gs_smem[tid] = zero ? 0.0f : g;
        }
    }
    __syncthreads();
    softmax_table<R>(gs_smem, tab);  // masked_softmax once per mask pattern        :245-254
    __syncthreads();
    if (slab == 0 && blockIdx.x == 0 && tid < R) a.gs[(int64_t)b * R + tid] = gs_smem[tid];
    if (!live) return;
    int pat[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pat[j] = (int)((mw >> (8 * j + 1)) & ((1u << R) - 1u)) * (R + 1);
    float *ob = a.out + (int64_t)b * (2 * a.C + 1) * a.P + p0;
    if (slab == 0) {
        const float4 c4 = make_float4(tab[pat[0] + R], tab[pat[1] + R], tab[pat[2] + R], tab[pat[3] + R]);
        st_stream4(ob + (int64_t)(2 * a.C) * a.P, c4);
        st_stream4(a.c_mask + (int64_t)b * a.P + p0, c4);
    }
    float4 wg[R];
#pragma unroll
    for (int r = 0; r < R; ++r) wg[r] = make_float4(tab[pat[0] + r], tab[pat[1] + r], tab[pat[2] + r], tab[pat[3] + r]);
#pragma unroll
    for (int k = 0; k < CC; ++k) {
        const int c = c0 + k;
        if (c >= a.C) break;
        float4 o = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
        for (int r = 0; r < R; ++r) {  // sum_r c_r * w_r, sequential over r    :238
            o.x = __fadd_rn(o.x, __fmul_rn(cr[k][r].x, wg[r].x));
            o.y = __fadd_rn(o.y, __fmul_rn(cr[k][r].y, wg[r].y));
            o.z = __fadd_rn(o.z, __fmul_rn(cr[k][r].z, wg[r].z));
            o.w = __fadd_rn(o.w, __fmul_rn(cr[k][r].w, wg[r].w));
        }
        st_stream4(ob + (int64_t)c * a.P, ct[k]);                             // cat[c_t, ...]  :243
        st_stream4(ob + (int64_t)(a.C + c) * a.P, o);
    }
}


// ---- single launch for pass 1 + 1b + 2: c_feats crosses HBM ONCE -------------------------------------
// The resident grid (2 CTAs per SM) is split into G groups of S CTAs; group g owns samples g, g + G, ...
// For its sample every CTA of the group
//   1. streams its share of the (channel, 1024-pixel chunk) items from HBM in batches of UN items, accumulates
//      the R masked dot products (pass 1) and already writes the c_t half of cat[c_t, ...] (it does not depend
//      on the similarities); then stores its partials and arrives on the sample's counter;
//   2. waits until the S CTAs of the group have arrived (one thread spins on an acquire load; the other groups
//      are not involved - K3p's post-mortem: the hand-off must be per group of SMs, not global), folds the S
//      partials in fixed order in double and builds the softmax table per mask pattern;
//   3. walks its batches again in REVERSE order for sum_r w_r c_r and c_mask: the last batch is still in
//      registers, the `keep` batches before it were parked in shared memory, the rest is what this CTA left
//      in L2 microseconds ago (G samples in flight are G * C * f * P * 4 B = 84 MB at B = 8, 128 x 5 x 64 x 64,
//      of the 126 MB; read with evict-first loads).  ncu at cfg2: 87 MB read from DRAM (the 3-launch form: 179 MB).
// Every CTA of the grid is resident (grid <= SMs x occupancy), so the spin cannot deadlock.
template <int R>
struct CmGroupCfg {
    static constexpr int UN = R <= 3 ? 4 : (R == 4 ? 3 : 2);  // items per batch: UN * (R + 1) 16 B loads in flight per thread
    static constexpr int kBatchBytes = UN * R * 256 * 16;     // reference features of one batch parked in shared memory
};

#ifdef MT_DEV_PROBES
// developer timeline probe (probe builds only, tools/dbg_cm_timeline.py): per CTA globaltimer stamps of the first sample
// [0] entry, [1] pass 1 done (arrived), [2] hand-off passed (all CTAs of the group arrived), [3] table built, [4] pass 2 done
__device__ unsigned long long g_cm_timeline[1024 * 8];
__device__ __forceinline__ void cm_stamp(int slot) {
    if (threadIdx.x == 0 && blockIdx.x < 1024) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
        g_cm_timeline[blockIdx.x * 8 + slot] = t;
    }
}
#define MT_CM_STAMP(slot) cm_stamp(slot)
#else
#define MT_CM_STAMP(slot)
#endif

template <int R>
__global__ void __launch_bounds__(256, 2) cm_group_kernel(const CmArgs a, const int keep) {
    constexpr int G2 = 2 * R, TABF = (1 << R) * (R + 1), UN = CmGroupCfg<R>::UN;
    constexpr int kMw = 4;  // mask words cached per thread (one per 1024-pixel chunk) when the sample has <= kMw chunks
    __shared__ float red[G2 * 32];
    __shared__ double dred[256];
    __shared__ float gs_smem[R];
    __shared__ float tab[TABF];
    extern __shared__ __align__(16) uint8_t cm_dyn[];
    float4 *park = reinterpret_cast<float4 *>(cm_dyn);  // [keep][UN][R][256]
    pdl_launch();
    MT_CM_STAMP(0);
    const int tid = threadIdx.x;
    const int g = (int)blockIdx.x % a.G, s = (int)blockIdx.x / a.G;
    if (s >= a.S) return;
    const int NI = a.C * a.chunks;
    const int lo = (int)((int64_t)s * NI / a.S), hi = (int)((int64_t)(s + 1) * NI / a.S);
    const int nb = (hi - lo + UN - 1) / UN;  // batches of this CTA
    const int fP = a.f * a.P;  // 32-bit offsets within a sample (the launcher checks (2C + 1) * f * P < 2^31)
    const bool mw_cached = a.chunks <= kMw;
    bool waited = false;  // griddepcontrol.wait (cm_masks complete) once, after the first feature loads are in flight
    float4 cr[UN][R];     // reference features of the batch in flight; the last batch of pass 1 stays here for pass 2

    auto mask_word = [&](const uint32_t (&mwq)[kMw], const unsigned char *pm, int q, int p) -> uint32_t {
        if (mw_cached) {
            uint32_t w = mwq[0];
#pragma unroll
            for (int j = 1; j < kMw; ++j) w = q == j ? mwq[j] : w;
            return w;
        }
        return __ldcg(reinterpret_cast<const uint32_t *>(pm + p));
    };
    auto load_cr = [&](const float *fb, int bi, bool stream) {
        const int it = lo + bi * UN;
#pragma unroll
        for (int k = 0; k < UN; ++k) {
            // slots past the CTA's range / the chunk's end load a valid (clamped) address and are skipped by the
            // consumers: unconditional loads keep the register live ranges apart (ptxas spilled otherwise)
            const int i = min(it + k, hi - 1), c = i / a.chunks, p = (i - c * a.chunks) * 1024 + tid * 4;
            const float *base = fb + (c * fP + min(p, a.P - 4));
#pragma unroll
            for (int r = 0; r < R; ++r)
                cr[k][r] = stream ? ld_stream4(base + (r + 1) * a.P)
                                  : __ldg(reinterpret_cast<const float4 *>(base + (r + 1) * a.P));
        }
    };
    // ---------------- pass 1: partial dot products of this CTA's items, c_t copied through; arrives, does not wait ----------------
    auto pass1 = [&](int b, uint32_t (&mwq)[kMw], int np) {
        const float *fb = a.c_feats + (int64_t)b * a.C * fP;
        const unsigned char *pm = a.pmask + (int64_t)b * a.P;
        float *ob = a.out + (int64_t)b * (2 * a.C + 1) * a.P;
        float acc[G2];
#pragma unroll
        for (int r = 0; r < G2; ++r) acc[r] = 0.0f;
#pragma unroll 1
        for (int bi = 0; bi < nb; ++bi) {
            const int it = lo + bi * UN;
            float4 ct[UN];
#pragma unroll
            for (int k = 0; k < UN; ++k) {
                const int i = min(it + k, hi - 1), c = i / a.chunks, p = (i - c * a.chunks) * 1024 + tid * 4;
                ct[k] = __ldg(reinterpret_cast<const float4 *>(fb + (c * fP + min(p, a.P - 4))));
            }
            load_cr(fb, bi, false);  // default L2 policy: part of it is read again in pass 2
            if (!waited) { pdl_wait(); waited = true; }
            if (bi == 0 && mw_cached) {
#pragma unroll
                for (int j = 0; j < kMw; ++j)
                    mwq[j] = (j < a.chunks && j * 1024 + tid * 4 < a.P) ? __ldcg(reinterpret_cast<const uint32_t *>(pm + j * 1024 + tid * 4)) : 0u;
            }
#pragma unroll
            for (int k = 0; k < UN; ++k) {
                const int i = it + k, c = i / a.chunks, q = i - c * a.chunks, p = q * 1024 + tid * 4;
                if (i >= hi || p >= a.P) continue;
                const uint32_t mw = mask_word(mwq, pm, q, p);
                st_stream4(ob + (c * a.P + p), ct[k]);                             // cat[c_t, ...]  :243
#pragma unroll
                for (int r = 0; r < R; ++r) {  // vt' * vr'                  :220
                    const uint32_t m = mw & (mw >> (r + 1)) & 0x01010101u;
                    const float4 vm = make_float4((float)(m & 1u), (float)((m >> 8) & 1u), (float)((m >> 16) & 1u),
                                                  (float)((m >> 24) & 1u));
                    if (c == 0) acc[R + r] += (vm.x + vm.y) + (vm.z + vm.w);       // :221 (once per pixel)
                    acc[r] += vm.x * ct[k].x * cr[k][r].x;                         // :226
                    acc[r] += vm.y * ct[k].y * cr[k][r].y;
                    acc[r] += vm.z * ct[k].z * cr[k][r].z;
                    acc[r] += vm.w * ct[k].w * cr[k][r].w;
                    if (bi < np) park[((bi * UN + k) * R + r) * 256 + tid] = cr[k][r];
                }
            }
        }
        if (!waited) { pdl_wait(); waited = true; }
        block_sum<G2>(acc, red);
        if (tid == 0) {
            float *o = a.gpart + ((int64_t)b * a.S + s) * G2;
#pragma unroll
            for (int r = 0; r < G2; ++r) o[r] = acc[r];
            __threadfence();
            atomicAdd(a.counters + b, 1u);
        }
    };
    // ---------------- hand-off inside the group, gs[b, :] (fixed order, double), softmax table ----------------
    auto handoff = [&](int b) {
        if (tid == 0) {
            unsigned int seen;
            do {  // the S CTAs of this group only
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(seen) : "l"(a.counters + b) : "memory");
                if (seen < (unsigned int)a.S) __nanosleep(40);
            } while (seen < (unsigned int)a.S);
        }
        __syncthreads();
        if (b == g) MT_CM_STAMP(2);
        constexpr int kSlots = 256 / G2;
        double v = 0.0;
        if (tid < kSlots * G2) {
            const int r = tid % G2, i0 = tid / G2;
            const float *o = a.gpart + (int64_t)b * a.S * G2 + r;
#pragma unroll 4
            for (int i = i0; i < a.S; i += kSlots) v += (double)__ldcg(o + (int64_t)i * G2);
        }
        dred[tid] = v;
        __syncthreads();
        if (tid < R) {
            double d = 0.0, vs = 0.0;
            for (int sl = 0; sl < kSlots; ++sl) { d += dred[sl * G2 + tid]; vs += dred[sl * G2 + R + tid]; }
            const bool zero = vs < 1e-4;                                       // :222
            const float v_sum = (float)vs + (zero ? 1.0f : 0.0f);              // :223
            const float gg = (float)d / (v_sum * (float)a.C);                  // :225-227
            gs_smem[tid] = zero ? 0.0f : gg;                                   // :228
            if (s == 0) a.gs[(int64_t)b * R + tid] = gs_smem[tid];
        }
        __syncthreads();
        softmax_table<R>(gs_smem, tab);
        __syncthreads();
    };
    // ---------------- pass 2: sum_r w_r c_r and c_mask ----------------
    // operands: batch nb - 1 from registers if `last_in_regs`, batches 0 .. np - 1 (the oldest in L2) from shared memory,
    // the rest from L2, most recently read first, each requested one step ahead while a parked batch is processed
    auto pass2 = [&](int b, const uint32_t (&mwq)[kMw], int np, bool last_in_regs) {
        const float *fb = a.c_feats + (int64_t)b * a.C * fP;
        const unsigned char *pm = a.pmask + (int64_t)b * a.P;
        float *ob = a.out + (int64_t)b * (2 * a.C + 1) * a.P;
        // one item: the weights of its 4 pixels are table rows selected by the mask bytes
        auto emit = [&](int i, auto &&ref) {
            const int c = i / a.chunks, q = i - c * a.chunks, p = q * 1024 + tid * 4;
            if (i >= hi || p >= a.P) return;
            const uint32_t mw = mask_word(mwq, pm, q, p);
            int pat[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) pat[j] = (int)((mw >> (8 * j + 1)) & ((1u << R) - 1u)) * (R + 1);
            if (c == 0) {
                const float4 c4 = make_float4(tab[pat[0] + R], tab[pat[1] + R], tab[pat[2] + R], tab[pat[3] + R]);
                st_stream4(ob + (2 * a.C * a.P + p), c4);
                st_stream4(a.c_mask + ((int64_t)b * a.P + p), c4);
            }
            float4 o = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
            for (int r = 0; r < R; ++r) {  // sum_r c_r * w_r, sequential over r    :238
                const float4 v = ref(r);
                o.x = __fadd_rn(o.x, __fmul_rn(v.x, tab[pat[0] + r]));
                o.y = __fadd_rn(o.y, __fmul_rn(v.y, tab[pat[1] + r]));
                o.z = __fadd_rn(o.z, __fmul_rn(v.z, tab[pat[2] + r]));
                o.w = __fadd_rn(o.w, __fmul_rn(v.w, tab[pat[3] + r]));
            }
            st_stream4(ob + ((a.C + c) * a.P + p), o);
        };
        auto emit_regs = [&](int bi) {
#pragma unroll
            for (int k = 0; k < UN; ++k) emit(lo + bi * UN + k, [&](int r) { return cr[k][r]; });
        };
        auto emit_parked = [&](int bi) {  // straight from shared memory, 4 registers at a time
#pragma unroll
            for (int k = 0; k < UN; ++k) emit(lo + bi * UN + k, [&](int r) { return park[((bi * UN + k) * R + r) * 256 + tid]; });
        };
        if (nb > 0) {
            int j = nb - 1;        // next register / L2 batch
            int q = 0;             // next parked batch
            if (last_in_regs) { emit_regs(j); --j; }
            if (j >= np) load_cr(fb, j, true);
#pragma unroll 1
            while (j >= np || q < np) {
                if (q < np) { emit_parked(q); ++q; }
                if (j >= np) {
                    emit_regs(j);
                    --j;
                    if (j >= np) load_cr(fb, j, true);
                }
            }
        }
    };

    // Handing the batches out dynamically inside the group (tickets, per-batch partial rows) narrowed the spread of the
    // pass-1 finish times from 6.4 to 4 us (one batch is ~4 us) but cost as much per batch: step 61.9 vs 61.5 us.  Not kept.
    // A software-pipelined form (pass 1 of the group's next sample before pass 2 of the current one, two samples per
    // group in flight, G = 4) hid the hand-off but was 5 - 10 % slower in the step (profiles/r2_experiments.md): with
    // half as many items per CTA and sample the batches are short (3 + 3 + 1 items) and every other sample has no parked
    // batches.  Not kept.
    uint32_t mwq[kMw] = {0u, 0u, 0u, 0u};
    const int np = min(keep, nb - 1);
#pragma unroll 1
    for (int b = g; b < a.B; b += a.G) {
        pass1(b, mwq, np);
        if (b == g) MT_CM_STAMP(1);
        handoff(b);
        if (b == g) MT_CM_STAMP(3);
        pass2(b, mwq, np, true);
        if (b == g) MT_CM_STAMP(4);
        __syncthreads();  // red / tab / park are reused by the next sample of this group
    }
}

// resident CTAs of cm_group_kernel<R> on this device (<= 2 per SM) and the batches each may park in shared memory
template <int R>
int cm_group_ctas(int *keep_out) {
    static int n = 0, keep = 0;
    if (n == 0) {
        cudaFuncAttributes fa;
        int dev = 0, smem_sm = 0, occ = 0;
        if (cudaFuncGetAttributes(&fa, cm_group_kernel<R>) != cudaSuccess || cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev) != cudaSuccess)
            return 0;
        // two CTAs per SM: each gets half of the SM's shared memory minus its static part and the 1 KB the system reserves
        int dyn = smem_sm / 2 - (int)fa.sharedSizeBytes - 1024;
        int kp = dyn / CmGroupCfg<R>::kBatchBytes;
        if (kp > 8) kp = 8;
        if (kp < 0) kp = 0;
        const int bytes = kp * CmGroupCfg<R>::kBatchBytes;
        if (cudaFuncSetAttribute(cm_group_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) != cudaSuccess) return 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, cm_group_kernel<R>, 256, bytes) != cudaSuccess || occ < 1) return 0;
        keep = kp;
        n = sm_count() * (occ > 2 ? 2 : occ);
    }
    *keep_out = keep;
    return n;
}

template <int R>
int launch_cm(CmArgs a, cudaStream_t st) {
    a.b_off = 0;
    const int mode = tuning("MT_CM_TABLE", 2);  // 2: grouped single launch, 1: sim | copy2 (table), 0: sim | weights | copy
    if constexpr (R <= 7) {
        int keep = 0;
        const int ctas = (mode == 2 && (int64_t)(2 * a.C + 1) * a.f * a.P < (1ll << 31)) ? cm_group_ctas<R>(&keep) : 0;
        // batches parked in shared memory between the passes.  Default 0 since the kernels ahead of this one stopped
        // pinning the SMs' shared-memory split (pdl_sync in mt_common.cuh): without dynamic shared memory the kernel
        // runs with the full L1, which holds a CTA's most recent pass-1 lines for pass 2 - 44.0 -> 38.2 us per call at
        // B = 8 (cfg2 step 61.9 -> 56.4 us); parking 2 batches in shared memory gave the same time as parking none
        // while the split was pinned
        keep = max(0, min(keep, tuning("MT_CM_KEEP", 0)));
        if (ctas > 0) {
            // samples in flight: as many as keep their features (C * f * P * 4 B each) within ~90 MB of L2
            const int64_t sample_bytes = (int64_t)a.C * a.f * a.P * 4;
            int64_t g = tuning("MT_CM_GROUPS", 0);
            if (g <= 0) g = (int64_t)tuning("MT_CM_L2_MB", 90) * 1000000 / sample_bytes;
            if (g > a.B) g = a.B;
            if (g > ctas) g = ctas;
            if (g < 1) g = 1;
            a.G = (int)g;
            a.S = ctas / a.G;
            if (a.S > kMaxGroupCtas) a.S = kMaxGroupCtas;
            launch(cm_masks_kernel, dim3((a.P + 255) / 256, a.B), 256, 0, st, a);
            launch(cm_group_kernel<R>, dim3(a.G * a.S), 256, (size_t)keep * CmGroupCfg<R>::kBatchBytes, st, a, keep);
            return launch_status("mt_cm_match_fwd");
        }
    }
    launch(cm_masks_kernel, dim3((a.P + 255) / 256, a.B), 256, 0, st, a);
    const int cc = tuning("MT_CM_COPY_CH", kCopyChannels);
    a.nparts = a.chunks * ((a.C + a.sim_ch - 1) / a.sim_ch);
    const int slabs = (a.C + a.sim_ch - 1) / a.sim_ch;
    dim3 g1(a.chunks, slabs, a.B);
    if (a.sim_ch == 2) launch(cm_sim_kernel<R, 2>, g1, 256, 0, st, a);
    else launch(cm_sim_kernel<R, 4>, g1, 256, 0, st, a);
    if (R <= 7 && mode) {  // pass 1b folded into pass 2 (the mask byte holds <= 7 references)
        if (cc == 2) launch(cm_copy2_kernel<R, 2>, dim3(a.chunks, (a.C + 1) / 2, a.B), 256, 0, st, a);
        else launch(cm_copy2_kernel<R, 4>, dim3(a.chunks, (a.C + 3) / 4, a.B), 256, 0, st, a);
        return launch_status("mt_cm_match_fwd");
    }
    launch(cm_weights_kernel<R>, dim3(a.chunks, a.B), 256, 0, st, a);
    if (cc == 2) launch(cm_copy_kernel<R, 2>, dim3(a.chunks, (a.C + 1) / 2, a.B), 256, 0, st, a);
    else launch(cm_copy_kernel<R, 4>, dim3(a.chunks, (a.C + 3) / 4, a.B), 256, 0, st, a);
    return launch_status("mt_cm_match_fwd");
}

int sim_channels() { return tuning("MT_CM_SIM_CH", kSimChannels) == 2 ? 2 : 4; }

int64_t align256(int64_t v) { return (v + 255) & ~int64_t(255); }

}  // namespace
}  // namespace mt

using namespace mt;

extern "C" int64_t mt_cm_workspace_bytes(int B, int C, int f, int h, int w) {
    if (B <= 0 || C <= 0 || f < 2 || h <= 0 || w <= 0) return 0;
    const int64_t P = (int64_t)h * w, R = f - 1;
    const int64_t chunks = (P + 1023) / 1024, nparts = chunks * ((C + 1) / 2);  // finest pass-1 split
    return align256(B * f * P * 4) + align256(B * nparts * 2 * R * 4) + align256(B * R * 4) +
           align256(B * R * P * 4) + align256(B * P) + align256((int64_t)B * 4) +
           align256((int64_t)B * kMaxGroupCtas * 2 * R * 4);
}

extern "C" int mt_cm_match_fwd(const float *c_feats, const float *v_t, const float *v_aligned,
                               float *out, float *c_mask, void *workspace, int B, int C, int f,
                               int h, int w, int H, int W, mt_stream_t stream) {
    MT_REQUIRE(c_feats && v_t && v_aligned && out && c_mask && workspace, "mt_cm_match_fwd: NULL argument");
    MT_REQUIRE(B > 0 && C > 0 && h > 0 && w > 0 && H > 0 && W > 0, "mt_cm_match_fwd: empty shape");
    MT_REQUIRE(f >= 2 && f - 1 <= kMaxRefs, "mt_cm_match_fwd: needs 1..%d reference frames, got %d", kMaxRefs, f - 1);
    MT_REQUIRE(B <= 65535, "mt_cm_match_fwd: B > 65535");
    MT_REQUIRE(((int64_t)h * w) % 4 == 0, "mt_cm_match_fwd: h*w must be a multiple of 4 (got %dx%d)", h, w);
    MT_REQUIRE(aligned16(c_feats) && aligned16(out) && aligned16(c_mask) && aligned16(workspace),
               "mt_cm_match_fwd: pointers must be 16 B aligned");
    CmArgs a;
    a.c_feats = c_feats; a.v_t = v_t; a.v_al = v_aligned; a.out = out; a.c_mask = c_mask;
    a.B = B; a.C = C; a.f = f; a.h = h; a.w = w; a.H = H; a.W = W; a.P = h * w; a.R = f - 1;
    a.chunks = (a.P + 1023) / 1024;
    a.sim_ch = sim_channels();
    a.nparts = a.chunks * ((C + a.sim_ch - 1) / a.sim_ch);
    char *ws = reinterpret_cast<char *>(workspace);
    a.masks = reinterpret_cast<float *>(ws);
    ws += align256((int64_t)B * f * a.P * 4);
    a.partials = reinterpret_cast<float *>(ws);
    ws += align256((int64_t)B * a.chunks * ((C + 1) / 2) * 2 * a.R * 4);
    a.gs = reinterpret_cast<float *>(ws);
    ws += align256((int64_t)B * a.R * 4);
    a.weights = reinterpret_cast<float *>(ws);
    ws += align256((int64_t)B * a.R * a.P * 4);
    a.pmask = reinterpret_cast<unsigned char *>(ws);
    ws += align256((int64_t)B * a.P);
    a.counters = reinterpret_cast<unsigned int *>(ws);
    ws += align256((int64_t)B * 4);
    a.gpart = reinterpret_cast<float *>(ws);
    a.G = a.S = 0;
    a.copy_reverse = tuning("MT_CM_COPY_REVERSE", 1);
    cudaStream_t st = (cudaStream_t)stream;
    switch (a.R) {
        case 1: return launch_cm<1>(a, st);
        case 2: return launch_cm<2>(a, st);
        case 3: return launch_cm<3>(a, st);
        case 4: return launch_cm<4>(a, st);
        case 5: return launch_cm<5>(a, st);
        case 6: return launch_cm<6>(a, st);
        case 7: return launch_cm<7>(a, st);
        default: return launch_cm<8>(a, st);
    }
}

// gs (B, f-1) as left in the workspace by the last mt_cm_match_fwd (for tests)
extern "C" const float *mt_cm_workspace_gs(const void *workspace, int B, int C, int f, int h, int w) {
    const int64_t P = (int64_t)h * w, R = f - 1;
    const int64_t chunks = (P + 1023) / 1024, nparts = chunks * ((C + 1) / 2);
    return reinterpret_cast<const float *>(reinterpret_cast<const char *>(workspace) +
                                           align256(B * f * P * 4) + align256(B * nparts * 2 * R * 4));
}

#ifdef MT_DEV_PROBES
extern "C" __attribute__((visibility("default"))) int mt_debug_cm_timeline(unsigned long long *dst, int n) {
    cudaDeviceSynchronize();
    return cudaMemcpyFromSymbol(dst, mt::g_cm_timeline, sizeof(unsigned long long) * (n < 8192 ? n : 8192)) == cudaSuccess ? 0 : -2;
}
#endif
