// mt_common.cuh - shared host/device helpers for libmt_b200.so (sm_100a only).
//
// Arithmetic contract (see DESIGN.md "bit-exactness"): every expression whose
// rounding decides an index, a mask bit or a threshold is written with explicit
// round-to-nearest intrinsics (__fadd_rn / __fmul_rn / __fmaf_rn) in exactly the
// order the reference's CPU path (ATen, torch 2.11) evaluates it, and the
// library is compiled with -fmad=false so nvcc cannot contract anything else.
#pragma once

#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "mt_b200.h"

namespace mt {

// ---- host side ------------------------------------------------------------
void set_error(const char *fmt, ...);
int launch_status(const char *what);  // cudaGetLastError -> MT_OK / MT_ERR_CUDA
int sm_count();
// integer tuning knob from the environment (read once per name), else `dflt`
int tuning(const char *name, int dflt);

#define MT_REQUIRE(cond, ...)            \
    do {                                 \
        if (!(cond)) {                   \
            ::mt::set_error(__VA_ARGS__); \
            return MT_ERR_INVALID;       \
        }                                \
    } while (0)

// Every kernel of the library is launched through launch(): with programmatic dependent
// launch (PDL) the CTAs of kernel N+1 are scheduled into SM slots as the last wave of
// kernel N drains; they block in pdl_sync() until N has completed and flushed.  At the
// batch sizes of this path kernels last 10-50 us, so the 2-4 us launch gaps matter.
bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline void launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                   Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    (void)cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);  // status: launch_status()
}

static inline bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
// the vector path of a kernel reads 4 consecutive elements of type T in one access (16 B of float, 8 B of half)
template <typename T>
static inline bool aligned_vec4(const void *p) {
    return (reinterpret_cast<uintptr_t>(p) & (4 * sizeof(T) - 1)) == 0;
}

// Network operands (the CNN output, the inputs of the losses) may arrive in fp16 / bf16 under autocast: the element
// type of such an operand is a dtype code MT_DT_*.  Calls f(T{}) with T = float, __half or __nv_bfloat16.
template <typename Fn>
inline int with_dtype(int dt, const char *who, Fn &&f) {
    switch (dt) {
        case MT_DT_F32: return f(float{});
        case MT_DT_F16: return f(__half{});
        case MT_DT_BF16: return f(__nv_bfloat16{});
        default: break;
    }
    set_error("%s: unknown dtype code %d", who, dt);
    return MT_ERR_INVALID;
}

// The memory layout of a network operand (the CNN input the packs write, the CNN output the composite / fill kernels
// read) is a layout code MT_LAYOUT_*.  Calls f(std::bool_constant<NHWC>{}); any other code is an error.
template <typename Fn>
inline int with_layout(int layout, const char *who, Fn &&f) {
    if (layout == MT_LAYOUT_NCHW) return f(std::false_type{});
    if (layout == MT_LAYOUT_NHWC) return f(std::true_type{});
    set_error("%s: unknown layout code %d", who, layout);
    return MT_ERR_INVALID;
}

// workspace layout used by the reducing kernels
constexpr int kMaxReduceBlocks = 16384;
constexpr int kPartialsPerBlock = 8;  // up to two float4 rows per CTA
constexpr int64_t kWsTicketBytes = 256;
constexpr int64_t kWorkspaceBytes = kWsTicketBytes + int64_t(kMaxReduceBlocks) * kPartialsPerBlock * 4;

// ---- device side ----------------------------------------------------------
#ifdef __CUDACC__

// First statement of every kernel.  wait: the previous kernel in the stream has completed
// and its writes are visible.  launch_dependents AFTER the wait: the next kernel may only
// be scheduled once every CTA of this one has started, so waiting CTAs can never occupy
// the slots this kernel still needs.  Exception: the persistent kernels that hold ~200 KB of
// shared memory per SM (corr_tc.cu, warp_tma.cu) only wait and leave the trigger to their
// exit - dependents pre-launched beside them would pin the SM's shared-memory / L1 split at its
// maximum-shared-memory setting for the whole PDL chain behind them (measured in corr_tc.cu).
__device__ __forceinline__ void pdl_sync() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// The two halves separately, for kernels whose first loads do not depend on the previous kernel of the
// stream (see cm.cu): launch_dependents first, the wait where the dependent loads begin.  Safe only
// when the previous kernel itself waited before it called launch_dependents (every kernel of this
// library does): then everything older than it has completed.
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

constexpr float kMean0 = 0.485f, kMean1 = 0.456f, kMean2 = 0.406f;  // model_chn.py:32-37
constexpr float kStd0 = 0.229f, kStd1 = 0.224f, kStd2 = 0.225f;

__device__ __forceinline__ float chan_mean(int c) { return c == 0 ? kMean0 : (c == 1 ? kMean1 : kMean2); }
__device__ __forceinline__ float chan_std(int c) { return c == 0 ? kStd0 : (c == 1 ? kStd1 : kStd2); }

// streaming (touch-once) global accesses: keep them out of L1, evict-first in L2
__device__ __forceinline__ float4 ld_stream4(const float *p) {
    return __ldcs(reinterpret_cast<const float4 *>(p));
}
__device__ __forceinline__ float ld_stream1(const float *p) { return __ldcs(p); }
__device__ __forceinline__ void st_stream4(float *p, float4 v) {
    __stcs(reinterpret_cast<float4 *>(p), v);
}
__device__ __forceinline__ void st_stream1(float *p, float v) { __stcs(p, v); }

// fp16 / bf16 operands: widened to float on load (exact), gradients narrowed on store (round to nearest even)
__device__ __forceinline__ float widen(__half v) { return __half2float(v); }
__device__ __forceinline__ float widen(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T>
__device__ __forceinline__ T narrow(float v);
template <>
__device__ __forceinline__ __half narrow<__half>(float v) { return __float2half_rn(v); }
template <>
__device__ __forceinline__ __nv_bfloat16 narrow<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// Vec<VEC>: VEC consecutive elements in float registers.  The float overloads are the fp32 path; the templates read
// and write 2-byte element types (one 8-byte access for VEC = 4).
template <int VEC>
struct Vec;
template <>
struct Vec<1> {
    float v[1];
    __device__ __forceinline__ void load_stream(const float *p) { v[0] = ld_stream1(p); }
    __device__ __forceinline__ void load_cached(const float *p) { v[0] = __ldg(p); }
    __device__ __forceinline__ void store_stream(float *p) const { st_stream1(p, v[0]); }
    template <typename T>
    __device__ __forceinline__ void load_stream(const T *p) { v[0] = widen(__ldcs(p)); }
    template <typename T>
    __device__ __forceinline__ void store_stream(T *p) const { __stcs(p, narrow<T>(v[0])); }
    // plain store (any state space: the shared-memory stage of an NHWC tile)
    template <typename T>
    __device__ __forceinline__ void store_plain(T *p) const {
        if constexpr (sizeof(T) == 4) *p = v[0];
        else *p = narrow<T>(v[0]);
    }
};
template <>
struct Vec<4> {
    float v[4];
    __device__ __forceinline__ void load_stream(const float *p) {
        float4 t = ld_stream4(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void load_cached(const float *p) {
        float4 t = __ldg(reinterpret_cast<const float4 *>(p));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void store_stream(float *p) const {
        st_stream4(p, make_float4(v[0], v[1], v[2], v[3]));
    }
    template <typename T>
    __device__ __forceinline__ void load_stream(const T *p) {
        static_assert(sizeof(T) == 2, "2-byte element types only");
        const uint2 u = __ldcs(reinterpret_cast<const uint2 *>(p));
        const T *e = reinterpret_cast<const T *>(&u);
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = widen(e[i]);
    }
    template <typename T>
    __device__ __forceinline__ void store_stream(T *p) const {
        static_assert(sizeof(T) == 2, "2-byte element types only");
        uint2 u;
        T *e = reinterpret_cast<T *>(&u);
#pragma unroll
        for (int i = 0; i < 4; ++i) e[i] = narrow<T>(v[i]);
        __stcs(reinterpret_cast<uint2 *>(p), u);
    }
    template <typename T>
    __device__ __forceinline__ void store_plain(T *p) const {
        if constexpr (sizeof(T) == 4) {
            *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
            uint2 u;
            T *e = reinterpret_cast<T *>(&u);
#pragma unroll
            for (int i = 0; i < 4; ++i) e[i] = narrow<T>(v[i]);
            *reinterpret_cast<uint2 *>(p) = u;
        }
    }
};

// ---- channels-last (NHWC) network operands ----------------------------------------------------------------------
// In NHWC the C channels of a pixel are adjacent, so the VEC consecutive pixels of a thread are VEC * C consecutive
// elements.  Reads take them as C vectors and de-interleave in registers.  Writes go through a shared-memory stage
// in output order (each thread's run at threadIdx.x * VEC * C), which the CTA then writes out as one contiguous,
// coalesced run: VEC * C * 4 B per thread (36, 40, 12 B per pixel) does not map onto 16-byte vector stores.
template <int VEC, int C, typename T>
__device__ __forceinline__ void load_nhwc(Vec<VEC> (&o)[C], const T *p) {
    Vec<VEC> r[C];
#pragma unroll
    for (int j = 0; j < C; ++j) r[j].load_stream(p + j * VEC);
#pragma unroll
    for (int i = 0; i < VEC; ++i)
#pragma unroll
        for (int c = 0; c < C; ++c) o[c].v[i] = r[(i * C + c) / VEC].v[(i * C + c) % VEC];
}

template <int VEC, int C, typename T>
__device__ __forceinline__ void stage_nhwc(T *stage, const Vec<VEC> (&o)[C]) {
    Vec<VEC> r[C];
#pragma unroll
    for (int i = 0; i < VEC; ++i)
#pragma unroll
        for (int c = 0; c < C; ++c) r[(i * C + c) / VEC].v[(i * C + c) % VEC] = o[c].v[i];
    T *s = stage + threadIdx.x * (VEC * C);
#pragma unroll
    for (int j = 0; j < C; ++j) r[j].store_plain(s + j * VEC);
}

// n staged elements to dst (after a __syncthreads): 16-byte streaming stores when dst is 16-byte aligned and n fills
// them, else one element per thread and instruction (still one contiguous run per warp)
template <typename T>
__device__ __forceinline__ void stage_out(T *dst, const T *stage, int n) {
    constexpr int E = 16 / sizeof(T);
    if ((reinterpret_cast<uintptr_t>(dst) & 15u) == 0 && n % E == 0) {
        for (int i = threadIdx.x; i < n / E; i += blockDim.x)
            __stcs(reinterpret_cast<uint4 *>(dst) + i, reinterpret_cast<const uint4 *>(stage)[i]);
    } else {
        for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = stage[i];
    }
}

// the shared-memory stage of an NHWC tile of N elements of T (one array per kernel instantiation that asks for it)
template <typename T, int N>
__device__ __forceinline__ T *nhwc_stage() {
    __shared__ __align__(16) unsigned char raw[N * sizeof(T)];
    return reinterpret_cast<T *>(raw);
}

__device__ __forceinline__ float clamp01(float a) { return fminf(fmaxf(a, 0.0f), 1.0f); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Sum of K per-thread values over the CTA; result valid in thread 0.
// smem: K * 32 floats.  Fixed order => deterministic for a fixed launch shape.
template <int K>
__device__ __forceinline__ void block_sum(float (&v)[K], float *smem) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        v[k] = warp_sum(v[k]);
        if (lane == 0) smem[k * 32 + wid] = v[k];
    }
    __syncthreads();
    if (wid == 0) {
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float t = lane < nw ? smem[k * 32 + lane] : 0.0f;
            v[k] = warp_sum(t);
        }
    }
}

// Grid-wide deterministic reduction tail: every CTA stores its K partials, the
// last CTA to arrive (ticket) sums all partials in a fixed order in double and
// calls fin(totals).  The ticket is left at 0 again.
template <int K, typename Fin>
__device__ __forceinline__ void grid_reduce_finish(float (&v)[K], void *workspace, float *smem, Fin fin) {
    static_assert(K <= kPartialsPerBlock, "too many partials");
    unsigned int *ticket = reinterpret_cast<unsigned int *>(workspace);
    float *partials = reinterpret_cast<float *>(reinterpret_cast<char *>(workspace) + kWsTicketBytes);
    __shared__ bool is_last;
    const unsigned int nblocks = gridDim.x * gridDim.y * gridDim.z;
    const unsigned int bid = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    constexpr int ROWS = (K + 3) / 4;  // float4 rows per CTA (stride kPartialsPerBlock / 4 rows)
    constexpr int RSTRIDE = kPartialsPerBlock / 4;
    block_sum<K>(v, smem);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int j = 0; j < ROWS; ++j) {
            float4 mine = make_float4(0.f, 0.f, 0.f, 0.f);
            float *mp = &mine.x;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (4 * j + k < K) mp[k] = v[4 * j + k];
            reinterpret_cast<float4 *>(partials)[bid * RSTRIDE + j] = mine;
        }
        __threadfence();
        unsigned int t = atomicAdd(ticket, 1u);
        is_last = (t == nblocks - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    double acc[K];
#pragma unroll
    for (int k = 0; k < K; ++k) acc[k] = 0.0;
    // 8 rows of partials in flight per thread: a plain loop here is a chain of exposed
    // L2 latencies (measured: 90 us for 16 K partials)
    constexpr int U = 8 / ROWS;
    for (unsigned int i0 = threadIdx.x; i0 < nblocks; i0 += U * blockDim.x) {
        float4 row[U][ROWS];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const unsigned int i = i0 + u * blockDim.x;
#pragma unroll
            for (int j = 0; j < ROWS; ++j)
                row[u][j] = i < nblocks ? __ldcg(reinterpret_cast<const float4 *>(partials) + i * RSTRIDE + j)
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
#pragma unroll
            for (int j = 0; j < ROWS; ++j) {
                const float r4[4] = {row[u][j].x, row[u][j].y, row[u][j].z, row[u][j].w};
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (4 * j + k < K) acc[4 * j + k] += (double)r4[k];
            }
        }
    }
    __shared__ double dsm[K * 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        acc[k] = warp_sum(acc[k]);
        if (lane == 0) dsm[k * 32 + wid] = acc[k];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot[K];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            tot[k] = 0.0;
            for (int w = 0; w < nw; ++w) tot[k] += dsm[k * 32 + w];
        }
        fin(tot);
        *ticket = 0u;
    }
}

#endif  // __CUDACC__
}  // namespace mt
