// corr_tc.cu - K2 on the 5th-generation tensor cores: tcgen05.mma (kind::tf32),
// operands staged by TMA, accumulators in TMEM, masks + L2 normalisation fused.
//
// Replaces CorrelationVGG.correlation_masked_4d, master_thesis/model_dfpn.py:534-565 (a7):
//   out[b,f,m,n] = sum_k ft[b,k,m] fr[b,k,f,n] * sa[b,m] * sb[b,f,n]
//   sa = v_t / (||ft * v_t||_2 + 1e-9)     (:551-560)     sb likewise for the reference (:561-562)
// i.e. the reference's "mask, normalise, matmul" with the two normalisations factored out of
// the contraction.  Masked rows / columns come out exactly 0 (scale 0 times a finite sum).
//
// One CTA computes one 256 x 256 output tile (= a whole (b, f) frame for the reference's
// 16 x 16 feature maps): two M = 128 accumulators of N = 256 columns fill the 512 TMEM columns,
// so every operand byte is loaded exactly once (128 x 128 tiles loaded everything twice:
// 7 TB/s of L2->SM traffic, tensor pipe 21 % active, profiles/).  K = C in slices of 32, 3-stage
// TMA ring (64 KB per stage).
//
// Warp roles (10 warps): 0 = TMA producer; 1 = TMEM owner + single-thread MMA issuer;
// 2..9 = norm + epilogue.  While the MMA warp consumes a stage, thread t of the 8 worker warps
// reads row t of the A tile and column t of the B tile from the same shared-memory stage
// (de-swizzled) and accumulates their sums of squares: the L2 norms cost no extra pass over
// the features and no extra launch (a separate scales kernel was 26 of 64 us at B=32, F=4).
// The smem slot is released by the MMA commit AND one arrival per worker warp.
// Epilogue: tcgen05.ld 32 lanes x 32 columns -> * sa[m] * sb[n] -> 128 B per-row stores.
//
// Data layout.  The features arrive fp32 and MN-major: ft (B,C,P) and fr (B,C,F,P) have the
// pixel index contiguous, the contraction index (channel) strided.  They are consumed AS IS:
// kind::tf32 reads fp32 words from shared memory (10-bit mantissa used), and both operands use
// MN-major shared-memory descriptors.  For MN-major tf32 operands the ONLY legal shared-memory
// layout is "128 B swizzle with a 32 B base" (UMMA layout type 1, Swizzle<2,5,2>: the four 32 B
// chunks of a 128 B row are permuted by the row index mod 4; a plain SWIZZLE_128B descriptor
// is silently ignored - the first version of this kernel produced zeros).  TMA boxes of
// {32 pixels = 128 B, 32 channels, 8 pixel groups} with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B land
// exactly in that canonical layout:
//   4 channel rows x 128 B = one 512 B swizzle atom; SBO = 512 B between 4-channel groups;
//   LBO = BK * 128 B between 32-pixel groups; one MMA (K = 8) spans two atoms.
//
// fp16 / bf16 features (the VGG's output under autocast) run the same single-CTA kernel as kind::f16, through the
// operand traits CorrOp<T>: the exact half values are multiplied with fp32 accumulation, the two norm scales applied
// in the fp32 epilogue and the volume rounded once, on store, to the features' dtype.  For 16-bit MN-major operands
// the canonical layout is the ordinary 128 B swizzle (UMMA layout type 2, Swizzle<3,4,3>: the eight 16 B chunks of
// a 128 B row are permuted by the row index mod 8), NOT the tf32 "32 B base" one.  TMA boxes of {64 pixels = 128 B,
// 64 channels, pixel groups} with CU_TENSOR_MAP_SWIZZLE_128B land in it:
//   8 channel rows x 128 B = one 1024 B atom; SBO = 1024 B between 8-channel groups;
//   LBO = BK * 128 B between 64-pixel groups; one MMA (K = 16) spans two atoms.
// A stage holds 128 B per pixel in both cases (32 fp32 or 64 half channels), so the rings and tile shapes are shared.
#include <cuda.h>

#include <type_traits>

#include "mt_common.cuh"
#include "mt_tma.cuh"

namespace mt {

// L1 mode of the launchers (see CorrTcArgs): prediction to compare with, loss scalar, optional int8 signs, partial sums
struct CorrL1 {
    const void *pred;   // in the features' element type
    float *loss;
    signed char *sign;
    float *partials;
};

namespace {

constexpr int kTile = 256;        // largest output tile: TM rows (one or two UMMA M = 128 halves) x TN <= 256 columns
constexpr int kBK = 32;
constexpr int kUmmaK = 8;         // tf32: 32 B of K per instruction
// The correlation kernels only wait and leave griddepcontrol.launch_dependents to their exit (see pdl_sync).  With the
// library's default trigger right after the wait, the next kernel's CTAs would take their SM slots while this kernel
// runs: it holds ~200 KB of shared memory per SM, the pre-launched CTAs arrive while the SM is in its
// maximum-shared-memory configuration, and because from then on an SM is never empty between PDL-chained kernels the
// configuration (a few KB of L1) sticks - the gather kernels that follow run with almost no L1.  Measured
// (profiles/r2_experiments.md, call Z): warp_l1_fwd at 256 x 256 77 -> 121 us several launches after a correlation;
// cfg3 step 431 -> 364 us, cfg1 20.0 -> 18.4 us, default workload 100.9 -> 97.7 us with the trigger left to the exit.
constexpr bool kPairDefault = true;   // CTA-pair kernel for large batches (see the heuristic in corr4d_tc_launch_ex)

// MN-major, SWIZZLE_128B_BASE32B shared-memory matrix descriptor (sm_100 "version 1").
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);            // start address  [0,14)
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16;   // leading byte offset [16,30)
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32;   // stride byte offset  [32,46)
    d |= (uint64_t)1 << 46;                               // descriptor version (Blackwell)
    d |= (uint64_t)1 << 61;                               // layout type: SWIZZLE_128B_BASE32B
    return d;
}
// kind::tf32, fp32 accumulate, A and B MN-major, M x N
constexpr uint32_t instr_desc(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// byte offset of element (pixel p of the tile, channel k of the stage) in a staged operand:
// [8 pixel groups][32 channels][128 B], 32 B chunks XOR-ed with (k mod 4)  (Swizzle<2,5,2>)
__device__ __forceinline__ uint32_t staged_offset(int p, int k) {
    const int g = p >> 5, px = p & 31;
    return (uint32_t)(g * (kBK * 128) + k * 128 + ((((px >> 3) ^ (k & 3)) << 5) | ((px & 7) << 2)));
}

// Operand traits of corr_tc_kernel: how features of element type T are staged, normalised and multiplied.
template <typename T>
struct CorrOp;
template <>
struct CorrOp<float> {  // kind::tf32 on the fp32 words
    static constexpr int kBK = 32, kUmmaK = 8, kPhase = 4, kAtomBytes = 512, kGroupPx = 32;
    static constexpr CUtensorMapDataType kTmaType = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    static constexpr CUtensorMapSwizzle kTmaSwizzle = CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
    static constexpr uint32_t instr(int M, int N) { return instr_desc(M, N); }
    __device__ static uint64_t desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) { return umma_desc(saddr, lbo, sbo); }
    __device__ static void mma(uint32_t d, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
        umma_tf32(d, ad, bd, idesc, acc);
    }
    __device__ static uint32_t offset(int p, int k) { return staged_offset(p, k); }
    __device__ static float load(const uint8_t *p) { return *reinterpret_cast<const float *>(p); }
};
template <typename T, uint32_t kFmt, CUtensorMapDataType kTma>
struct CorrOpHalf {  // kind::f16; kFmt: a / b format of the instruction descriptor (F16 = 0, BF16 = 1)
    static constexpr int kBK = 64, kUmmaK = 16, kPhase = 8, kAtomBytes = 1024, kGroupPx = 64;
    static constexpr CUtensorMapDataType kTmaType = kTma;
    static constexpr CUtensorMapSwizzle kTmaSwizzle = CU_TENSOR_MAP_SWIZZLE_128B;
    // fp32 accumulate, A and B MN-major, M x N
    static constexpr uint32_t instr(int M, int N) {
        return (1u << 4) | (kFmt << 7) | (kFmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
               ((uint32_t)(M >> 4) << 24);
    }
    // MN-major SWIZZLE_128B descriptor (sm_100 "version 1", layout type 2)
    __device__ static uint64_t desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
        uint64_t d = 0;
        d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
        d |= (uint64_t)((lbo >> 4) & 0x3FFFu) << 16;
        d |= (uint64_t)((sbo >> 4) & 0x3FFFu) << 32;
        d |= (uint64_t)1 << 46;
        d |= (uint64_t)2 << 61;
        return d;
    }
    __device__ static void mma(uint32_t d, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
            ::"r"(d), "l"(ad), "l"(bd), "r"(idesc), "r"(acc) : "memory");
    }
    // [pixel groups of 64][64 channels][128 B], 16 B chunks XOR-ed with (k mod 8)  (Swizzle<3,4,3>)
    __device__ static uint32_t offset(int p, int k) {
        const int g = p >> 6, px = p & 63;
        return (uint32_t)(g * (kBK * 128) + k * 128 + ((((px >> 3) ^ (k & 7)) << 4) | ((px & 7) << 1)));
    }
    __device__ static float load(const uint8_t *p) { return widen(*reinterpret_cast<const T *>(p)); }
};
template <>
struct CorrOp<__half> : CorrOpHalf<__half, 0u, CU_TENSOR_MAP_DATA_TYPE_FLOAT16> {};
template <>
struct CorrOp<__nv_bfloat16> : CorrOpHalf<__nv_bfloat16, 1u, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16> {};

struct CorrTcArgs {
    // visibilities at feature resolution (mask_mode 0; NULL = all ones), or full-resolution masks m
    // (mask_mode 1): v = 1 - m[nearest source pixel], CorrelationVGG.forward model_dfpn.py:521-526
    const float *vt; int64_t vt_sb;                // (B, P) | (B, MH, MW)
    const float *vr; int64_t vr_sb, vr_sf;         // (B, F, P) | (B, F, MH, MW)
    int mask_mode, MH, MW, fw;
    float msy, msx;                                // MH / fh, MW / fw in fp32 (ATen nearest: floor(dst * scale))
    void *out;                                     // (B, F, P, P) in the features' dtype; unused in L1 mode
    // L1 mode (pred != NULL): the volume is not written; the epilogue compares it with `pred` (B, F, P, P) instead and
    // accumulates sum |pred - corr| (F.l1_loss(corr, corr_y), model_dfpn.py:254-257, SURVEY 8f-3).  sign (optional):
    // sign(pred - corr) as int8, all the backward pass needs.  partials: one float per (CTA, epilogue warp); the last
    // epilogue warp of the grid to finish (ticket) folds them in a fixed order and writes the mean to loss[0].
    const void *pred;                              // in the features' element type T
    signed char *sign;
    float *partials;
    unsigned int *ticket;                          // zero between launches: counts the epilogue warps that are done
    float *loss;
    double inv_count;                              // 1 / (B F P P)
    int C, F, P, tiles_m, tiles_n, n_tiles;
};

// visibility of feature pixel p of plane `base` (see CorrTcArgs)
__device__ __forceinline__ float corr_vis(const float *base, int p, const CorrTcArgs &a) {
    if (!base) return 1.0f;
    if (!a.mask_mode) return __ldg(base + p);
    const int y = p / a.fw, x = p - y * a.fw;
    const int ys = min((int)floorf(__fmul_rn((float)y, a.msy)), a.MH - 1);
    const int xs = min((int)floorf(__fmul_rn((float)x, a.msx)), a.MW - 1);
    return __fsub_rn(1.0f, __ldg(base + (int64_t)ys * a.MW + xs));
}

constexpr int kEpiPitch = 36;     // floats per staged row: 144 B keeps float4 alignment, conflict-free both ways

__device__ __forceinline__ signed char sign_i8(float d) { return d > 0.0f ? 1 : (d < 0.0f ? -1 : 0); }

// Epilogue of one 32-row x TN-column block of a tile (one warp = one TMEM lane quarter): tcgen05.ld 32 lanes x 32
// columns -> * sa[row] * sb[col] -> transposed through the warp's private staging tile `st` -> 128 B-per-row
// coalesced streaming stores of the volume, or (L1) the same rows of `pred` loaded instead (requested before the
// TMEM read so that their latency hides under it) and |pred - corr| accumulated into `acc`.
// `off0`: element offset of (first row of the block, first column of the tile) in the (B, F, P, P) volume.
// OT: element type of the volume and of `pred` (float, or the half features' type: each value of the volume rounded
// once, to nearest even; in L1 mode that rounded value, widened again, is compared with the widened `pred` - the
// eager l1_loss of two half volumes runs in fp32 under autocast).
template <typename OT> __device__ __forceinline__ float4 widen4(const float4 &v) { return v; }
template <typename OT> __device__ __forceinline__ float4 widen4(const uint2 &u) {
    const OT *e = reinterpret_cast<const OT *>(&u);
    return make_float4(widen(e[0]), widen(e[1]), widen(e[2]), widen(e[3]));
}
template <int TN, bool L1, typename OT = float>
__device__ __forceinline__ void corr_epi_block(const CorrTcArgs &a, uint32_t taddr, float sa, const float *sbv, float *st,
                                               int64_t off0, int lane, float &acc) {
    const int rr = lane >> 3, c4 = (lane & 7) * 4;  // read-back: 4 rows x 8 float4 per instruction
    using Pred4 = std::conditional_t<sizeof(OT) == 4, float4, uint2>;  // 4 elements of pred: 16 B of fp32, 8 B of half
    const OT *pred = static_cast<const OT *>(a.pred);
#pragma unroll 1
    for (int c0 = 0; c0 < TN; c0 += 32) {
        // pred rows: the first half is requested before the TMEM read, the second once the accumulator registers
        // are free again (the lines were brought into L2 while the main loop ran, see corr_epi_prefetch)
        Pred4 p[2][4];
        if (L1) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                p[0][j] = __ldcs(reinterpret_cast<const Pred4 *>(pred + off0 + (int64_t)(j * 4 + rr) * a.P + c0 + c4));
        }
        {
            float v[32];
            tmem_ld32(taddr + (uint32_t)c0, v);
#pragma unroll
            for (int i = 0; i < 32; i += 4) {
                float4 o;
                o.x = v[i] * sa * sbv[c0 + i];
                o.y = v[i + 1] * sa * sbv[c0 + i + 1];
                o.z = v[i + 2] * sa * sbv[c0 + i + 2];
                o.w = v[i + 3] * sa * sbv[c0 + i + 3];
                *reinterpret_cast<float4 *>(st + lane * kEpiPitch + i) = o;  // row = lane
            }
        }
        if (L1) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                p[1][j] = __ldcs(reinterpret_cast<const Pred4 *>(pred + off0 + (int64_t)((4 + j) * 4 + rr) * a.P + c0 + c4));
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int row = j * 4 + rr;
            const float4 o = *reinterpret_cast<const float4 *>(st + row * kEpiPitch + c4);
            const int64_t off = off0 + (int64_t)row * a.P + c0 + c4;
            if (L1) {
                const float4 pj = widen4<OT>(p[j >> 2][j & 3]);
                float4 v = o;
                if constexpr (sizeof(OT) == 2)  // the value the store mode writes, widened again
                    v = make_float4(widen(narrow<OT>(o.x)), widen(narrow<OT>(o.y)), widen(narrow<OT>(o.z)),
                                    widen(narrow<OT>(o.w)));
                const float dx = pj.x - v.x, dy = pj.y - v.y, dz = pj.z - v.z, dw = pj.w - v.w;
                acc += (fabsf(dx) + fabsf(dy)) + (fabsf(dz) + fabsf(dw));
                if (a.sign) {
                    char4 sg;
                    sg.x = sign_i8(dx); sg.y = sign_i8(dy); sg.z = sign_i8(dz); sg.w = sign_i8(dw);
                    *reinterpret_cast<char4 *>(a.sign + off) = sg;
                }
            } else if constexpr (sizeof(OT) == 4) {
                __stcs(reinterpret_cast<float4 *>(static_cast<float *>(a.out) + off), o);
            } else {
                uint2 u;
                OT *e = reinterpret_cast<OT *>(&u);
                e[0] = narrow<OT>(o.x); e[1] = narrow<OT>(o.y); e[2] = narrow<OT>(o.z); e[3] = narrow<OT>(o.w);
                __stcs(reinterpret_cast<uint2 *>(static_cast<OT *>(a.out) + off), u);
            }
        }
        __syncwarp();
    }
}

// L1 mode: lane = row of a 32-row block; asks the L2 for the TN columns of that row of `pred` (elements of OT), one
// prefetch per 128 B line.  Issued by the epilogue warps before they wait for the accumulators, so the lines arrive
// while the main loop of the tile runs.
template <int TN, typename OT = float>
__device__ __forceinline__ void corr_epi_prefetch(const CorrTcArgs &a, int64_t off0, int lane) {
    const OT *row = static_cast<const OT *>(a.pred) + off0 + (int64_t)lane * a.P;
#pragma unroll
    for (int c = 0; c < TN; c += 128 / (int)sizeof(OT)) asm volatile("prefetch.global.L2 [%0];" ::"l"(row + c));
}

// L1 mode, end of an epilogue warp's tile loop: publish the warp's partial sum; the last warp of the grid to arrive
// sums all n_slots partials (lane-strided, then a butterfly, in double: the order depends on the launch shape only),
// writes the mean and re-arms the ticket.  No second launch (a one-CTA fold kernel cost 5.5 us, ncu g2).
__device__ __forceinline__ void corr_l1_tail(const CorrTcArgs &a, float acc, int slot, int n_slots, int lane) {
    acc = warp_sum(acc);
    unsigned int t = 0u;
    if (lane == 0) {
        a.partials[slot] = acc;
        __threadfence();
        t = atomicAdd(a.ticket, 1u);
    }
    t = __shfl_sync(0xffffffffu, t, 0);
    if (t != (unsigned int)n_slots - 1u) return;
    __threadfence();
    double s = 0.0;
    for (int i = lane; i < n_slots; i += 32) s += (double)__ldcg(a.partials + i);
    s = warp_sum(s);
    if (lane == 0) {
        a.loss[0] = (float)(s * a.inv_count);
        *a.ticket = 0u;
    }
}

constexpr int kNormWarps = 8;     // one thread per row of the A tile / column of the B tile
constexpr int kEpiWarps = 4;      // one per TMEM lane quarter
constexpr int kThreadsP = (2 + kNormWarps + kEpiWarps) * 32;
constexpr int kEpiBytes = kEpiWarps * 32 * kEpiPitch * 4;

template <int TM, int TN, int STAGES>
constexpr int smem_bytes_p() {
    return STAGES * ((TM + TN) * kBK * 4) + kEpiBytes + 2 * (kTile + kTile) * 4 /*scales*/ + 256 /*barriers*/ +
           1024 /*alignment*/;
}

// Persistent kernel: one CTA per SM walks the output tiles (TM rows x TN columns of one (b, f) frame) in a
// static round-robin.  TM = 256, TN = 256 loads every operand byte once (large batches); smaller tiles split a
// frame over 2 .. 8 CTAs so that small batches still occupy the machine (the operands are then re-read from L2).
// Warp roles (14 warps):
//   warp 0      TMA producer: runs ahead over tile boundaries, bounded only by the smem ring
//   warp 1      TMEM owner + single-thread tcgen05.mma issuer; accumulator buffers of 2 x TN fp32 columns
//               (two M = 128 halves): two buffers for TN <= 128, so the MMAs of tile i + 1 start while the
//               epilogue of tile i is still draining its buffer
//   warps 2-9   norms: thread t accumulates sum x^2 of row t of the A tile and column t of the B tile from the
//               staged (swizzled) operands while the tensor cores consume the same stage, then publishes the
//               row / column scales of the tile (double-buffered)
//   warps 10-13 epilogue: tcgen05.ld 32 lanes x 32 columns -> * sa[m] * sb[n] -> transposed through a private
//               4.5 KB staging tile -> 128 B-per-row coalesced streaming stores (4 full lines per instruction; the
//               first version stored 16 B per lane straight from the TMEM layout: 32 half-used sectors per
//               instruction, which made the epilogue as long as the main loop)
// Barriers: full/empty per smem stage (empty = MMA commit + one arrival per norm warp), tmem_full / tmem_empty and
// scales_ready per accumulator buffer.
// T: element type of the features (CorrOp<T>); the volume is written in it.
template <typename T, int TM, int TN, int kStages>
__global__ void __launch_bounds__(kThreadsP, 1)
corr_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
               const CorrTcArgs a) {
    using Op = CorrOp<T>;
    static_assert(Op::kBK * sizeof(T) == kBK * 4, "a stage holds 128 B per pixel for every operand type");
    constexpr int kHalves = TM / 128;                 // UMMA M = 128 accumulators per tile
    constexpr int kStageBytesA = TM * Op::kBK * (int)sizeof(T), kStageBytesB = TN * Op::kBK * (int)sizeof(T);
    constexpr int kBufCols = kHalves * TN;            // TMEM columns per accumulator buffer
    constexpr int kBufs = 2 * kBufCols <= 512 ? 2 : 1;  // accumulator buffers
    extern __shared__ uint8_t smem_raw[];
    // 1024 B alignment (swizzle atoms) as an OFFSET from the declared array: a round trip through uintptr_t loses
    // the shared address space and every access below became a generic LD.E / ST.E (ncu r2e: the norm warps'
    // 64 loads per stage and the epilogue staging were all generic; stall reason "lg")
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *smem_a = smem;
    uint8_t *smem_b = smem + kStages * kStageBytesA;
    float *epi = reinterpret_cast<float *>(smem + kStages * (kStageBytesA + kStageBytesB));
    float *s_sa = epi + kEpiWarps * 32 * kEpiPitch;   // [2][kTile] row scales
    float *s_sb = s_sa + 2 * kTile;                   // [2][kTile] column scales (TN used)
    uint64_t *bars = reinterpret_cast<uint64_t *>(s_sb + 2 * kTile);
    uint64_t *full = bars, *empty = bars + kStages, *tmem_full = bars + 2 * kStages, *tmem_empty = tmem_full + 2,
             *scales_ready = tmem_empty + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(scales_ready + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_k = a.C / Op::kBK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
        for (int s = 0; s < kStages; ++s) {
            mbar_init(smem_u32(full + s), 1);
            mbar_init(smem_u32(empty + s), 1 + kNormWarps);  // MMA commit + one arrival per norm warp
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(smem_u32(tmem_full + i), 1);
            mbar_init(smem_u32(tmem_empty + i), kEpiWarps);
            mbar_init(smem_u32(scales_ready + i), kNormWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: all 512 columns (1 CTA per SM)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    // everything above is on-chip setup and overlaps the tail of the previous kernel (PDL)
    pdl_wait();

    const int tiles_per_frame = a.tiles_m * a.tiles_n;
    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
                const int frame = tile / tiles_per_frame, r = tile - frame * tiles_per_frame;
                const int m_tile = r / a.tiles_n, n_tile = r - m_tile * a.tiles_n;
                const int b = frame / a.F, f = frame - b * a.F;
                for (int kb = 0; kb < num_k; ++kb, ++it) {
                    const int s = it % kStages;
                    const uint32_t ph = (it / kStages) & 1;
                    mbar_wait(smem_u32(empty + s), ph ^ 1);
                    mbar_expect_tx(smem_u32(full + s), kStageBytesA + kStageBytesB);
                    // A: (pixel-in-group G, channel C, pixel group P/G, batch B), G = Op::kGroupPx
                    tma_load_4d(smem_u32(smem_a + s * kStageBytesA), &map_a, smem_u32(full + s), 0, kb * Op::kBK,
                                m_tile * (TM / Op::kGroupPx), b);
                    // B: (pixel-in-group G, channel C, pixel group P/G, frame F, batch B)
                    tma_load_5d(smem_u32(smem_b + s * kStageBytesB), &map_b, smem_u32(full + s), 0, kb * Op::kBK,
                                n_tile * (TN / Op::kGroupPx), f, b);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one elected lane) =====
        if (lane == 0) {
            constexpr uint32_t idesc = Op::instr(128, TN);
            uint32_t it = 0;
            int ti = 0;
            for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++ti) {
                const int buf = ti % kBufs;
                const uint32_t use = (uint32_t)(ti / kBufs);
                mbar_wait(smem_u32(tmem_empty + buf), (use & 1) ^ 1);  // the epilogue has drained this buffer
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t acc = tmem_base + buf * kBufCols;
                for (int kb = 0; kb < num_k; ++kb, ++it) {
                    const int s = it % kStages;
                    const uint32_t ph = (it / kStages) & 1;
                    mbar_wait(smem_u32(full + s), ph);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a0 = smem_u32(smem_a + s * kStageBytesA), b0 = smem_u32(smem_b + s * kStageBytesB);
                    // K advance inside the stage: next kUmmaK channels = two atoms (tf32 +1024 B, f16 +2048 B);
                    // M halves: the A stage's pixel groups of the first and the second 128 pixels
                    constexpr int kKStep = (Op::kUmmaK / Op::kPhase) * Op::kAtomBytes;
                    constexpr int kHalfStep = (128 / Op::kGroupPx) * Op::kBK * 128;
#pragma unroll
                    for (int j = 0; j < Op::kBK / Op::kUmmaK; ++j) {
                        const uint64_t bd = Op::desc(b0 + j * kKStep, Op::kBK * 128, Op::kAtomBytes);
#pragma unroll
                        for (int h = 0; h < kHalves; ++h) {
                            const uint64_t ad = Op::desc(a0 + h * kHalfStep + j * kKStep, Op::kBK * 128, Op::kAtomBytes);
                            Op::mma(acc + h * TN, ad, bd, idesc, (kb | j) != 0 ? 1u : 0u);
                        }
                    }
                    umma_commit(smem_u32(empty + s));  // frees the smem slot when these MMAs retire
                }
                umma_commit(smem_u32(tmem_full + buf));  // accumulators of this tile complete
            }
        }
    } else if (warp < 2 + kNormWarps) {
        // ===== norm warps =====
        // thread -> row ra of the A tile and / or column cb of the B tile (warp-uniform: TM, TN are multiples of 64).
        // Small tiles give the two operands to different warps, large ones give every thread one of each.
        const int t = threadIdx.x - 64;  // 0..255
        constexpr bool kSplit = TM + TN <= 256;
        const bool has_a = t < TM, has_b = kSplit ? (t >= TM && t < TM + TN) : (t < TN);
        const int ta = has_a ? t : 0, tb = has_b ? (kSplit ? t - TM : t) : 0;
        // the swizzle phase repeats every kPhase channels: channel k = kPhase j + r lives at base[r] + atom * j,
        // so the loop below is kBK LDS with immediate offsets + kBK FFMA per operand, no address math (half values
        // are widened before they are squared)
        uint32_t base_a[Op::kPhase], base_b[Op::kPhase];
#pragma unroll
        for (int r = 0; r < Op::kPhase; ++r) { base_a[r] = Op::offset(ta, r); base_b[r] = Op::offset(tb, r); }
        uint32_t it = 0;
        int ti = 0;
        for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++ti) {
            const int frame = tile / tiles_per_frame, r0 = tile - frame * tiles_per_frame;
            const int m_tile = r0 / a.tiles_n, n_tile = r0 - m_tile * a.tiles_n;
            const int b = frame / a.F, f = frame - b * a.F;
            // the visibilities are needed at the end of the main loop only: request them first
            const float vt = corr_vis(a.vt ? a.vt + (int64_t)b * a.vt_sb : nullptr, m_tile * TM + ta, a);
            const float vr = corr_vis(a.vr ? a.vr + (int64_t)b * a.vr_sb + (int64_t)f * a.vr_sf : nullptr,
                                      n_tile * TN + tb, a);
            float qa[4] = {0.f, 0.f, 0.f, 0.f}, qb[4] = {0.f, 0.f, 0.f, 0.f};
            for (int kb = 0; kb < num_k; ++kb, ++it) {
                const int s = it % kStages;
                const uint32_t ph = (it / kStages) & 1;
                mbar_wait(smem_u32(full + s), ph);
                const uint8_t *pa = smem_a + s * kStageBytesA, *pb = smem_b + s * kStageBytesB;
                if (has_a) {
#pragma unroll
                    for (int r = 0; r < Op::kPhase; ++r) {
#pragma unroll
                        for (int j = 0; j < Op::kBK / Op::kPhase; ++j) {
                            const float va = Op::load(pa + base_a[r] + j * Op::kAtomBytes);
                            qa[r & 3] = __fmaf_rn(va, va, qa[r & 3]);
                        }
                    }
                }
                if (has_b) {
#pragma unroll
                    for (int r = 0; r < Op::kPhase; ++r) {
#pragma unroll
                        for (int j = 0; j < Op::kBK / Op::kPhase; ++j) {
                            const float vb = Op::load(pb + base_b[r] + j * Op::kAtomBytes);
                            qb[r & 3] = __fmaf_rn(vb, vb, qb[r & 3]);
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(smem_u32(empty + s));
            }
            const float ssa = (qa[0] + qa[1]) + (qa[2] + qa[3]), ssb = (qb[0] + qb[1]) + (qb[2] + qb[3]);
            const int buf = ti % kBufs;
            const uint32_t use = (uint32_t)(ti / kBufs);
            // the scale tables of this buffer are free once the epilogue of its previous tile has finished
            mbar_wait(smem_u32(tmem_empty + buf), (use & 1) ^ 1);
            // scales: v / (|v| * ||f|| + 1e-9)   (||f * v|| = |v| * ||f||)
            if (has_a) s_sa[buf * kTile + ta] = __fdiv_rn(vt, __fadd_rn(__fmul_rn(fabsf(vt), sqrtf(ssa)), 1e-9f));
            if (has_b) s_sb[buf * kTile + tb] = __fdiv_rn(vr, __fadd_rn(__fmul_rn(fabsf(vr), sqrtf(ssb)), 1e-9f));
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(scales_ready + buf));
        }
    } else {
        // ===== epilogue warps =====
        // TMEM lane-quarter rule: warp w may touch lanes 32*(w%4)..32*(w%4)+31; warps 10..13 cover all four
        const int lq = warp & 3, ew = warp - (2 + kNormWarps);
        float *st = epi + ew * 32 * kEpiPitch;
        float l1_acc = 0.0f;
        int ti = 0;
        for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++ti) {
            const int frame = tile / tiles_per_frame, r0 = tile - frame * tiles_per_frame;
            const int m_tile = r0 / a.tiles_n, n_tile = r0 - m_tile * a.tiles_n;
            const int buf = ti % kBufs;
            const uint32_t use = (uint32_t)(ti / kBufs);
            if (a.pred) {
#pragma unroll
                for (int h = 0; h < kHalves; ++h)
                    corr_epi_prefetch<TN, T>(a, ((int64_t)frame * a.P + m_tile * TM + h * 128 + lq * 32) * a.P + n_tile * TN, lane);
            }
            mbar_wait(smem_u32(scales_ready + buf), use & 1);
            mbar_wait(smem_u32(tmem_full + buf), use & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const float *sbv = s_sb + buf * kTile;
#pragma unroll 1
            for (int h = 0; h < kHalves; ++h) {
                const int row0 = h * 128 + lq * 32;  // first row of this warp's 32-row block
                const float sa = s_sa[buf * kTile + row0 + lane];
                const int64_t off0 = ((int64_t)frame * a.P + m_tile * TM + row0) * a.P + n_tile * TN;
                const uint32_t taddr = tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)(buf * kBufCols + h * TN);
                if (a.pred) corr_epi_block<TN, true, T>(a, taddr, sa, sbv, st, off0, lane, l1_acc);
                else corr_epi_block<TN, false, T>(a, taddr, sa, sbv, st, off0, lane, l1_acc);
            }
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(tmem_empty + buf));
        }
        if (a.pred) corr_l1_tail(a, l1_acc, blockIdx.x * kEpiWarps + ew, gridDim.x * kEpiWarps, lane);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
    }
}


// ======================================================================================================
// CTA-PAIR variant (tcgen05 cta_group::2).  ncu on the single-CTA kernel above: the 128 B/clk of shared-memory
// bandwidth per SM - TMA writes + UMMA operand reads + the norm warps' reads - bound it, not HBM or the tensor
// pipe.  Two CTAs of a cluster on the two SMs of a TPC compute one 256 x TN tile with M = 256 instructions: each
// CTA stages ITS 128 rows of A and ITS TN / 2 columns of B (half the TMA writes and half the operand reads per
// SM), the leader's single thread issues the MMAs for both tensor cores, each CTA's TMEM receives its 128
// rows x TN columns, so two accumulator buffers fit even for whole-frame tiles (TN = 256).
// Hand-offs that cross the pair:
//   * peer_full[s]  (leader): the peer's relay thread (its otherwise idle warp 1) forwards "my stage s has landed";
//   * empty[s], tmem_full[b]: tcgen05.commit ... multicast::cluster arrives in both CTAs;
//   * tmem_empty[b] (both): every epilogue warp arrives locally and on the peer - the leader may overwrite the
//     accumulators, and either CTA's norm warps the scale tables, only when BOTH epilogues have drained them;
//   * column scales: a CTA only sees its own TN / 2 columns of B, so its B-norm warps write sb into both CTAs'
//     tables (st.shared::cluster) and arrive on both scales_ready[b].
// ======================================================================================================
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t rank) {
    uint32_t d;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(d) : "r"(saddr), "r"(rank));
    return d;
}
__device__ __forceinline__ void mbar_arrive_remote(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// relaxed: for a thread that only forwards a signal.  A release arrive waits for the thread's previous remote
// operation to be performed, which serialised the relay at one remote round trip (~1.2 us) per pipeline stage.
__device__ __forceinline__ void mbar_arrive_remote_relaxed(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void st_remote_f32(uint32_t cluster_addr, float v) {
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(cluster_addr), "f"(v) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// wait with acquire at cluster scope: the phase may have been completed by the other CTA of the pair
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0, spins = 0;
    do {
#ifdef MT_PAIR_TESTWAIT
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.test_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
#else
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
#endif
        if (!ok && ++spins > (1u << 28)) __trap();
    } while (!ok);
}
__device__ __forceinline__ void umma2_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
    const uint32_t z = 0u;  // disable-output-lane mask: none
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(z) : "memory");
}
__device__ __forceinline__ void umma2_commit(uint32_t bar) {  // arrives on the barrier at this offset in BOTH CTAs
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(bar), "h"(mask) : "memory");
}

template <int TN, int STAGES>
constexpr int smem_bytes_pair() {
    return STAGES * ((128 + TN / 2) * kBK * 4) + kEpiBytes + 2 * (128 + kTile) * 4 /*scales*/ + 512 /*barriers*/ +
           1024 /*alignment*/;
}

template <int TN, int kStages>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreadsP, 1)
corr_tc2_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                const CorrTcArgs a) {
    constexpr int TNH = TN / 2;                        // B columns staged by each CTA
    constexpr int kStageBytesA = 128 * kBK * 4, kStageBytesB = TNH * kBK * 4;
    constexpr int kBufs = 2;                           // accumulator buffers of TN columns (128 lanes per CTA)
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *smem_a = smem;
    uint8_t *smem_b = smem + kStages * kStageBytesA;
    float *epi = reinterpret_cast<float *>(smem + kStages * (kStageBytesA + kStageBytesB));
    float *s_sa = epi + kEpiWarps * 32 * kEpiPitch;   // [2][128] row scales of this CTA's rows
    float *s_sb = s_sa + 2 * 128;                     // [2][kTile] column scales of the whole tile
    uint64_t *bars = reinterpret_cast<uint64_t *>(s_sb + 2 * kTile);
    uint64_t *full = bars, *empty = bars + kStages, *peer_full = bars + 2 * kStages, *tmem_full = bars + 3 * kStages,
             *tmem_empty = tmem_full + 2, *scales_ready = tmem_empty + 2;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(scales_ready + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank(), other = rank ^ 1u;
    const int pair = (int)blockIdx.x >> 1, npairs = (int)gridDim.x >> 1;
    const int num_k = a.C / kBK;

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_a) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&map_b) : "memory");
        for (int s = 0; s < kStages; ++s) {
            mbar_init(smem_u32(full + s), 1);
            mbar_init(smem_u32(empty + s), 1 + kNormWarps);  // MMA commit (multicast) + one arrival per local norm warp
            mbar_init(smem_u32(peer_full + s), 1);           // leader only: the peer's relay
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(smem_u32(tmem_full + i), 1);
            mbar_init(smem_u32(tmem_empty + i), 2 * kEpiWarps);               // the epilogue warps of both CTAs
            mbar_init(smem_u32(scales_ready + i), kNormWarps + kNormWarps / 2);  // local norm warps + the peer's B-norm warps
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: all 512 columns in both CTAs of the pair (the same warp id in both issues the alloc)
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                     ::"r"(smem_u32(tmem_slot)), "n"(512) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_sync_all();  // barriers of both CTAs initialised before anyone arrives remotely
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();

    const int tiles_per_frame = a.tiles_m * a.tiles_n;
    if (warp == 0) {
        // ===== TMA producer: this CTA's 128 rows of A and TN / 2 columns of B =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int tile = pair; tile < a.n_tiles; tile += npairs) {
                const int frame = tile / tiles_per_frame, r = tile - frame * tiles_per_frame;
                const int m_tile = r / a.tiles_n, n_tile = r - m_tile * a.tiles_n;
                const int b = frame / a.F, f = frame - b * a.F;
                for (int kb = 0; kb < num_k; ++kb, ++it) {
                    const int s = it % kStages;
                    const uint32_t ph = (it / kStages) & 1;
                    mbar_wait(smem_u32(empty + s), ph ^ 1);
                    mbar_expect_tx(smem_u32(full + s), kStageBytesA + kStageBytesB);
                    tma_load_4d(smem_u32(smem_a + s * kStageBytesA), &map_a, smem_u32(full + s), 0, kb * kBK,
                                m_tile * (kTile / 32) + (int)rank * 4, b);
                    tma_load_5d(smem_u32(smem_b + s * kStageBytesB), &map_b, smem_u32(full + s), 0, kb * kBK,
                                n_tile * (TN / 32) + (int)rank * (TNH / 32), f, b);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0 && rank == 0) {
            // ===== MMA issuer (leader CTA, one thread): M = 256 over the pair =====
            constexpr uint32_t idesc = instr_desc(256, TN);
            uint32_t it = 0;
            int ti = 0;
            for (int tile = pair; tile < a.n_tiles; tile += npairs, ++ti) {
                const int buf = ti % kBufs;
                const uint32_t use = (uint32_t)(ti / kBufs);
                mbar_wait_cluster(smem_u32(tmem_empty + buf), (use & 1) ^ 1);  // both epilogues have drained this buffer
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t acc = tmem_base + buf * TN;
                for (int kb = 0; kb < num_k; ++kb, ++it) {
                    const int s = it % kStages;
                    const uint32_t ph = (it / kStages) & 1;
                    mbar_wait(smem_u32(full + s), ph);
                    mbar_wait(smem_u32(peer_full + s), ph);  // remote arrival; the operands are read by the async proxy only
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint32_t a0 = smem_u32(smem_a + s * kStageBytesA), b0 = smem_u32(smem_b + s * kStageBytesB);
#pragma unroll
                    for (int j = 0; j < kBK / kUmmaK; ++j)
                        umma2_tf32(acc, umma_desc(a0 + j * 1024, kBK * 128, 512), umma_desc(b0 + j * 1024, kBK * 128, 512),
                                   idesc, (kb | j) != 0 ? 1u : 0u);
                    umma2_commit(smem_u32(empty + s));  // frees stage s in both CTAs when these MMAs retire
                }
                umma2_commit(smem_u32(tmem_full + buf));
            }
        } else if (lane == 0) {
            // ===== relay (peer CTA): tell the leader that this CTA's stage has landed =====
            const uint32_t leader_bar = mapa_u32(smem_u32(peer_full), 0);
            uint32_t it = 0;
            for (int tile = pair; tile < a.n_tiles; tile += npairs) {
                for (int kb = 0; kb < num_k; ++kb, ++it) {
                    const int s = it % kStages;
                    mbar_wait(smem_u32(full + s), (it / kStages) & 1);
                    mbar_arrive_remote_relaxed(leader_bar + (uint32_t)s * 8u);
                }
            }
        }
    } else if (warp < 2 + kNormWarps) {
        // ===== norm warps: threads 0..127 one row of this CTA's A half, threads 128..128+TNH-1 one of its B columns =====
        const int t = threadIdx.x - 64;
        const bool has_a = t < 128, has_b = t >= 128 && t < 128 + TNH;
        const int ta = has_a ? t : 0, tb = has_b ? t - 128 : 0;
        uint32_t base[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) base[r] = staged_offset(has_a ? ta : tb, r);
        uint32_t it = 0;
        int ti = 0;
        for (int tile = pair; tile < a.n_tiles; tile += npairs, ++ti) {
            const int frame = tile / tiles_per_frame, r0 = tile - frame * tiles_per_frame;
            const int m_tile = r0 / a.tiles_n, n_tile = r0 - m_tile * a.tiles_n;
            const int b = frame / a.F, f = frame - b * a.F;
            const float vis = has_a ? corr_vis(a.vt ? a.vt + (int64_t)b * a.vt_sb : nullptr, m_tile * kTile + (int)rank * 128 + ta, a)
                                    : corr_vis(a.vr ? a.vr + (int64_t)b * a.vr_sb + (int64_t)f * a.vr_sf : nullptr,
                                               n_tile * TN + (int)rank * TNH + tb, a);
            float q[4] = {0.f, 0.f, 0.f, 0.f};
            for (int kb = 0; kb < num_k; ++kb, ++it) {
                const int s = it % kStages;
                const uint32_t ph = (it / kStages) & 1;
                mbar_wait(smem_u32(full + s), ph);
                const uint8_t *ps = has_a ? smem_a + s * kStageBytesA : smem_b + s * kStageBytesB;
                if (has_a || has_b) {
#pragma unroll
                    for (int r = 0; r < 4; ++r) {
#pragma unroll
                        for (int j = 0; j < kBK / 4; ++j) {
                            const float v = *reinterpret_cast<const float *>(ps + base[r] + j * 512);
                            q[r] = __fmaf_rn(v, v, q[r]);
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(smem_u32(empty + s));
            }
            const float ss = (q[0] + q[1]) + (q[2] + q[3]);
            const int buf = ti % kBufs;
            const uint32_t use = (uint32_t)(ti / kBufs);
            // the scale tables of this buffer (here and in the peer) are free once both epilogues are done with them
            mbar_wait_cluster(smem_u32(tmem_empty + buf), (use & 1) ^ 1);
            const float sc = __fdiv_rn(vis, __fadd_rn(__fmul_rn(fabsf(vis), sqrtf(ss)), 1e-9f));
            if (has_a) s_sa[buf * 128 + ta] = sc;
            if (has_b) {
                float *dst = s_sb + buf * kTile + (int)rank * TNH + tb;
                *dst = sc;
                st_remote_f32(mapa_u32(smem_u32(dst), other), sc);
            }
            asm volatile("fence.acq_rel.cluster;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(smem_u32(scales_ready + buf));
                if (t >= 128) mbar_arrive_remote(mapa_u32(smem_u32(scales_ready + buf), other));
            }
        }
    } else {
        // ===== epilogue warps: this CTA's 128 rows x TN columns =====
        const int lq = warp & 3, ew = warp - (2 + kNormWarps);
        float *st = epi + ew * 32 * kEpiPitch;
        float l1_acc = 0.0f;
        int ti = 0;
        for (int tile = pair; tile < a.n_tiles; tile += npairs, ++ti) {
            const int frame = tile / tiles_per_frame, r0 = tile - frame * tiles_per_frame;
            const int m_tile = r0 / a.tiles_n, n_tile = r0 - m_tile * a.tiles_n;
            const int buf = ti % kBufs;
            const uint32_t use = (uint32_t)(ti / kBufs);
            const int row0 = lq * 32;
            const int64_t off0 = ((int64_t)frame * a.P + m_tile * kTile + (int)rank * 128 + row0) * a.P + n_tile * TN;
            if (a.pred) corr_epi_prefetch<TN>(a, off0, lane);
            mbar_wait_cluster(smem_u32(scales_ready + buf), use & 1);
            mbar_wait(smem_u32(tmem_full + buf), use & 1);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const float *sbv = s_sb + buf * kTile;
            const float sa = s_sa[buf * 128 + row0 + lane];
            const uint32_t taddr = tmem_base + ((uint32_t)(lq * 32) << 16) + (uint32_t)(buf * TN);
            if (a.pred) corr_epi_block<TN, true>(a, taddr, sa, sbv, st, off0, lane, l1_acc);
            else corr_epi_block<TN, false>(a, taddr, sa, sbv, st, off0, lane, l1_acc);
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            __syncwarp();
            if (lane == 0) {
                mbar_arrive(smem_u32(tmem_empty + buf));
                mbar_arrive_remote(mapa_u32(smem_u32(tmem_empty + buf), other));
            }
        }
        if (a.pred) corr_l1_tail(a, l1_acc, blockIdx.x * kEpiWarps + ew, gridDim.x * kEpiWarps, lane);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    cluster_sync_all();  // no CTA leaves (or frees TMEM) while its peer may still signal it
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
    }
}

// backward of mean |pred - corr| w.r.t. pred: sign * grad / count.  Thread = 4 consecutive elements (one 4-byte load,
// one coalesced 16-byte store), 4 such groups a block stride apart per thread for loads in flight.
// T: element type of pred and g_pred; a half gradient is the fp32 one rounded to nearest even (one 8-byte store)
template <typename T = float>
__global__ void __launch_bounds__(256) corr_l1_bwd_kernel(const signed char *__restrict__ sign,
                                                          const float *__restrict__ grad_loss, float inv_count,
                                                          void *__restrict__ g_pred, int64_t n4) {
    pdl_sync();
    const float g = __fmul_rn(__ldg(grad_loss), inv_count);
    const int64_t i0 = (int64_t)blockIdx.x * (4 * 256) + threadIdx.x;
    int w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int64_t i = i0 + k * 256;
        w[k] = i < n4 ? __ldcs(reinterpret_cast<const int *>(sign) + i) : 0;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int64_t i = i0 + k * 256;
        if (i >= n4) break;
        float4 r;
        r.x = (float)(signed char)(w[k] & 0xff) * g;
        r.y = (float)(signed char)((w[k] >> 8) & 0xff) * g;
        r.z = (float)(signed char)((w[k] >> 16) & 0xff) * g;
        r.w = (float)(signed char)((w[k] >> 24) & 0xff) * g;
        if constexpr (sizeof(T) == 4) {
            __stcs(reinterpret_cast<float4 *>(static_cast<T *>(g_pred)) + i, r);
        } else {
            uint2 u;
            T *e = reinterpret_cast<T *>(&u);
            e[0] = narrow<T>(r.x); e[1] = narrow<T>(r.y); e[2] = narrow<T>(r.z); e[3] = narrow<T>(r.w);
            __stcs(reinterpret_cast<uint2 *>(static_cast<T *>(g_pred)) + i, u);
        }
    }
}

}  // namespace

// ticket (16 bytes, zero between launches) + one partial per (CTA, epilogue warp) of up to 2 x 148 CTAs, with slack
int64_t corr4d_l1_workspace_bytes() { return 16 + 2 * 148 * kEpiWarps * 4 * 2; }

int corr4d_l1_bwd_launch(const signed char *sign, const float *grad_loss, void *g_pred, int64_t n, cudaStream_t st,
                         int dtype) {
    return with_dtype(dtype, "mt_corr4d_l1_bwd_dt", [&](auto t) {
        using T = decltype(t);
        MT_REQUIRE(n > 0 && n % 4 == 0 && aligned16(sign) && aligned_vec4<T>(g_pred),
                   "mt_corr4d_l1_bwd: n must be a multiple of 4, sign 16 B and g_pred %d B aligned", 4 * (int)sizeof(T));
        const int64_t n4 = n / 4;
        launch(corr_l1_bwd_kernel<T>, dim3((unsigned)((n4 + 1023) / 1024)), dim3(256), 0, st, sign, grad_loss,
               (float)(1.0 / (double)n), g_pred, n4);
        return launch_status("mt_corr4d_l1_bwd");
    });
}

int corr4d_tc_supported(int C, int P) {
    if (tuning("MT_CORR_SIMT", 0)) return 0;
    return (P % kTile == 0 && C % kBK == 0 && C >= kBK && P <= 65536) ? 1 : 0;
}

int64_t corr4d_tc_workspace_bytes(int B, int C, int F, int P) {
    (void)B; (void)C; (void)F; (void)P;
    return 0;  // norms are fused into the GEMM: no scratch
}

// The single-CTA launch of corr_tc_kernel<T> for the tile shape tm x tn
template <typename T>
static int corr_tc_single_go(const CUtensorMap &map_a, const CUtensorMap &map_b, const CorrTcArgs &a, int tm, int tn,
                             cudaStream_t st) {
    int ctas = sm_count();
    if (ctas > a.n_tiles) ctas = a.n_tiles;
    dim3 grid(ctas);
#define MT_CORR_GO(TMV, TNV, STG)                                                                    \
    do {                                                                                             \
        static_assert(smem_bytes_p<TMV, TNV, STG>() <= 227 * 1024, "stage ring exceeds the shared memory of an SM"); \
        cudaError_t e = cudaFuncSetAttribute(corr_tc_kernel<T, TMV, TNV, STG>,                       \
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes_p<TMV, TNV, STG>()); \
        if (e != cudaSuccess) {                                                                      \
            set_error("mt_corr4d_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));             \
            return MT_ERR_CUDA;                                                                      \
        }                                                                                            \
        launch(corr_tc_kernel<T, TMV, TNV, STG>, grid, dim3(kThreadsP), (size_t)smem_bytes_p<TMV, TNV, STG>(), st, map_a, map_b, a); \
    } while (0)
    if (tm == 256) {
        if (tn == 256) MT_CORR_GO(256, 256, 3);       // 3 x 64 KB
        else if (tn == 128) MT_CORR_GO(256, 128, 4);  // 4 x 48 KB
        else MT_CORR_GO(256, 64, 5);                  // 5 x 40 KB
    } else {
        if (tn == 256) MT_CORR_GO(128, 256, 4);       // 4 x 48 KB
        else if (tn == 128) MT_CORR_GO(128, 128, 6);  // 6 x 32 KB
        else MT_CORR_GO(128, 64, 8);                  // 8 x 24 KB
    }
#undef MT_CORR_GO
    return launch_status("mt_corr4d_fwd");
}

// tensor-map parameters of the operand traits CorrOp<T>
struct CorrMapSpec {
    CUtensorMapDataType type;
    CUtensorMapSwizzle swizzle;
    int esize, group_px, bk;
};
template <typename T>
static CorrMapSpec corr_map_spec() {
    return {CorrOp<T>::kTmaType, CorrOp<T>::kTmaSwizzle, (int)sizeof(T), CorrOp<T>::kGroupPx, CorrOp<T>::kBK};
}

// Strided form.  ft (B, C, P): strides ft_sb, ft_sc; fr (B, C, F, P): fr_sb, fr_sc, fr_sf (elements; the pixel index
// is contiguous).  Masks: see CorrTcArgs.  dtype (MT_DT_*): element type of ft / fr and of the volume `out` (or of
// `pred` in L1 mode); fp16 / bf16 features run the single-CTA kind::f16 kernel (no CTA pairs).
int corr4d_tc_launch_ex(const void *ft, int64_t ft_sb, int64_t ft_sc, const void *fr, int64_t fr_sb, int64_t fr_sc,
                        int64_t fr_sf, const float *vt, int64_t vt_sb, const float *vr, int64_t vr_sb, int64_t vr_sf,
                        int mask_mode, int MH, int MW, int fh, int fw, void *out, int B, int C, int F, int P,
                        cudaStream_t st, const CorrL1 *l1, int dtype) {
    CorrMapSpec ms{};
    const int drc = with_dtype(dtype, "mt_corr4d_fwd", [&](auto t) {
        ms = corr_map_spec<decltype(t)>();
        return MT_OK;
    });
    if (drc) return drc;
    const bool half = dtype != MT_DT_F32;
    MT_REQUIRE(C % ms.bk == 0, "mt_corr4d_fwd: C = %d is not a multiple of %d channels", C, ms.bk);
    MT_REQUIRE(aligned16(ft) && aligned16(fr) && (l1 || aligned16(out)), "mt_corr4d_fwd: pointers must be 16 B aligned");
    MT_REQUIRE(!l1 || (l1->pred && l1->loss && l1->partials && aligned16(l1->pred) && aligned16(l1->sign)),
               "mt_corr4d_vgg_l1_fwd: pred, loss and workspace are required, pred / sign 16 B aligned");
    const int64_t smask = 16 / ms.esize - 1;  // tensor-map strides are multiples of 16 B
    MT_REQUIRE(!((ft_sb | ft_sc | fr_sb | fr_sc | fr_sf) & smask) && ft_sc > 0 && fr_sc > 0 && (B == 1 || (ft_sb > 0 && fr_sb > 0)) &&
               (F == 1 || fr_sf > 0) && ft_sb >= 0 && fr_sb >= 0 && fr_sf >= 0,
               "mt_corr4d_fwd: feature strides must be positive multiples of 16 B (%d elements)", (int)smask + 1);
    EncodeTiledFn enc = encode_fn();
    if (!enc) {
        set_error("mt_corr4d_fwd: cuTensorMapEncodeTiled is not available from the driver");
        return MT_ERR_NO_DEVICE;
    }
    // Tile shape TM x TN.  256 x 256 = a whole frame per CTA: every operand byte loaded once, but one tile per (b, f)
    // frame; smaller tiles split a frame over 2 / 4 / 8 CTAs (operands re-read from L2) so that a small batch still
    // fills the 148 SMs, and leave room for two TMEM accumulator buffers (epilogue under the next main loop).
    // Swept on B200 (profiles/r2_experiments.md).  MT_CORR_TM / MT_CORR_TN override.
    const int frames = B * F * (P / kTile);
    int tm = tuning("MT_CORR_TM", 0), tn = tuning("MT_CORR_TN", 0);
    const bool tn_given = tn == 256 || tn == 128 || tn == 64, tm_given = tm == 256 || tm == 128;
    if (!tn_given || !tm_given) {
        const int sms = sm_count();
        int atm, atn;
        // whole frames per CTA once the batch fills the machine; below that, split a frame into as many tiles as it takes
        // to put a tile on ~85 % of the SMs.  Re-swept after the kernel stopped pre-launching its dependents
        // (profiles/r2_experiments.md, calls AH / AI): 32 frames 256 x 128 -> 128 x 128: 21.3 -> 17.3 us (default step
        // 98.4 -> 94.4 us); 16 frames 128 x 128 -> 128 x 64: 17.0 -> 15.9 us (step 26.7 -> 24.8 us)
        const int need = (sms * 85 + frames * 100 - 1) / (frames * 100);  // tiles per frame wanted
        if (frames * 2 >= sms) { atm = 256; atn = 256; }
        else if (need <= 2) { atm = 256; atn = 128; }
        else if (need <= 4) { atm = 128; atn = 128; }
        else { atm = 128; atn = 64; }
        if (!tm_given) tm = tn_given ? 256 : atm;
        if (!tn_given) tn = atn;
    }
    if (P % tn) tn = 64;
    // CTA pairs (cta_group::2): whole-frame tiles on two SMs.  MT_CORR_2CTA = 1 forces, 0 disables; default: when the
    // batch fills the pairs (see profiles/r2_experiments.md).  fp32 features only: half features always take the
    // single-CTA kernel
    // ncu (profiles/r2_experiments.md): 128 frames 29.8 vs 28.5 us, 256 frames 49.3 vs 51.4 us, 512 frames 84.4 vs 98.6 us
    // (pairs vs single CTAs); graph-replayed cfg3 step at 256 / 512 frames: +1.2 % / -1.2 %.  The pairs win once every
    // pair has ~5 whole-frame tiles; at 512 frames they run at 85 % of the HBM roofline (5.6 TB/s), where the op -
    // bandwidth-bound from cold DRAM at 73 flop/B - cannot go much faster
    int pair = tuning("MT_CORR_2CTA", -1);
    if (pair < 0) pair = kPairDefault && !tm_given && !tn_given && frames * 2 >= sm_count() * 5 ? 1 : 0;
    if (half) pair = 0;
    if (pair && !tn_given) tn = 256;
    if (pair && tn == 64) tn = 128;
    CUtensorMap map_a, map_b;
    {
        // ft (B, C, P) viewed as (G, C, P/G, B), G = pixels per 128 B (32 fp32, 64 half): strides in bytes for dims 1..3
        const int G = ms.group_px, es = ms.esize;
        cuuint64_t dims[4] = {(cuuint64_t)G, (cuuint64_t)C, (cuuint64_t)(P / G), (cuuint64_t)B};
        cuuint64_t strides[3] = {(cuuint64_t)ft_sc * es, 128, (cuuint64_t)(B > 1 ? ft_sb : (int64_t)C * P) * es};
        cuuint32_t box[4] = {(cuuint32_t)G, (cuuint32_t)ms.bk, (cuuint32_t)((pair ? 128 : tm) / G), 1};
        cuuint32_t estr[4] = {1, 1, 1, 1};
        CUresult r = enc(&map_a, ms.type, 4, const_cast<void *>(ft), dims, strides, box,
                         estr, CU_TENSOR_MAP_INTERLEAVE_NONE, ms.swizzle,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("mt_corr4d_fwd: cuTensorMapEncodeTiled(A) failed with %d", (int)r);
            return MT_ERR_CUDA;
        }
    }
    {
        // fr (B, C, F, P) viewed as (G, C, P/G, F, B)
        const int G = ms.group_px, es = ms.esize;
        cuuint64_t dims[5] = {(cuuint64_t)G, (cuuint64_t)C, (cuuint64_t)(P / G), (cuuint64_t)F, (cuuint64_t)B};
        cuuint64_t strides[4] = {(cuuint64_t)fr_sc * es, 128, (cuuint64_t)(F > 1 ? fr_sf : (int64_t)P) * es,
                                 (cuuint64_t)(B > 1 ? fr_sb : (int64_t)C * F * P) * es};
        cuuint32_t box[5] = {(cuuint32_t)G, (cuuint32_t)ms.bk, (cuuint32_t)((pair ? tn / 2 : tn) / G), 1, 1};
        cuuint32_t estr[5] = {1, 1, 1, 1, 1};
        CUresult r = enc(&map_b, ms.type, 5, const_cast<void *>(fr), dims, strides, box,
                         estr, CU_TENSOR_MAP_INTERLEAVE_NONE, ms.swizzle,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            set_error("mt_corr4d_fwd: cuTensorMapEncodeTiled(B) failed with %d", (int)r);
            return MT_ERR_CUDA;
        }
    }
    CorrTcArgs a;
    a.vt = vt; a.vt_sb = vt_sb; a.vr = vr; a.vr_sb = vr_sb; a.vr_sf = vr_sf;
    a.mask_mode = mask_mode; a.MH = MH; a.MW = MW; a.fw = fw > 0 ? fw : 1;
    a.msy = mask_mode ? (float)MH / (float)fh : 1.0f;
    a.msx = mask_mode ? (float)MW / (float)fw : 1.0f;
    a.out = out; a.C = C; a.F = F; a.P = P;
    a.pred = l1 ? l1->pred : nullptr; a.sign = l1 ? l1->sign : nullptr; a.loss = l1 ? l1->loss : nullptr;
    a.ticket = l1 ? reinterpret_cast<unsigned int *>(l1->partials) : nullptr;   // workspace: ticket header, then partials
    a.partials = l1 ? l1->partials + 4 : nullptr;
    a.inv_count = 1.0 / ((double)B * F * P * P);
    a.tiles_m = P / (pair ? kTile : tm); a.tiles_n = P / tn;
    const int64_t n_tiles = (int64_t)B * F * a.tiles_m * a.tiles_n;
    MT_REQUIRE(n_tiles < (1ll << 30), "mt_corr4d_fwd: too many tiles");
    a.n_tiles = (int)n_tiles;
    if (pair) {
        int npairs = sm_count() / 2;
        if (npairs > a.n_tiles) npairs = a.n_tiles;
        // cluster of two CTAs (compile-time __cluster_dims__) + programmatic dependent launch
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * npairs);
        cfg.blockDim = dim3(kThreadsP);
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = pdl_enabled() ? 1 : 0;
#define MT_CORR_PAIR_GO(TNV, STG)                                                                    \
    do {                                                                                             \
        static_assert(smem_bytes_pair<TNV, STG>() <= 227 * 1024, "stage ring exceeds the shared memory of an SM"); \
        cudaError_t e = cudaFuncSetAttribute(corr_tc2_kernel<TNV, STG>,                              \
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes_pair<TNV, STG>()); \
        if (e != cudaSuccess) {                                                                      \
            set_error("mt_corr4d_fwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));             \
            return MT_ERR_CUDA;                                                                      \
        }                                                                                            \
        cfg.dynamicSmemBytes = (size_t)smem_bytes_pair<TNV, STG>();                                  \
        (void)cudaLaunchKernelEx(&cfg, corr_tc2_kernel<TNV, STG>, map_a, map_b, a);                  \
    } while (0)
        if (tn == 256) MT_CORR_PAIR_GO(256, 6);  // 6 x 32 KB per CTA
        else MT_CORR_PAIR_GO(128, 8);            // 8 x 24 KB per CTA
#undef MT_CORR_PAIR_GO
        return launch_status("mt_corr4d_fwd");
    }
    if (dtype == MT_DT_F16) return corr_tc_single_go<__half>(map_a, map_b, a, tm, tn, st);
    if (dtype == MT_DT_BF16) return corr_tc_single_go<__nv_bfloat16>(map_a, map_b, a, tm, tn, st);
    return corr_tc_single_go<float>(map_a, map_b, a, tm, tn, st);
}

int corr4d_tc_launch(const float *ft, const float *vt, const float *fr, const float *vr, float *out, void *ws,
                     int64_t ws_bytes, int B, int C, int F, int P, cudaStream_t st) {
    (void)ws; (void)ws_bytes;
    return corr4d_tc_launch_ex(ft, (int64_t)C * P, P, fr, (int64_t)C * F * P, (int64_t)F * P, P, vt, P, vr,
                               (int64_t)F * P, P, 0, 0, 0, 0, 0, out, B, C, F, P, st, nullptr, MT_DT_F32);
}

}  // namespace mt
