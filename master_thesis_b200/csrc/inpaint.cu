// inpaint.cu - composite + hole update of L independent target frames of a clip ("lanes") in one launch.
//
// Replaces (reference file:line), for the batched inference loops of plug.chn_inpaint_ff / chn_inpaint_cp:
//   CHN.forward composite            master_thesis/model_chn.py:83-84
//   hole update in CHN.inpaint_ff    master_thesis/model_chn.py:128-131
//   hole update + finalisation in CHN.inpaint_cp   master_thesis/model_chn.py:242-248
//
// chn_fill_kernel (chn.cu) computes ONE hole percentage over its whole batch, the reference's sum(m) * 100 / numel at
// B = 1.  Here lane i is the F = 1 step of one target frame; it owns state slot slots[i] and gets its own percentage,
// folded in a fixed order (a ticket per lane, the last CTA of the lane sums the lane's CTA partials in double), so
// one launch serves L loop conditions without atomics on floats and without a host sync.  The per-element arithmetic
// is chn_fill_kernel's, in the same operation order: y_comp, m_new, x_new and the percentage of every lane are
// bit-identical to mt_chn_fill_step at B = 1 on that lane (for {0,1} masks the float partials are exact integers, so
// the fold order cannot change the sum).
//
// In place: x_t / m_t may alias x_state[slot] / m_state[slot].  Every thread requests all operands of its pixels
// before its first store and no other thread touches those pixels.
#include "mt_common.cuh"

namespace mt {
namespace {

bool mult4(int64_t v) { return (v & 3) == 0; }

struct LanesArgs {
    const void *nn_out;                     // (L,3,P) contiguous, element type T of chn_fill_lanes_kernel
    const float *x_t; int64_t xt_sl, xt_sc;
    const float *m_t; int64_t mt_sl;
    const float *v_map0; int64_t vm_sl;
    const int *slots;                       // (L) state slot of each lane, unique
    float *y_out; int64_t yo_ss, yo_sc;     // written through the slot table
    float *m_state; int64_t ms_ss;
    float *x_state; int64_t xs_ss, xs_sc;
    float *per_out;                         // per_out[slot]
    void *ws;
    int64_t P; int chunks; int force; double e;
};

// Workspace: one ticket word per lane at a FIXED offset, sized for the largest lane count a launch accepts (grid.y),
// then the per-lane CTA partials.  The tickets do not move with L: a buffer zeroed once serves calls of any lane count
// in any order (every call re-arms the tickets of the lanes it used; the partials need no zeroing).
constexpr int kMaxLanes = 65535;
constexpr int64_t kLaneTicketBytes = (int64_t(kMaxLanes) * 4 + kWsTicketBytes - 1) / kWsTicketBytes * kWsTicketBytes;

int lane_block_cap(int L) {
    int n = sm_count() * 8 / L;
    if (n > kMaxReduceBlocks) n = kMaxReduceBlocks;
    return n < 1 ? 1 : n;
}

template <typename T, int VEC>
__global__ void __launch_bounds__(256) chn_fill_lanes_kernel(const LanesArgs a) {
    pdl_sync();
    const T *nn_out = static_cast<const T *>(a.nn_out);
    __shared__ float red[32];
    __shared__ bool is_last;
    const int lane = blockIdx.y;
    const int64_t slot = a.slots[lane];
    float acc[1] = {0.0f};
    for (int ch = blockIdx.x; ch < a.chunks; ch += gridDim.x) {
        const int64_t p0 = ((int64_t)ch * blockDim.x + threadIdx.x) * VEC;
        if (p0 >= a.P) continue;
        Vec<VEC> m, vm, vt, o[3], xt[3];
        m.load_stream(a.m_t + lane * a.mt_sl + p0);
        vm.load_stream(a.v_map0 + lane * a.vm_sl + p0);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            o[c].load_stream(nn_out + ((int64_t)lane * 3 + c) * a.P + p0);
            xt[c].load_stream(a.x_t + lane * a.xt_sl + c * a.xt_sc + p0);
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            vt.v[i] = __fsub_rn(1.0f, m.v[i]);    // v_t = 1 - m_t, as the loops pass it
            m.v[i] = __fsub_rn(m.v[i], vm.v[i]);  // m_t - v_map[:, :, 0]       :128
            acc[0] += m.v[i];
        }
        if (a.force) {  // model_chn.py:246-248 forced by the pass: m = 0, x = y_comp
            Vec<VEC> z;
#pragma unroll
            for (int i = 0; i < VEC; ++i) z.v[i] = 0.0f;
            z.store_stream(a.m_state + slot * a.ms_ss + p0);
        } else {
            m.store_stream(a.m_state + slot * a.ms_ss + p0);
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const float mean = chan_mean(c), s = chan_std(c);  // fill colour == mean, model_chn.py:102-104
            Vec<VEC> yc, xn;
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                const float yh = clamp01(__fadd_rn(__fmul_rn(o[c].v[i], s), mean));            // :83
                yc.v[i] = __fadd_rn(__fmul_rn(vt.v[i], xt[c].v[i]),                             // :84
                                    __fmul_rn(__fsub_rn(1.0f, vt.v[i]), yh));
                xn.v[i] = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, m.v[i]), yc.v[i]), __fmul_rn(m.v[i], mean));  // :129-130
            }
            yc.store_stream(a.y_out + slot * a.yo_ss + c * a.yo_sc + p0);
            (a.force ? yc : xn).store_stream(a.x_state + slot * a.xs_ss + c * a.xs_sc + p0);
        }
    }
    // per-lane fold: CTA partial -> workspace, the last CTA of the lane sums the lane's partials in a fixed order
    block_sum<1>(acc, red);
    unsigned int *ticket = reinterpret_cast<unsigned int *>(a.ws) + lane;
    float *partials = reinterpret_cast<float *>(reinterpret_cast<char *>(a.ws) + kLaneTicketBytes) +
                      (int64_t)lane * gridDim.x;
    if (threadIdx.x == 0) {
        partials[blockIdx.x] = acc[0];
        __threadfence();
        is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    double sum = 0.0;
    for (unsigned int i = threadIdx.x; i < gridDim.x; i += blockDim.x) sum += (double)__ldcg(partials + i);
    __shared__ double dsm[32];
    const int wl = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    sum = warp_sum(sum);
    if (wl == 0) dsm[wid] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        double tot = 0.0;
        for (int w = 0; w < nw; ++w) tot += dsm[w];
        a.per_out[slot] = (float)tot * 100.0f / (float)a.P;  // sum(m)*100/numel of the lane   :131
        *ticket = 0u;
    }
}

// model_chn.py:246-248 (`if float(per) < e: m = 0, y = y_comp`), decided on the device from the lane's completed
// reduction: runs after chn_fill_lanes_kernel (PDL wait) and rewrites only the lanes whose percentage is below e.
template <int VEC>
__global__ void __launch_bounds__(256) chn_finalize_lanes_kernel(const LanesArgs a) {
    pdl_sync();
    const int64_t slot = a.slots[blockIdx.y];
    if (!((double)a.per_out[slot] < a.e)) return;  // the float32 percentage widened, as `float(per) < e` compares
    for (int ch = blockIdx.x; ch < a.chunks; ch += gridDim.x) {
        const int64_t p0 = ((int64_t)ch * blockDim.x + threadIdx.x) * VEC;
        if (p0 >= a.P) continue;
        Vec<VEC> y[3], z;
#pragma unroll
        for (int c = 0; c < 3; ++c) y[c].load_stream(a.y_out + slot * a.yo_ss + c * a.yo_sc + p0);
#pragma unroll
        for (int i = 0; i < VEC; ++i) z.v[i] = 0.0f;
        z.store_stream(a.m_state + slot * a.ms_ss + p0);
#pragma unroll
        for (int c = 0; c < 3; ++c) y[c].store_stream(a.x_state + slot * a.xs_ss + c * a.xs_sc + p0);
    }
}

}  // namespace
}  // namespace mt

using namespace mt;

extern "C" int64_t mt_chn_fill_lanes_workspace_bytes(int L) {
    if (L < 1 || L > kMaxLanes) return 0;
    return kLaneTicketBytes + (int64_t)L * lane_block_cap(L) * 4;
}

extern "C" int mt_chn_fill_lanes_dt(int nn_dtype, const void *nn_out, const float *x_t, int64_t xt_sl,
                                    int64_t xt_sc, const float *m_t, int64_t mt_sl, const float *v_map0,
                                    int64_t vm_sl, const int *slots, float *y_out, int64_t yo_ss, int64_t yo_sc,
                                    float *m_state, int64_t ms_ss, float *x_state, int64_t xs_ss, int64_t xs_sc,
                                    float *per_out, void *workspace, int L, int64_t P, int finalize, double e,
                                    int force, mt_stream_t stream) {
    MT_REQUIRE(nn_out && x_t && m_t && v_map0 && slots && y_out && m_state && x_state && per_out && workspace,
               "mt_chn_fill_lanes: NULL argument");
    MT_REQUIRE(L >= 1 && L <= kMaxLanes && P > 0, "mt_chn_fill_lanes: bad shape (L = %d, P = %lld)", L, (long long)P);
    MT_REQUIRE(y_out != nn_out && m_state != nn_out && x_state != nn_out && per_out != nn_out,
               "mt_chn_fill_lanes: an output aliases nn_out");
    return with_dtype(nn_dtype, "mt_chn_fill_lanes", [&](auto tag) {
        using T = decltype(tag);
        LanesArgs a{nn_out, x_t, xt_sl, xt_sc, m_t, mt_sl, v_map0, vm_sl, slots, y_out, yo_ss, yo_sc,
                    m_state, ms_ss, x_state, xs_ss, xs_sc, per_out, workspace, P, 0, force ? 1 : 0, e};
        const bool v4 = mult4(P) && aligned_vec4<T>(nn_out) && aligned16(x_t) && aligned16(m_t) &&
                        aligned16(v_map0) && aligned16(y_out) && aligned16(m_state) && aligned16(x_state) &&
                        mult4(xt_sl) && mult4(xt_sc) && mult4(mt_sl) && mult4(vm_sl) && mult4(yo_ss) &&
                        mult4(yo_sc) && mult4(ms_ss) && mult4(xs_ss) && mult4(xs_sc);
        const int vec = v4 ? 4 : 1;
        const int64_t chunks = (P + 256 * vec - 1) / (256 * vec);
        MT_REQUIRE(chunks < (1ll << 31), "mt_chn_fill_lanes: plane too large");
        a.chunks = (int)chunks;
        const int cap = lane_block_cap(L);
        const dim3 grid((unsigned)(chunks < cap ? chunks : cap), (unsigned)L);
        const cudaStream_t st = (cudaStream_t)stream;
        if (v4) launch(chn_fill_lanes_kernel<T, 4>, grid, 256, 0, st, a);
        else launch(chn_fill_lanes_kernel<T, 1>, grid, 256, 0, st, a);
        int rc = launch_status("mt_chn_fill_lanes");
        if (rc || !finalize || force) return rc;
        if (v4) launch(chn_finalize_lanes_kernel<4>, grid, 256, 0, st, a);
        else launch(chn_finalize_lanes_kernel<1>, grid, 256, 0, st, a);
        return launch_status("mt_chn_fill_lanes (finalize)");
    });
}

extern "C" int mt_chn_fill_lanes(const float *nn_out, const float *x_t, int64_t xt_sl, int64_t xt_sc,
                                 const float *m_t, int64_t mt_sl, const float *v_map0, int64_t vm_sl,
                                 const int *slots, float *y_out, int64_t yo_ss, int64_t yo_sc, float *m_state,
                                 int64_t ms_ss, float *x_state, int64_t xs_ss, int64_t xs_sc, float *per_out,
                                 void *workspace, int L, int64_t P, int finalize, double e, int force,
                                 mt_stream_t stream) {
    return mt_chn_fill_lanes_dt(MT_DT_F32, nn_out, x_t, xt_sl, xt_sc, m_t, mt_sl, v_map0, vm_sl, slots, y_out, yo_ss,
                                yo_sc, m_state, ms_ss, x_state, xs_ss, xs_sc, per_out, workspace, L, P, finalize, e,
                                force, stream);
}
