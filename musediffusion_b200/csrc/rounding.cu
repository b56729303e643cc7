// Nearest-word-embedding rounding (get_efficient_knn, MuseDiffusion/models/rounding.py:21-28) and the final
// lm_head logits + argmax (models/network.py:91-93, run/sample.py:219-220), each fused with its row reduction so the
// [V, M] distance / [M, V] logit matrix never reaches HBM.  fp32 arithmetic (the reference's), register-blocked
// 8 tokens x 4 vocabulary rows per thread, operands staged in padded shared memory, any D that is a multiple of 4.
#include "common.cuh"
#include "musediff_b200.h"

namespace md {
int num_sms();

constexpr int RD = 128;          // embedding columns staged per pass (wider rows are contracted in RD-column slices)
constexpr int RT = 128;          // tokens per block
constexpr int RV = 64;           // vocabulary rows per chunk
constexpr int RLD = RD + 4;      // padded row stride (floats): shifts consecutive rows by 4 banks
constexpr int kRoundThreads = 256;
constexpr int kRoundSmem = (RT * RLD + RV * RLD + RV + RT) * 4;

struct Best {
    float b, s;   // best and second-best key
    int i;        // index of best
};
MD_DEVINL void best_push(Best& r, float key, int idx) {
    if (key < r.b || (key == r.b && idx < r.i)) { r.s = r.b; r.b = key; r.i = idx; }
    else if (key < r.s) r.s = key;
}
MD_DEVINL void best_merge(Best& r, float ob, float os, int oi) {
    const float lose = fmaxf(r.b, ob);
    if (ob < r.b || (ob == r.b && oi < r.i)) { r.b = ob; r.i = oi; }
    r.s = fminf(fminf(r.s, os), lose);
}

// rows [row0, row0 + n_rows) x columns [d0, d0 + RD) of a [rows_total, D] fp32 matrix -> smem [n_rows][RLD]; zeros outside
MD_DEVINL void stage_slice(float* dst, const float* src, int64_t row0, int n_rows, int64_t rows_total, int D, int d0) {
    for (int i = threadIdx.x; i < n_rows * (RD / 4); i += kRoundThreads) {
        const int r = i >> 5, c = (i & 31) << 2;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (row0 + r < rows_total && d0 + c < D) v = *reinterpret_cast<const float4*>(src + (row0 + r) * D + d0 + c);
        *reinterpret_cast<float4*>(dst + r * RLD + c) = v;
    }
}

// MODE 0: key = clamp(|E_v|^2 + |x|^2 - 2 x.E_v, 0)   (argmin distance)
// MODE 1: key = -(x.E_v + bias_v)                      (argmax logit)
// Any D % 4 == 0: the contraction runs over RD-column slices (zero-filled past D, which adds exact zeros); every sum
// keeps the single-slice operation order within a slice and adds the slices in order (D <= 128: one slice).
template <int MODE>
__global__ void __launch_bounds__(kRoundThreads, 2)
round_kernel(const float* __restrict__ x, const float* __restrict__ E, const float* __restrict__ bias,
             int32_t* __restrict__ out_idx, float* __restrict__ out_margin, int64_t M, int V, int D) {
    extern __shared__ float rsm[];
    float* xs = rsm;                    // [RT][RLD]
    float* es = xs + RT * RLD;          // [RV][RLD]
    float* en = es + RV * RLD;          // [RV]  |E_v|^2 or bias
    float* xn = en + RV;                // [RT]  |x|^2
    const int tid = threadIdx.x;
    const int vg = tid & 15, tg = tid >> 4;
    const int64_t tok0 = (int64_t)blockIdx.x * RT;
    const int n_slices = (D + RD - 1) / RD;

    // ---- |x|^2 (2 threads per token row), slice by slice; the last slice stays staged
    float xsq = 0.f;
    for (int sl = 0; sl < n_slices; ++sl) {
        if (sl > 0) __syncthreads();
        stage_slice(xs, x, tok0, RT, M, D, sl * RD);
        __syncthreads();
        if (MODE == 0) {
            const int r = tid >> 1, h = tid & 1;
            float s = 0.f;
            for (int c = h * 64; c < h * 64 + 64; ++c) { const float v = xs[r * RLD + c]; s = fmaf(v, v, s); }
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            xsq += s;
        }
    }
    if (MODE == 0 && (tid & 1) == 0) xn[tid >> 1] = xsq;

    Best best[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { best[i].b = INFINITY; best[i].s = INFINITY; best[i].i = 0x7fffffff; }

    const int n_chunks = (V + RV - 1) / RV;
    for (int ch = 0; ch < n_chunks; ++ch) {
        const int v0 = ch * RV;
        float acc[8][4];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        float esq = 0.f;
        for (int sl = 0; sl < n_slices; ++sl) {
            const int d0 = sl * RD;
            __syncthreads();   // previous slice / chunk fully consumed (and xn visible on the first pass)
            if (n_slices > 1) stage_slice(xs, x, tok0, RT, M, D, d0);
            stage_slice(es, E, v0, RV, V, D, d0);
            __syncthreads();
            if (MODE == 0) {
                // 4 threads per vocabulary row: |E_v|^2
                const int r = tid >> 2, h = tid & 3;
                float s = 0.f;
                for (int c = h * 32; c < h * 32 + 32; ++c) { const float v = es[r * RLD + c]; s = fmaf(v, v, s); }
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                esq += s;
            }
            const int dlim = min(RD, D - d0);
#pragma unroll 4
            for (int d = 0; d < dlim; d += 4) {
                float4 ev[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) ev[j] = *reinterpret_cast<const float4*>(es + (vg + 16 * j) * RLD + d);
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float4 xv = *reinterpret_cast<const float4*>(xs + (tg * 8 + i) * RLD + d);
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        acc[i][j] = fmaf(xv.x, ev[j].x, acc[i][j]);
                        acc[i][j] = fmaf(xv.y, ev[j].y, acc[i][j]);
                        acc[i][j] = fmaf(xv.z, ev[j].z, acc[i][j]);
                        acc[i][j] = fmaf(xv.w, ev[j].w, acc[i][j]);
                    }
                }
            }
        }
        {
            const int r = tid >> 2, h = tid & 3;
            if (h == 0) en[r] = (MODE == 0) ? esq : ((v0 + r < V) ? bias[v0 + r] : 0.f);
        }
        __syncthreads();   // en[] written above is visible
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int v = v0 + vg + 16 * j;
            if (v < V) {
                const float e = en[vg + 16 * j];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    float key;
                    if (MODE == 0) key = fmaxf(__fsub_rn(__fadd_rn(e, xn[tg * 8 + i]), __fmul_rn(2.0f, acc[i][j])), 0.0f);
                    else key = -(acc[i][j] + e);
                    best_push(best[i], key, v);
                }
            }
        }
    }
    // ---- merge the 16 vocabulary-group threads of each token group (lanes differing in the low 4 bits)
#pragma unroll
    for (int i = 0; i < 8; ++i) {
#pragma unroll
        for (int o = 1; o < 16; o <<= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best[i].b, o);
            const float os = __shfl_xor_sync(0xffffffffu, best[i].s, o);
            const int oi = __shfl_xor_sync(0xffffffffu, best[i].i, o);
            best_merge(best[i], ob, os, oi);
        }
        const int64_t tok = tok0 + tg * 8 + i;
        if (vg == 0 && tok < M) {
            out_idx[tok] = best[i].i < V ? best[i].i : 0;      // MODE 1, every logit NaN: no key was taken, id 0
            if (out_margin != nullptr) out_margin[tok] = best[i].s - best[i].b;
        }
    }
}

template <int MODE>
static int launch_round(const float* x, const float* E, const float* bias, int32_t* idx, float* margin, int64_t M, int V, int D,
                        cudaStream_t stream) {
    auto kern = round_kernel<MODE>;
    static bool attr_set[kMaxDevices] = {false};
    if (ensure_dyn_smem(kern, kRoundSmem, attr_set, "cudaFuncSetAttribute(round)")) return MD_ERR_CUDA;
    const int64_t grid = (M + RT - 1) / RT;
    kern<<<(unsigned)grid, kRoundThreads, kRoundSmem, stream>>>(x, E, bias, idx, margin, M, V, D);
    return check_cuda(cudaGetLastError(), "round launch");
}

}  // namespace md

using namespace md;

extern "C" __attribute__((visibility("default"))) int md_round_argmin(const float* x, const float* E, int32_t* idx, float* margin, int64_t M, int V, int D,
                               cudaStream_t stream) {
    if (D <= 0 || D % 4 != 0) { set_last_error("md_round_argmin: D=%d must be a positive multiple of 4", D); return MD_ERR_ARG; }
    if (V <= 0) { set_last_error("md_round_argmin: empty vocabulary"); return MD_ERR_ARG; }
    if (M == 0) return MD_OK;
    return launch_round<0>(x, E, nullptr, idx, margin, M, V, D, stream);
}

extern "C" __attribute__((visibility("default"))) int md_logits_argmax(const float* x, const float* E, const float* bias, int32_t* tok, float* margin, int64_t M,
                                int V, int D, cudaStream_t stream) {
    if (D <= 0 || D % 4 != 0) { set_last_error("md_logits_argmax: D=%d must be a positive multiple of 4", D); return MD_ERR_ARG; }
    if (V <= 0 || bias == nullptr) { set_last_error("md_logits_argmax: bad arguments"); return MD_ERR_ARG; }
    if (M == 0) return MD_OK;
    return launch_round<1>(x, E, bias, tok, margin, M, V, D, stream);
}
