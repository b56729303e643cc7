// Nearest-word-embedding rounding and lm_head argmax on the tensor cores (sm_100a).
//
//   idx[m] = argmin_v ( |E_v|^2 - 2 x_m . E_v )      get_efficient_knn, MuseDiffusion/models/rounding.py:21-28
//   tok[m] = argmax_v ( x_m . E_v + b_v )            get_logits + argmax, models/network.py:91-93, run/sample.py:219-220
//
// The [V, M] distance / [M, V] logit matrix never reaches HBM: it lives in TMEM and is reduced per row in the
// epilogue.  fp32 fidelity on bf16 tensor cores comes from splitting both operands, x = xh + xl and E = Eh + El
// (bf16 each), and accumulating the four partial products in fp32:
//     x.E ~ xh.Eh + xh.El + xl.Eh + xl.El          (dropped split residuals <= 2^-15 sum_d |x_d E_d|; DESIGN.md 4.4)
// which is ONE K = 4D contraction whose k-blocks read [xh|xl] and [Eh|El] at remapped column offsets.
//
// Structure = the persistent tcgen05 GEMM of gemm.cu (TMA producer warp, MMA warp, 8 epilogue warps, two TMEM
// accumulators) with (1) a CTA that walks ALL n-tiles of one 128-row block before moving on, so the epilogue threads
// (thread = row) keep a running (best, second, index) across the vocabulary, (2) an argmin epilogue instead of a
// store.  |x_m|^2 is constant per row and cannot change the argmin; the reference's clamp(dist, 0) only matters for
// exact hits (x == E_v bit for bit), where it creates ties — see DESIGN.md section 2.
#include <math.h>

#include "common.cuh"
#include "musediff_b200.h"

namespace md {
int num_sms();
int make_tmap_2d(CUtensorMap* tm, const void* base, int is_f32, uint64_t rows, uint64_t cols, uint64_t row_stride_elems,
                 uint32_t box_rows, uint32_t box_cols);

constexpr int RT_BM = 128, RT_BN = 256, RT_BK = 64;
constexpr int RT_STAGES = 4;
constexpr int RT_A_BYTES = RT_BM * RT_BK * 2, RT_B_BYTES = RT_BN * RT_BK * 2;
constexpr int RT_STAGE_BYTES = RT_A_BYTES + RT_B_BYTES;
constexpr int RT_THREADS = 320;
constexpr int RT_SMEM = 1024 + RT_STAGES * RT_STAGE_BYTES + 2 * RT_BN * 4 /*per-column constants, double buffered*/ +
                        128 * 3 * 4 /*half merge*/ + 256;

struct RoundTcArgs {
    int64_t M;
    int V, Vp, D;          // Vp = V padded to a multiple of RT_BN (padding columns carry +inf constants)
    const float* cst;      // [Vp]  MODE 0: |E_v|^2   MODE 1: bias_v   (padding: +inf / -inf handled on the host)
    int32_t* idx;          // [M]
    float* margin;         // optional [M]
};

// fp32 [rows, D] -> bf16 [rows, copies * 2Dp] = copies x [hi | 0 | lo | 0] split (Dp >= D: half width, zero columns
// D..Dp-1 so that a contraction over Dp columns equals the one over D), one float4 per thread
__global__ void __launch_bounds__(256) split_bf16_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out, int64_t rows,
                                                         int D, int Dp, int copies) {
    const int vec = Dp >> 2;
    const int64_t total = rows * vec;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / vec;
        const int c = (int)(i - r * vec) << 2;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c < D)
            asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(x + r * D + c));
        const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
        const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
        const __nv_bfloat162 l0 = __floats2bfloat162_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2bfloat162_rn(v.z - f1.x, v.w - f1.y);
        for (int k = 0; k < copies; ++k) {
            __nv_bfloat16* o = out + (r * copies + k) * 2 * Dp + c;
            *reinterpret_cast<uint2*>(o) = make_uint2(*reinterpret_cast<const uint32_t*>(&h0), *reinterpret_cast<const uint32_t*>(&h1));
            *reinterpret_cast<uint2*>(o + Dp) = make_uint2(*reinterpret_cast<const uint32_t*>(&l0), *reinterpret_cast<const uint32_t*>(&l1));
        }
    }
}

// E fp32 [V, D] -> E2 bf16 [Vp, 2Dp] = [hi | 0 | lo | 0] (zero rows beyond V, zero columns D..Dp-1), |E_v|^2 over the D real
// columns (fp32, +inf beyond V) and, optionally, the rows
// clamped to [-1, 1] (what clip_denoised makes of a rounded x0, diffusion.py:323-324: the posterior kernel then gathers them
// ready-made instead of clamping 128 values per token and step)
__global__ void __launch_bounds__(128) embed_prepare_kernel(const float* __restrict__ E, __nv_bfloat16* __restrict__ E2,
                                                            float* __restrict__ sqnorm, float* __restrict__ E_clamped, int V, int Vp, int D,
                                                            int Dp) {
    const int v = blockIdx.x;
    float s = 0.f;
    for (int d = threadIdx.x; d < Dp; d += blockDim.x) {
        const bool real = v < V && d < D;
        const float e = real ? E[(size_t)v * D + d] : 0.f;
        const __nv_bfloat16 h = __float2bfloat16_rn(e);
        E2[(size_t)v * 2 * Dp + d] = h;
        E2[(size_t)v * 2 * Dp + Dp + d] = __float2bfloat16_rn(e - __bfloat162float(h));
        if (E_clamped != nullptr && real) E_clamped[(size_t)v * D + d] = fminf(fmaxf(e, -1.0f), 1.0f);
        if (d < D) s = fmaf(e, e, s);
    }
    __shared__ float red[4];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) sqnorm[v] = (v < V) ? (red[0] + red[1] + red[2] + red[3]) : INFINITY;
}

struct Best3 {
    float b, s;
    int i;
};
MD_DEVINL void best3_push(Best3& r, float key, int idx) {
    if (key < r.b) { r.s = r.b; r.b = key; r.i = idx; }      // columns arrive in increasing index order: '<' keeps the lowest index on ties
    else if (key < r.s) r.s = key;
}

template <int MODE>
__global__ void __launch_bounds__(RT_THREADS, 1)
round_tc_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const RoundTcArgs p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;
    uint8_t* sB = smem + RT_STAGES * RT_A_BYTES;
    float* sCst = reinterpret_cast<float*>(smem + RT_STAGES * RT_STAGE_BYTES);     // [2][RT_BN]
    float* sMerge = sCst + 2 * RT_BN;                                              // [128][3]: best, second, index of column half 1
    uint64_t* bars = reinterpret_cast<uint64_t*>(sMerge + 128 * 3);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + RT_STAGES;
    uint64_t* tfull_bar = bars + 2 * RT_STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n_tiles = p.Vp / RT_BN;
    const int m_tiles = (int)((p.M + RT_BM - 1) / RT_BM);
    const int kb_per_seg = p.D / RT_BK;          // k-blocks per operand half (2 for D = 128)
    const int num_kb = 4 * kb_per_seg;           // segments: (xh,Eh) (xh,El) (xl,Eh) (xl,El)

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        for (int s = 0; s < RT_STAGES; ++s) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tfull_bar[s], 1);
            mbar_init(&tempty_bar[s], 256);
        }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc<512>(tmem_slot);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        int stage = 0;
        uint32_t phase = 0;
        for (int m_blk = blockIdx.x; m_blk < m_tiles; m_blk += gridDim.x)
            for (int n_blk = 0; n_blk < n_tiles; ++n_blk)
                for (int kb = 0; kb < num_kb; ++kb) {
                    const int seg = kb / kb_per_seg, kk = kb - seg * kb_per_seg;
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_arrive_expect_tx_w(&full_bar[stage], RT_STAGE_BYTES);
                    tma_load_2d_w(sA + stage * RT_A_BYTES, &tmA, &full_bar[stage], (seg >> 1) * p.D + kk * RT_BK, m_blk * RT_BM);
                    tma_load_2d_w(sB + stage * RT_B_BYTES, &tmB, &full_bar[stage], (seg & 1) * p.D + kk * RT_BK, n_blk * RT_BN);
                    if (++stage == RT_STAGES) { stage = 0; phase ^= 1; }
                }
    } else if (warp == 1) {
        constexpr uint32_t idesc = make_idesc_bf16(RT_BM, RT_BN);
        int stage = 0, acc = 0;
        uint32_t phase = 0, acc_phase = 0;
        for (int m_blk = blockIdx.x; m_blk < m_tiles; m_blk += gridDim.x)
            for (int n_blk = 0; n_blk < n_tiles; ++n_blk) {
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * RT_BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint64_t a_desc = make_sdesc_sw128(smem_u32(sA + stage * RT_A_BYTES));
                    const uint64_t b_desc = make_sdesc_sw128(smem_u32(sB + stage * RT_B_BYTES));
#pragma unroll
                    for (int k = 0; k < RT_BK / 16; ++k) umma_ss_w(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0);
                    tc_commit_w(&empty_bar[stage]);
                    if (++stage == RT_STAGES) { stage = 0; phase ^= 1; }
                }
                tc_commit_w(&tfull_bar[acc]);
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
    } else {
        const int ew = warp - 2;
        const int q = warp & 3;
        const int hsel = ew >> 2;                 // column half of the tile this warp reduces
        const int tid_e = threadIdx.x - 64;
        const int r = q * 32 + lane;              // row inside the block
        int acc = 0;
        uint32_t acc_phase = 0;
        for (int m_blk = blockIdx.x; m_blk < m_tiles; m_blk += gridDim.x) {
            Best3 best;
            best.b = INFINITY; best.s = INFINITY; best.i = 0x7fffffff;
            for (int n_blk = 0; n_blk < n_tiles; ++n_blk) {
                const int n0 = n_blk * RT_BN;
                sCst[acc * RT_BN + tid_e] = p.cst[n0 + tid_e];       // 256 epilogue threads <-> 256 columns
                named_bar_sync(1, 256);
                mbar_wait(&tfull_bar[acc], acc_phase);
                tc_fence_after();
                const float* cs = sCst + acc * RT_BN + hsel * (RT_BN / 2);
#pragma unroll 1
                for (int c = 0; c < RT_BN / 2 / 32; ++c) {
                    uint32_t v[32];
                    tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * RT_BN + hsel * (RT_BN / 2) + c * 32, v);
                    tc_wait_ld();
                    const int col0 = n0 + hsel * (RT_BN / 2) + c * 32;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float dot = __uint_as_float(v[j]);
                        const float key = (MODE == 0) ? fmaf(-2.0f, dot, cs[c * 32 + j]) : -(dot + cs[c * 32 + j]);
                        best3_push(best, key, col0 + j);
                    }
                }
                tc_fence_before();
                mbar_arrive(&tempty_bar[acc]);
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
            // merge the two column halves of every row (half 1 -> smem -> half 0), lowest index wins ties
            if (hsel == 1) {
                sMerge[r * 3 + 0] = best.b;
                sMerge[r * 3 + 1] = best.s;
                sMerge[r * 3 + 2] = __int_as_float(best.i);
            }
            named_bar_sync(2, 256);
            if (hsel == 0) {
                const float ob = sMerge[r * 3 + 0], os = sMerge[r * 3 + 1];
                const int oi = __float_as_int(sMerge[r * 3 + 2]);
                const float lose = fmaxf(best.b, ob);
                if (ob < best.b || (ob == best.b && oi < best.i)) { best.b = ob; best.i = oi; }
                best.s = fminf(fminf(best.s, os), lose);
                const int64_t row = (int64_t)m_blk * RT_BM + r;
                if (row < p.M) {
                    // no key compared below +inf (a NaN / inf row of x, or every logit -inf / NaN): id 0, as torch.argmax
                    p.idx[row] = best.i < p.V ? best.i : 0;
                    if (p.margin != nullptr) p.margin[row] = best.s - best.b;
                }
            }
            named_bar_sync(2, 256);      // sMerge may be rewritten for the next row block
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc<512>(tmem_base);
}

static int ew_grid2(int64_t items) {
    const int64_t blocks = (items + 255) / 256, cap = (int64_t)num_sms() * 8;
    return (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}

}  // namespace md

using namespace md;

extern "C" __attribute__((visibility("default"))) int md_round_tc_padded_vocab(int V) { return (V + RT_BN - 1) / RT_BN * RT_BN; }

static bool padded_width_ok(int D, int Dp) { return D > 0 && D % 4 == 0 && Dp >= D && Dp % RT_BK == 0; }

extern "C" __attribute__((visibility("default"))) int md_embed_split_padded(const float* E, int V, int D, int Dp, void* E2, float* sqnorm,
                                                                          float* E_clamped, cudaStream_t stream) {
    if (V <= 0 || !padded_width_ok(D, Dp)) {
        set_last_error("md_embed_split_padded: D=%d must be a positive multiple of 4, Dp=%d a multiple of %d >= D", D, Dp, RT_BK);
        return MD_ERR_ARG;
    }
    const int Vp = md_round_tc_padded_vocab(V);
    embed_prepare_kernel<<<Vp, 128, 0, stream>>>(E, reinterpret_cast<__nv_bfloat16*>(E2), sqnorm, E_clamped, V, Vp, D, Dp);
    return check_cuda(cudaGetLastError(), "embed_split launch");
}

extern "C" __attribute__((visibility("default"))) int md_embed_split(const float* E, int V, int D, void* E2, float* sqnorm, float* E_clamped, cudaStream_t stream) {
    if (V <= 0 || D <= 0 || D % RT_BK != 0) { set_last_error("md_embed_split: D=%d must be a positive multiple of %d", D, RT_BK); return MD_ERR_ARG; }
    return md_embed_split_padded(E, V, D, D, E2, sqnorm, E_clamped, stream);
}

extern "C" __attribute__((visibility("default"))) int md_split_bf16(const float* x, void* out, int64_t rows, int D, int copies, cudaStream_t stream) {
    if (D <= 0 || D % 4 != 0 || copies < 1) { set_last_error("md_split_bf16: D=%d must be a positive multiple of 4, copies >= 1", D); return MD_ERR_ARG; }
    if (rows == 0) return MD_OK;
    split_bf16_kernel<<<ew_grid2(rows * (D / 4)), 256, 0, stream>>>(x, reinterpret_cast<__nv_bfloat16*>(out), rows, D, D, copies);
    return check_cuda(cudaGetLastError(), "split_bf16 launch");
}

extern "C" __attribute__((visibility("default"))) int md_round_argmin_tc_padded(const float* x, const void* E2, const float* cst, void* x2_ws, int32_t* idx,
                                                                              float* margin, int64_t M, int V, int D, int Dp, int mode,
                                                                              cudaStream_t stream) {
    if (!padded_width_ok(D, Dp)) {
        set_last_error("md_round_argmin_tc: D=%d must be a positive multiple of 4, Dp=%d a multiple of %d >= D", D, Dp, RT_BK);
        return MD_ERR_ARG;
    }
    if (V <= 0 || x2_ws == nullptr || cst == nullptr || E2 == nullptr) { set_last_error("md_round_argmin_tc: bad arguments"); return MD_ERR_ARG; }
    if (mode != 0 && mode != 1) { set_last_error("md_round_argmin_tc: mode must be 0 (argmin distance) or 1 (argmax logit)"); return MD_ERR_ARG; }
    if (M == 0) return MD_OK;
    const int Vp = md_round_tc_padded_vocab(V);
    if (x != nullptr) {       // x == NULL: x2_ws already holds the split (written by the producing GEMM's epilogue)
        split_bf16_kernel<<<ew_grid2(M * (Dp / 4)), 256, 0, stream>>>(x, reinterpret_cast<__nv_bfloat16*>(x2_ws), M, D, Dp, 1);
        if (int e = check_cuda(cudaGetLastError(), "split_bf16 launch")) return e;
    }
    // from here on the contraction runs over the padded width: the zero columns add exact zeros
    CUtensorMap tmA, tmB;
    if (int e = make_tmap_2d(&tmA, x2_ws, 0, (uint64_t)M, 2 * Dp, 2 * Dp, RT_BM, RT_BK)) return e;
    if (int e = make_tmap_2d(&tmB, E2, 0, (uint64_t)Vp, 2 * Dp, 2 * Dp, RT_BN, RT_BK)) return e;
    RoundTcArgs a;
    a.M = M; a.V = V; a.Vp = Vp; a.D = Dp; a.cst = cst; a.idx = idx; a.margin = margin;
    static bool attr0[kMaxDevices] = {false}, attr1[kMaxDevices] = {false};
    if (ensure_dyn_smem(round_tc_kernel<0>, RT_SMEM, attr0, "cudaFuncSetAttribute(round_tc)") ||
        ensure_dyn_smem(round_tc_kernel<1>, RT_SMEM, attr1, "cudaFuncSetAttribute(round_tc)"))
        return MD_ERR_CUDA;
    const int m_tiles = (int)((M + RT_BM - 1) / RT_BM);
    const int grid = m_tiles < num_sms() ? m_tiles : num_sms();
    if (mode == 0) round_tc_kernel<0><<<grid, RT_THREADS, RT_SMEM, stream>>>(tmA, tmB, a);
    else round_tc_kernel<1><<<grid, RT_THREADS, RT_SMEM, stream>>>(tmA, tmB, a);
    return check_cuda(cudaGetLastError(), "round_tc launch");
}

extern "C" __attribute__((visibility("default"))) int md_round_argmin_tc(const float* x, const void* E2, const float* cst, void* x2_ws, int32_t* idx, float* margin,
                                  int64_t M, int V, int D, int mode, cudaStream_t stream) {
    if (D % RT_BK != 0 || D <= 0) { set_last_error("md_round_argmin_tc: D=%d must be a positive multiple of %d", D, RT_BK); return MD_ERR_ARG; }
    return md_round_argmin_tc_padded(x, E2, cst, x2_ws, idx, margin, M, V, D, D, mode, stream);
}
