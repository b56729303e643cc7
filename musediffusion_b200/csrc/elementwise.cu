// HBM-bound kernels of the sampling path: fused posterior step, q_sample / noise init, LayerNorm, embedding gather,
// timestep-embedding MLP, casts.  Coalesced 128-bit accesses, warp-shuffle reductions, schedule coefficients in
// __constant__ memory, counter-based Philox noise generated in-kernel.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>

#include "common.cuh"
#include "musediff_b200.h"

namespace md {

// ----------------------------------------------------------------------------------------------
// error plumbing
// ----------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
void set_last_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return MD_OK;
    set_last_error("%s: %s (%s)", what, cudaGetErrorString(e), cudaGetErrorName(e));
    return MD_ERR_CUDA;
}
int num_sms();

// ----------------------------------------------------------------------------------------------
// schedule tables
// ----------------------------------------------------------------------------------------------
enum { TAB_C1 = 0, TAB_C2, TAB_LOGVAR, TAB_SR, TAB_SRM1, TAB_AB, TAB_ABP, TAB_SQRT_AB, TAB_SQRT_1MAB, TAB_COUNT };
constexpr int kConstTabs = 7;
__constant__ float c_sched[kConstTabs * MD_MAX_CONST_T];
// one table set per device (a process may drive several GPUs; __constant__ memory is per device already)
struct SchedState {
    float* dev = nullptr;   // [TAB_COUNT][T] device copy (q_sample tables, and T > MD_MAX_CONST_T)
    int T = 0;
    int cap = 0;
};
static SchedState g_sched[kMaxDevices];
static SchedState& sched_state() { return g_sched[current_device()]; }

struct SchedRef {
    const float* dev;  // device table or nullptr -> constant memory
    int T;
    MD_DEVINL float get(int tab, int t) const {
        return dev ? dev[tab * T + t] : c_sched[tab * MD_MAX_CONST_T + t];
    }
};
static SchedRef sched_ref() {
    const SchedState& st = sched_state();
    SchedRef s;
    s.T = st.T;
    s.dev = (st.T <= MD_MAX_CONST_T) ? nullptr : st.dev;
    return s;
}

// ----------------------------------------------------------------------------------------------
// Philox4x32-7 + inverse-CDF normals.  Seven rounds are the fewest that pass BigCrush (Salmon et al., SC'11, table 2;
// ten is the library default); each round is two 32x32->64 multiplies and two three-input XORs for four outputs.
// A normal costs: its share of the cipher (7 instructions), one LOP3 + one FFMA to turn 23 random bits into
// q = p - 0.5 (mantissa trick, no I2F — conversions run on the 16-lane XU pipe), and the quantile polynomial evaluated
// for two values per instruction (packed f32x2).
// ----------------------------------------------------------------------------------------------
constexpr int kPhiloxRounds = 7;
// Standard normal quantile, general path: Phi^-1(0.5 + q) = sqrt(2) erfinv(2q) for q = p - 0.5 in (-0.5, 0.5).  2|q| is
// exact and erfinvf is within 2 ulp over (-1, 1) (CUDA C++ Programming Guide, mathematical functions), so the result is
// within 2^-21 relative of the exact quantile at every q, well conditioned everywhere, and exactly odd (copysignf).
// Working from q, never from p = q + 0.5 (which rounds to exactly 1.0 for the topmost draw and would turn it into an
// outlier), both tails stop symmetrically at |n| = 5.30 (2|q| = 1 - 2^-23).
MD_DEVINL float norm_quantile_q(float q) {
    return copysignf(1.41421356f * erfinvf(2.0f * fabsf(q)), q);
}
// Quantile for the central band |p - 0.5| <= 0.3414 only (truncation |n| <= 1, the reference default top_p = 1):
// q * P5(q^2), minimax fit, max abs error 1.2e-6 in fp32 — 7 FMA-pipe instructions and no division.
MD_DEVINL float norm_quantile_central(float q) {
    const float r = q * q;
    float p = 643.067138671875f;
    p = fmaf(p, r, -38.967872619628906f);
    p = fmaf(p, r, 21.74688720703125f);
    p = fmaf(p, r, 5.587021827697754f);
    p = fmaf(p, r, 2.6269679069519043f);
    p = fmaf(p, r, 2.506624698638916f);
    return p * q;
}
// the same polynomial for two values per instruction (packed f32x2: 7 issue slots per pair)
MD_DEVINL uint64_t norm_quantile_central_x2(uint64_t q) {
    const uint64_t r = f2_mul(q, q);
    uint64_t p = f2_fma(f2_pack(643.067138671875f, 643.067138671875f), r, f2_pack(-38.967872619628906f, -38.967872619628906f));
    p = f2_fma(p, r, f2_pack(21.74688720703125f, 21.74688720703125f));
    p = f2_fma(p, r, f2_pack(5.587021827697754f, 5.587021827697754f));
    p = f2_fma(p, r, f2_pack(2.6269679069519043f, 2.6269679069519043f));
    p = f2_fma(p, r, f2_pack(2.506624698638916f, 2.506624698638916f));
    return f2_mul(p, q);
}
struct NoiseGen {
    uint32_t kx[kPhiloxRounds], ky[kPhiloxRounds];   // Philox round keys (key + round * Weyl constants), precomputed on the host
    uint32_t step_lo, step_hi;
    float q_scale, q_bias;     // q = p - 0.5 = (m - 1.5) * q_scale + q_bias, m = 1.f + (top 23 random bits) * 2^-23 (mantissa trick)
    int central;               // 1: |q| <= 0.3414 guaranteed -> polynomial quantile
    __host__ void init(uint64_t seed, uint64_t step, float top_p) {
        uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
        for (int r = 0; r < kPhiloxRounds; ++r) {
            kx[r] = k0;
            ky[r] = k1;
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        step_lo = (uint32_t)step;
        step_hi = (uint32_t)(step >> 32);
        double lo = 0.0, span = 1.0;
        if (top_p > 0.0f) {
            lo = 0.5 * erfc((double)top_p / sqrt(2.0));  // Phi(-top_p)
            span = 1.0 - 2.0 * lo;
        }
        // m = 1 + bits23 * 2^-23 in [1, 2);  u = (m - 1) + 2^-24 in (0, 1);  p = lo + u * span;
        // q = p - 0.5 = (m - 1.5) * span + (lo - 0.5 + 0.5 span) + span 2^-24, and lo - 0.5 + 0.5 span = 0 (symmetric band).
        // m - 1.5 is exact in fp32, so the two tails end at exactly -0.5 + 2^-24 and 0.5 - 2^-24 (|n| <= 5.30 untruncated)
        q_scale = (float)span;
        q_bias = (float)((lo - 0.5 + 0.5 * span) + span * 5.9604644775390625e-08);
        central = (top_p > 0.0f && top_p <= 1.0f) ? 1 : 0;
    }
    MD_DEVINL uint4 philox(uint4 c) const {
#pragma unroll
        for (int r = 0; r < kPhiloxRounds; ++r) {
            const uint64_t p0 = (uint64_t)0xD2511F53u * c.x;     // one IMAD.WIDE gives hi and lo
            const uint64_t p1 = (uint64_t)0xCD9E8D57u * c.z;
            c = make_uint4((uint32_t)(p1 >> 32) ^ c.y ^ kx[r], (uint32_t)p1, (uint32_t)(p0 >> 32) ^ c.w ^ ky[r], (uint32_t)p0);
        }
        return c;
    }
    MD_DEVINL float q_of(uint32_t bits) const {                 // 23 random bits -> q = p - 0.5: LOP3 + FADD + FFMA, no I2F
        return fmaf(__fadd_rn(__uint_as_float(0x3f800000u | (bits >> 9)), -1.5f), q_scale, q_bias);
    }
    // four normals for the aligned group of 4 elements starting at global element index 4*g
    template <bool kCentral>
    MD_DEVINL float4 draw4t(uint64_t g, uint32_t slo, uint32_t shi) const {      // step counter supplied by the caller
        const uint4 r = philox(make_uint4((uint32_t)g, (uint32_t)(g >> 32), slo, shi));
        if (kCentral) {
            float4 o;
            f2_unpack(norm_quantile_central_x2(f2_pack(q_of(r.x), q_of(r.y))), o.x, o.y);
            f2_unpack(norm_quantile_central_x2(f2_pack(q_of(r.z), q_of(r.w))), o.z, o.w);
            return o;
        }
        return make_float4(norm_quantile_q(q_of(r.x)), norm_quantile_q(q_of(r.y)), norm_quantile_q(q_of(r.z)), norm_quantile_q(q_of(r.w)));
    }
    template <bool kCentral>
    MD_DEVINL float4 draw4t(uint64_t g) const { return draw4t<kCentral>(g, step_lo, step_hi); }
    MD_DEVINL float4 draw4(uint64_t g) const { return central ? draw4t<true>(g) : draw4t<false>(g); }
};

// flat float4 index -> (token, first element inside the token, sequence).  64-bit divisions cost ~100 instructions
// each on the GPU, so the common power-of-two D goes through shifts and the sequence index through a 32-bit divide.
struct TokPos {
    int64_t tok;
    int d, b;
};
MD_DEVINL TokPos tok_pos(int64_t i, int vec_per_tok, int vshift, int L) {
    TokPos r;
    if (vshift >= 0) {
        r.tok = i >> vshift;
        r.d = (int)(i & (vec_per_tok - 1)) << 2;
    } else {
        r.tok = i / vec_per_tok;
        r.d = (int)(i - r.tok * vec_per_tok) << 2;
    }
    r.b = (int)((uint32_t)r.tok / (uint32_t)L);     // host guarantees tokens < 2^31
    return r;
}
static int vec_shift(int D) {
    const int v = D >> 2;
    if (v <= 0 || (v & (v - 1))) return -1;
    int s = 0;
    while ((1 << s) < v) ++s;
    return s;
}

MD_DEVINL float4 ld_stream_f4(const float* p) {
    float4 v;
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
MD_DEVINL void st_stream_f4(float* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

// ----------------------------------------------------------------------------------------------
// fused posterior step
// ----------------------------------------------------------------------------------------------
struct StepArgs {
    const float* x_t;
    const int32_t* idx;
    const float* pred_in;
    const float* E;
    const float* noise;
    const int32_t* t;
    int t_stride;            // 1 = one schedule index per sequence, 0 = one shared by the whole batch
    const int32_t* mask;
    int64_t mask_tok_stride, mask_d_stride;
    const float* x_start;
    float* x_out;
    __nv_bfloat16* out_bf16;
    float* pred_out;         // optional: processed pred_xstart
    float* mean_out;         // optional: posterior mean ("greedy_mean")
    int64_t seq_offset;
    int B, L, D, vshift;
    int bf16_ld;             // row stride of out_bf16 (>= D; its columns D..bf16_ld-1 are never written)
    float eta;
    int clip;
    NoiseGen rng;
    SchedRef sched;
    const unsigned long long* step_dev;   // optional: Philox step counter read from device memory (CUDA-graph replays)
};
MD_DEVINL void step_counter_of(const StepArgs& a, uint32_t& lo, uint32_t& hi) {
    lo = a.rng.step_lo;
    hi = a.rng.step_hi;
    if (a.step_dev != nullptr) {
        const unsigned long long s = *a.step_dev;
        lo = (uint32_t)s;
        hi = (uint32_t)(s >> 32);
    }
}

MD_DEVINL float clampf(float v, int clip) { return clip == 1 ? fminf(fmaxf(v, -1.0f), 1.0f) : v; }   // clip 2: rows pre-clamped

// per-timestep scalars of one reverse step (computed once per thread when the whole batch shares t)
struct StepCoef {
    float c1, c2, sd;            // DDPM: mean = c1 pred + c2 x ; sample = mean + sd n
    float sr, srm1, ca, cb, sn;  // DDIM
};
template <int MODE>
MD_DEVINL StepCoef step_coef(const SchedRef& sched, int t, float eta) {
    StepCoef k;
    const float nz = (t != 0) ? 1.0f : 0.0f;
    if (MODE == MD_STEP_DDPM) {
        k.c1 = sched.get(TAB_C1, t);
        k.c2 = sched.get(TAB_C2, t);
        k.sd = __fmul_rn(nz, expf(__fmul_rn(0.5f, sched.get(TAB_LOGVAR, t))));
    } else {
        k.sr = sched.get(TAB_SR, t);
        k.srm1 = sched.get(TAB_SRM1, t);
        const float ab = sched.get(TAB_AB, t), abp = sched.get(TAB_ABP, t);
        const float sigma = __fmul_rn(__fmul_rn(eta, __fsqrt_rn(__fdiv_rn(__fsub_rn(1.0f, abp), __fsub_rn(1.0f, ab)))),
                                      __fsqrt_rn(__fsub_rn(1.0f, __fdiv_rn(ab, abp))));
        k.ca = __fsqrt_rn(abp);
        k.cb = __fsqrt_rn(__fsub_rn(__fsub_rn(1.0f, abp), __fmul_rn(sigma, sigma)));
        k.sn = __fmul_rn(nz, sigma);
    }
    return k;
}
// one element: same fp32 operation sequence as the reference's torch expressions (no FMA contraction)
template <int MODE>
MD_DEVINL float step_mean(const StepCoef& k, float x, float p) {
    if (MODE == MD_STEP_DDPM) return __fadd_rn(__fmul_rn(k.c1, p), __fmul_rn(k.c2, x));
    return __fadd_rn(__fmul_rn(p, k.ca), __fmul_rn(k.cb, __fdiv_rn(__fsub_rn(__fmul_rn(k.sr, x), p), k.srm1)));
}
template <int MODE>
MD_DEVINL float step_noise_scale(const StepCoef& k) { return MODE == MD_STEP_DDPM ? k.sd : k.sn; }

constexpr int kStepUnroll = 4;   // float4 items in flight per thread: all loads of a group are issued before any math

// NOISE: 0 = external tensor, 1 = in-kernel Philox + central-band quantile (0 < top_p <= 1), 2 = Philox + general quantile.
// IdxT: int32_t when every element offset fits 31 bits (the usual case; 64-bit address arithmetic costs issue slots).
template <int MODE, int NOISE, typename IdxT>
__global__ void __launch_bounds__(256) posterior_step_kernel(const StepArgs a) {
    const int vec_per_tok = a.D >> 2;
    const IdxT total = (IdxT)((int64_t)a.B * a.L * vec_per_tok);
    const IdxT nthreads = (IdxT)gridDim.x * (IdxT)blockDim.x;
    const bool uniform_t = (a.t_stride == 0);
    StepCoef ku;
    if (uniform_t) ku = step_coef<MODE>(a.sched, a.t[0], a.eta);
    uint32_t slo, shi;
    step_counter_of(a, slo, shi);
    for (IdxT i0 = (IdxT)blockIdx.x * (IdxT)blockDim.x + (IdxT)threadIdx.x; i0 < total; i0 += nthreads * kStepUnroll) {
        IdxT off[kStepUnroll], tok[kStepUnroll];
        int bq[kStepUnroll], dd[kStepUnroll];
        bool ok[kStepUnroll];
        float4 x[kStepUnroll], pr[kStepUnroll], n[kStepUnroll];
        int32_t id[kStepUnroll], mk[kStepUnroll];
        // ---- phase 1: addresses + independent loads
#pragma unroll
        for (int u = 0; u < kStepUnroll; ++u) {
            const IdxT i = i0 + (IdxT)u * nthreads;
            ok[u] = i < total;
            const TokPos tp = tok_pos(ok[u] ? (int64_t)i : 0, vec_per_tok, a.vshift, a.L);
            tok[u] = (IdxT)tp.tok; dd[u] = tp.d; bq[u] = tp.b;
            off[u] = (IdxT)tp.tok * (IdxT)a.D + (IdxT)tp.d;
            if (ok[u]) {
                x[u] = ld_stream_f4(a.x_t + off[u]);
                id[u] = (a.idx != nullptr) ? a.idx[tok[u]] : 0;
                if (a.idx == nullptr) pr[u] = ld_stream_f4(a.pred_in + off[u]);
                if (NOISE == 0) n[u] = ld_stream_f4(a.noise + off[u]);
                mk[u] = (a.mask != nullptr && a.mask_d_stride == 0) ? a.mask[tok[u] * a.mask_tok_stride] : 1;
            }
        }
        // ---- phase 2: dependent gather of the rounded embedding rows (E is L2-resident)
        if (a.idx != nullptr) {
#pragma unroll
            for (int u = 0; u < kStepUnroll; ++u)
                if (ok[u]) pr[u] = *reinterpret_cast<const float4*>(a.E + (int64_t)id[u] * a.D + dd[u]);
        }
        // ---- phase 3: arithmetic + stores
#pragma unroll
        for (int u = 0; u < kStepUnroll; ++u) {
            if (!ok[u]) continue;
            const StepCoef k = uniform_t ? ku : step_coef<MODE>(a.sched, a.t[bq[u] * a.t_stride], a.eta);
            float4 p = pr[u];
            p.x = clampf(p.x, a.clip); p.y = clampf(p.y, a.clip); p.z = clampf(p.z, a.clip); p.w = clampf(p.w, a.clip);
            if (a.pred_out != nullptr) st_stream_f4(a.pred_out + off[u], p);
            const float4 nn = (NOISE == 0) ? n[u]
                              : a.rng.template draw4t<NOISE == 1>((uint64_t)(((a.seq_offset * a.L) * a.D + (int64_t)off[u]) >> 2), slo, shi);
            float4 mu;
            mu.x = step_mean<MODE>(k, x[u].x, p.x);
            mu.y = step_mean<MODE>(k, x[u].y, p.y);
            mu.z = step_mean<MODE>(k, x[u].z, p.z);
            mu.w = step_mean<MODE>(k, x[u].w, p.w);
            if (a.mean_out != nullptr) st_stream_f4(a.mean_out + off[u], mu);
            const float sc = step_noise_scale<MODE>(k);
            float4 o;
            o.x = __fadd_rn(mu.x, __fmul_rn(sc, nn.x));
            o.y = __fadd_rn(mu.y, __fmul_rn(sc, nn.y));
            o.z = __fadd_rn(mu.z, __fmul_rn(sc, nn.z));
            o.w = __fadd_rn(mu.w, __fmul_rn(sc, nn.w));
            if (a.mask != nullptr) {
                if (a.mask_d_stride == 0) {
                    // token-broadcast mask (what run/sample.py builds): x_start is touched only at kept positions
                    if (mk[u] == 0) o = *reinterpret_cast<const float4*>(a.x_start + off[u]);
                } else {
                    const int32_t* mp = a.mask + tok[u] * a.mask_tok_stride + (int64_t)dd[u] * a.mask_d_stride;
                    const int64_t ds = a.mask_d_stride;
                    const bool k0 = mp[0] == 0, k1 = mp[ds] == 0, k2 = mp[2 * ds] == 0, k3 = mp[3 * ds] == 0;
                    if (k0 | k1 | k2 | k3) {
                        const float4 xs = *reinterpret_cast<const float4*>(a.x_start + off[u]);
                        if (k0) o.x = xs.x;
                        if (k1) o.y = xs.y;
                        if (k2) o.z = xs.z;
                        if (k3) o.w = xs.w;
                    }
                }
            }
            st_stream_f4(a.x_out + off[u], o);
            if (a.out_bf16 != nullptr)
                *reinterpret_cast<uint2*>(a.out_bf16 + tok[u] * (IdxT)a.bf16_ld + (IdxT)dd[u]) =
                    make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
        }
    }
}

// Fast path for the shape the sampling loops actually use: D = 128 (one warp = one token row, lane = float4 column),
// token-broadcast or absent mask, fewer than 2^24 tokens.  Four tokens per warp iteration, all loads first; addresses
// are 32-bit and need no divisions (the per-sequence schedule index is only looked up when t is not shared).
template <int MODE, int NOISE, bool CLIP>
__global__ void __launch_bounds__(256) posterior_step_d128_kernel(const StepArgs a) {
    const int lane = threadIdx.x & 31;
    const int M = a.B * a.L;
    const int warp_global = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    const bool uniform_t = (a.t_stride == 0);
    StepCoef ku;
    if (uniform_t) ku = step_coef<MODE>(a.sched, a.t[0], a.eta);
    uint32_t slo, shi;
    step_counter_of(a, slo, shi);
    const uint64_t g_base = (uint64_t)(a.seq_offset * a.L) * 32u + (uint32_t)lane;     // float4 index of token 0, this lane
    for (int tok0 = warp_global * kStepUnroll; tok0 < M; tok0 += nwarps * kStepUnroll) {
        float4 x[kStepUnroll], pr[kStepUnroll], n[kStepUnroll];
        int32_t id[kStepUnroll], mk[kStepUnroll];
#pragma unroll
        for (int u = 0; u < kStepUnroll; ++u) {
            const int tok = tok0 + u;
            if (tok < M) {
                const uint32_t off = (uint32_t)tok * 128u + (uint32_t)lane * 4u;
                x[u] = ld_stream_f4(a.x_t + off);
                if (a.idx != nullptr) id[u] = a.idx[tok];
                else pr[u] = ld_stream_f4(a.pred_in + off);
                if (NOISE == 0) n[u] = ld_stream_f4(a.noise + off);
                mk[u] = (a.mask != nullptr) ? a.mask[(int64_t)tok * a.mask_tok_stride] : 1;
            }
        }
        if (a.idx != nullptr) {
#pragma unroll
            for (int u = 0; u < kStepUnroll; ++u)
                if (tok0 + u < M) pr[u] = *reinterpret_cast<const float4*>(a.E + (uint32_t)id[u] * 128u + (uint32_t)lane * 4u);
        }
#pragma unroll
        for (int u = 0; u < kStepUnroll; ++u) {
            const int tok = tok0 + u;
            if (tok >= M) break;
            const uint32_t off = (uint32_t)tok * 128u + (uint32_t)lane * 4u;
            const StepCoef k = uniform_t ? ku : step_coef<MODE>(a.sched, a.t[tok / a.L], a.eta);
            float4 p = pr[u];
            if (CLIP) { p.x = clampf(p.x, 1); p.y = clampf(p.y, 1); p.z = clampf(p.z, 1); p.w = clampf(p.w, 1); }
            if (a.pred_out != nullptr) st_stream_f4(a.pred_out + off, p);
            const float sc = step_noise_scale<MODE>(k);
            // sigma == 0 (DDIM with eta = 0, or t == 0): the product sc * n is exactly 0 for any finite n -> skip the RNG
            float4 nn = make_float4(0.f, 0.f, 0.f, 0.f);
            if (NOISE == 0) nn = n[u];
            else if (sc != 0.0f) nn = a.rng.template draw4t<NOISE == 1>(g_base + (uint64_t)tok * 32u, slo, shi);
            float4 mu;
            mu.x = step_mean<MODE>(k, x[u].x, p.x);
            mu.y = step_mean<MODE>(k, x[u].y, p.y);
            mu.z = step_mean<MODE>(k, x[u].z, p.z);
            mu.w = step_mean<MODE>(k, x[u].w, p.w);
            if (a.mean_out != nullptr) st_stream_f4(a.mean_out + off, mu);
            float4 o;
            o.x = __fadd_rn(mu.x, __fmul_rn(sc, nn.x));
            o.y = __fadd_rn(mu.y, __fmul_rn(sc, nn.y));
            o.z = __fadd_rn(mu.z, __fmul_rn(sc, nn.z));
            o.w = __fadd_rn(mu.w, __fmul_rn(sc, nn.w));
            if (mk[u] == 0) o = *reinterpret_cast<const float4*>(a.x_start + off);     // kept (conditioning) position
            st_stream_f4(a.x_out + off, o);
            if (a.out_bf16 != nullptr)
                *reinterpret_cast<uint2*>(a.out_bf16 + off) = make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
        }
    }
}

__global__ void __launch_bounds__(256)
xstart_from_eps_kernel(const float* x_t, const float* eps, const int32_t* t, int t_stride, float* out, int B, int L, int D,
                       int vshift, SchedRef s) {
    const int vec_per_tok = D >> 2;
    const int64_t total = (int64_t)B * L * vec_per_tok;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int tt = t[tok_pos(i, vec_per_tok, vshift, L).b * t_stride];
        const float sr = s.get(TAB_SR, tt), srm1 = s.get(TAB_SRM1, tt);
        const float4 x = ld_stream_f4(x_t + i * 4), e = ld_stream_f4(eps + i * 4);
        float4 o;
        o.x = __fsub_rn(__fmul_rn(sr, x.x), __fmul_rn(srm1, e.x));
        o.y = __fsub_rn(__fmul_rn(sr, x.y), __fmul_rn(srm1, e.y));
        o.z = __fsub_rn(__fmul_rn(sr, x.z), __fmul_rn(srm1, e.z));
        o.w = __fsub_rn(__fmul_rn(sr, x.w), __fmul_rn(srm1, e.w));
        st_stream_f4(out + i * 4, o);
    }
}

// ----------------------------------------------------------------------------------------------
// DPM-Solver++(2M) step (Lu et al., "DPM-Solver++", Algorithm 2): x' = a x + b (c0 p + c1 q), q = x0 of the previous
// evaluation read from (and p written back to) the history buffer in place
// ----------------------------------------------------------------------------------------------
struct DpmArgs {
    const float* x_t;
    const int32_t* idx;
    const float* pred_in;
    const float* E;
    float* hist;
    const float* coef;       // [n_coef, 4] = (a, b, c0, c1)
    const int32_t* cursor;   // optional: row *cursor - 1 (after md_step_advance), clamped to [0, n_coef - 1]
    int n_coef;
    const int32_t* mask;
    int64_t mask_tok_stride, mask_d_stride;
    const float* x_start;
    float* x_out;
    __nv_bfloat16* out_bf16;
    int B, L, D, vshift;
    int bf16_ld;
    int clip;
};
// Same load / gather / arithmetic phases as posterior_step_kernel: kStepUnroll float4 items in flight per thread, every
// load of a group issued before any store.  x_t is not read where a == 0 and the history not where c1 == 0.
template <typename IdxT>
__global__ void __launch_bounds__(256) dpm_solver_step_kernel(const DpmArgs a) {
    int row = 0;
    if (a.cursor != nullptr) row = min(max(*a.cursor - 1, 0), a.n_coef - 1);
    const float4 c = *reinterpret_cast<const float4*>(a.coef + 4 * row);
    const float ca = c.x, cb = c.y, c0 = c.z, c1 = c.w;
    const int vec_per_tok = a.D >> 2;
    const IdxT total = (IdxT)((int64_t)a.B * a.L * vec_per_tok);
    const IdxT nthreads = (IdxT)gridDim.x * (IdxT)blockDim.x;
    for (IdxT i0 = (IdxT)blockIdx.x * (IdxT)blockDim.x + (IdxT)threadIdx.x; i0 < total; i0 += nthreads * kStepUnroll) {
        IdxT off[kStepUnroll], tok[kStepUnroll];
        int dd[kStepUnroll];
        bool ok[kStepUnroll];
        float4 x[kStepUnroll], p[kStepUnroll], q[kStepUnroll];
        int32_t id[kStepUnroll], mk[kStepUnroll];
#pragma unroll
        for (int u = 0; u < kStepUnroll; ++u) {
            const IdxT i = i0 + (IdxT)u * nthreads;
            ok[u] = i < total;
            const TokPos tp = tok_pos(ok[u] ? (int64_t)i : 0, vec_per_tok, a.vshift, a.L);
            tok[u] = (IdxT)tp.tok; dd[u] = tp.d;
            off[u] = (IdxT)tp.tok * (IdxT)a.D + (IdxT)tp.d;
            if (ok[u]) {
                if (ca != 0.0f) x[u] = ld_stream_f4(a.x_t + off[u]);
                if (c1 != 0.0f) q[u] = ld_stream_f4(a.hist + off[u]);
                if (a.idx != nullptr) id[u] = a.idx[tok[u]];
                else p[u] = ld_stream_f4(a.pred_in + off[u]);
                mk[u] = (a.mask != nullptr && a.mask_d_stride == 0) ? a.mask[tok[u] * a.mask_tok_stride] : 1;
            }
        }
        if (a.idx != nullptr) {
#pragma unroll
            for (int u = 0; u < kStepUnroll; ++u)
                if (ok[u]) p[u] = *reinterpret_cast<const float4*>(a.E + (int64_t)id[u] * a.D + dd[u]);
        }
#pragma unroll
        for (int u = 0; u < kStepUnroll; ++u) {
            if (!ok[u]) continue;
            float4 pp = p[u];
            pp.x = clampf(pp.x, a.clip); pp.y = clampf(pp.y, a.clip); pp.z = clampf(pp.z, a.clip); pp.w = clampf(pp.w, a.clip);
            // first-order rows (c1 == 0) never read the history: a fresh buffer may hold NaN, and 0 * NaN = NaN
            float4 d;
            if (c1 != 0.0f) {
                d.x = __fadd_rn(__fmul_rn(c0, pp.x), __fmul_rn(c1, q[u].x));
                d.y = __fadd_rn(__fmul_rn(c0, pp.y), __fmul_rn(c1, q[u].y));
                d.z = __fadd_rn(__fmul_rn(c0, pp.z), __fmul_rn(c1, q[u].z));
                d.w = __fadd_rn(__fmul_rn(c0, pp.w), __fmul_rn(c1, q[u].w));
            } else {
                d = make_float4(__fmul_rn(c0, pp.x), __fmul_rn(c0, pp.y), __fmul_rn(c0, pp.z), __fmul_rn(c0, pp.w));
            }
            st_stream_f4(a.hist + off[u], pp);
            // a == 0 (the step to clean data): the output is b d, which is p itself for the row (0, 1, 1, 0)
            float4 o;
            if (ca != 0.0f) {
                o.x = __fadd_rn(__fmul_rn(ca, x[u].x), __fmul_rn(cb, d.x));
                o.y = __fadd_rn(__fmul_rn(ca, x[u].y), __fmul_rn(cb, d.y));
                o.z = __fadd_rn(__fmul_rn(ca, x[u].z), __fmul_rn(cb, d.z));
                o.w = __fadd_rn(__fmul_rn(ca, x[u].w), __fmul_rn(cb, d.w));
            } else {
                o = make_float4(__fmul_rn(cb, d.x), __fmul_rn(cb, d.y), __fmul_rn(cb, d.z), __fmul_rn(cb, d.w));
            }
            if (a.mask != nullptr) {
                if (a.mask_d_stride == 0) {
                    if (mk[u] == 0) o = *reinterpret_cast<const float4*>(a.x_start + off[u]);
                } else {
                    const int32_t* mp = a.mask + tok[u] * a.mask_tok_stride + (int64_t)dd[u] * a.mask_d_stride;
                    const int64_t ds = a.mask_d_stride;
                    const bool k0 = mp[0] == 0, k1 = mp[ds] == 0, k2 = mp[2 * ds] == 0, k3 = mp[3 * ds] == 0;
                    if (k0 | k1 | k2 | k3) {
                        const float4 xs = *reinterpret_cast<const float4*>(a.x_start + off[u]);
                        if (k0) o.x = xs.x;
                        if (k1) o.y = xs.y;
                        if (k2) o.z = xs.z;
                        if (k3) o.w = xs.w;
                    }
                }
            }
            st_stream_f4(a.x_out + off[u], o);
            if (a.out_bf16 != nullptr)
                *reinterpret_cast<uint2*>(a.out_bf16 + tok[u] * (IdxT)a.bf16_ld + (IdxT)dd[u]) =
                    make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
        }
    }
}

struct QSampleArgs {
    const float* x0;
    const float* noise;
    const int32_t* t;
    int t_stride;
    const int32_t* mask;
    int64_t mask_tok_stride, mask_d_stride;
    float* out;
    __nv_bfloat16* out_bf16;
    int64_t seq_offset;
    int B, L, D, vshift;
    int bf16_ld;             // row stride of out_bf16
    NoiseGen rng;
    const float* sched_dev;
    int T;
};
__global__ void __launch_bounds__(256) q_sample_kernel(const QSampleArgs a) {
    const int vec_per_tok = a.D >> 2;
    const int64_t total = (int64_t)a.B * a.L * vec_per_tok;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const TokPos tp = tok_pos(i, vec_per_tok, a.vshift, a.L);
        const int64_t tok = tp.tok;
        const int d = tp.d;
        const int64_t off = tok * a.D + d;
        const int t = a.t ? a.t[tp.b * a.t_stride] : -1;
        const float4 x = ld_stream_f4(a.x0 + off);
        float4 n;
        if (a.noise != nullptr) n = ld_stream_f4(a.noise + off);
        else n = a.rng.draw4((uint64_t)(((a.seq_offset * a.L) * a.D + off) >> 2));
        float4 o = n;
        if (t >= 0) {
            const float ca = a.sched_dev[TAB_SQRT_AB * a.T + t], cb = a.sched_dev[TAB_SQRT_1MAB * a.T + t];
            o.x = __fadd_rn(__fmul_rn(ca, x.x), __fmul_rn(cb, n.x));
            o.y = __fadd_rn(__fmul_rn(ca, x.y), __fmul_rn(cb, n.y));
            o.z = __fadd_rn(__fmul_rn(ca, x.z), __fmul_rn(cb, n.z));
            o.w = __fadd_rn(__fmul_rn(ca, x.w), __fmul_rn(cb, n.w));
        }
        if (a.mask != nullptr) {
            const int32_t* mp = a.mask + tok * a.mask_tok_stride + (int64_t)d * a.mask_d_stride;
            const int64_t ds = a.mask_d_stride;
            if (mp[0] == 0) o.x = x.x;
            if (mp[ds] == 0) o.y = x.y;
            if (mp[2 * ds] == 0) o.z = x.z;
            if (mp[3 * ds] == 0) o.w = x.w;
        }
        st_stream_f4(a.out + off, o);
        if (a.out_bf16 != nullptr)
            *reinterpret_cast<uint2*>(a.out_bf16 + tok * a.bf16_ld + d) = make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
    }
}

__global__ void __launch_bounds__(256) fill_normal_kernel(float* out, int64_t n, int64_t elem_offset, NoiseGen rng) {
    const int64_t nv = (n + 3) >> 2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = rng.draw4((uint64_t)((elem_offset >> 2) + i));
        const float vv[4] = {v.x, v.y, v.z, v.w};
        for (int j = 0; j < 4; ++j)
            if (i * 4 + j < n) out[i * 4 + j] = vv[j];
    }
}

// ----------------------------------------------------------------------------------------------
// hidden_dim == hidden_size models (network.py:141-149 without input_up_proj, :153-157 without output_down_proj):
// pre-LayerNorm sum pos[l] + x + emb_t[b] straight from the fp32 state, and the bf16 -> fp32 cast of the last hidden state
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) add_pos_time_kernel(const float* __restrict__ x, const float* __restrict__ pos, const float* __restrict__ temb,
                                                           int temb_stride, int L, int H, __nv_bfloat16* __restrict__ out, int64_t M) {
    const int vec = H >> 2;
    const int64_t total = M * vec;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t m = i / vec;
        const int c = (int)(i - m * vec) << 2;
        const int64_t b = m / L;
        const int l = (int)(m - b * L);
        const float4 v = ld_stream_f4(x + m * H + c);
        const float4 pp = *reinterpret_cast<const float4*>(pos + (int64_t)l * H + c);
        const float4 tt = *reinterpret_cast<const float4*>(temb + b * temb_stride + c);
        // same association as the reference: (pos + emb_x) + emb_t   (network.py:147)
        *reinterpret_cast<uint2*>(out + m * H + c) = make_uint2(pack_bf16x2((pp.x + v.x) + tt.x, (pp.y + v.y) + tt.y),
                                                                pack_bf16x2((pp.z + v.z) + tt.z, (pp.w + v.w) + tt.w));
    }
}
__global__ void __launch_bounds__(256) cast_bf16_f32_kernel(const __nv_bfloat16* __restrict__ in, float* __restrict__ out, int64_t n4) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const uint2 u = *reinterpret_cast<const uint2*>(in + i * 4);
        const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y);
        st_stream_f4(out + i * 4, make_float4(a.x, a.y, b.x, b.y));
    }
}

// ----------------------------------------------------------------------------------------------
// casts / gather
// ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) cast_f32_bf16_kernel(const float* in, __nv_bfloat16* out, int64_t n4) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = ld_stream_f4(in + i * 4);
        *reinterpret_cast<uint2*>(out + i * 4) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
    }
}
// fp32 [rows, D] -> bf16 rows of stride ld >= D (columns D..ld-1 untouched)
__global__ void __launch_bounds__(256) cast_f32_bf16_ld_kernel(const float* in, __nv_bfloat16* out, int64_t rows, int D, int ld) {
    const int vec = D >> 2;
    const int64_t total = rows * vec;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / vec;
        const int c = (int)(i - r * vec) << 2;
        const float4 v = ld_stream_f4(in + i * 4);
        *reinterpret_cast<uint2*>(out + r * ld + c) = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
    }
}
template <typename IdT>
__global__ void __launch_bounds__(256) embed_gather_kernel(const float* E, const IdT* ids, float* out, int64_t M, int V, int D,
                                                           int* err_flag) {
    const int vec_per_tok = D >> 2;
    const int64_t total = M * vec_per_tok;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t tok = i / vec_per_tok;
        const int d = (int)(i - tok * vec_per_tok) << 2;
        int64_t id = (int64_t)ids[tok];
        if (id < 0 || id >= V) { if (err_flag) atomicExch(err_flag, 1); id = 0; }
        st_stream_f4(out + tok * D + d, *reinterpret_cast<const float4*>(E + id * D + d));
    }
}

// ----------------------------------------------------------------------------------------------
// LayerNorm (bf16 in/out, fp32 statistics), one warp per row
// ----------------------------------------------------------------------------------------------
template <int VEC, bool kHoist>  // VEC 16-byte vectors (8 bf16) per lane: H = 256 * VEC; kHoist: gamma / beta live in registers
__global__ void __launch_bounds__(256) layernorm_kernel(const __nv_bfloat16* __restrict__ in,
                                                        const __nv_bfloat16* __restrict__ resid,
                                                        const float* __restrict__ gamma, const float* __restrict__ beta,
                                                        float eps, __nv_bfloat16* __restrict__ out, int64_t M) {
    constexpr int H = 256 * VEC;
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    // gamma / beta are the same for every row: re-loading them per row (6 KB against 4.6 KB of activations) made the
    // L1 data pipe, not HBM, the limiter once the SM clock drops under the power cap
    float hg[kHoist ? VEC * 8 : 1], hb[kHoist ? VEC * 8 : 1];
    if (kHoist) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const int c = (j * 32 + lane) * 8;
#pragma unroll
            for (int e = 0; e < 8; ++e) { hg[j * 8 + e] = gamma[c + e]; hb[j * 8 + e] = beta[c + e]; }
        }
    }
    for (int64_t row = warp_global; row < M; row += nwarps) {
        const __nv_bfloat16* p = in + row * H;
        float v[VEC * 8];
        uint4 u[VEC], ur[VEC];
#pragma unroll
        for (int j = 0; j < VEC; ++j) u[j] = *reinterpret_cast<const uint4*>(p + (j * 32 + lane) * 8);
        if (resid != nullptr) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) ur[j] = *reinterpret_cast<const uint4*>(resid + row * H + (j * 32 + lane) * 8);
        }
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const uint32_t w[4] = {u[j].x, u[j].y, u[j].z, u[j].w};
            const uint32_t wr[4] = {ur[j].x, ur[j].y, ur[j].z, ur[j].w};
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                float2 f = unpack_bf16x2(w[h]);
                if (resid != nullptr) {
                    const float2 g = unpack_bf16x2(wr[h]);
                    f.x += g.x;
                    f.y += g.y;
                }
                v[j * 8 + 2 * h] = f.x;
                v[j * 8 + 2 * h + 1] = f.y;
            }
        }
        float s = 0.f;
#pragma unroll
        for (int j = 0; j < VEC * 8; ++j) s += v[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        // correctly rounded: for a constant row c the sum H c is exact, and s / H is then exactly c at every width
        // (s * fl(1/H) is not for H = 1792, where a constant row came out as beta +- gamma * O(1) instead of beta)
        const float mean = __fdiv_rn(s, (float)H);
        float q = 0.f;
#pragma unroll
        for (int j = 0; j < VEC * 8; ++j) { const float dlt = v[j] - mean; q = fmaf(dlt, dlt, q); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        const float rstd = rsqrtf(q * (1.0f / H) + eps);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const int c = (j * 32 + lane) * 8;
            float y[8];
            if (kHoist) {
#pragma unroll
                for (int e = 0; e < 8; ++e) y[e] = fmaf((v[j * 8 + e] - mean) * rstd, hg[j * 8 + e], hb[j * 8 + e]);
            } else {
                const float4 g0 = *reinterpret_cast<const float4*>(gamma + c), g1 = *reinterpret_cast<const float4*>(gamma + c + 4);
                const float4 b0 = *reinterpret_cast<const float4*>(beta + c), b1 = *reinterpret_cast<const float4*>(beta + c + 4);
                const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
                const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                for (int e = 0; e < 8; ++e) y[e] = fmaf((v[j * 8 + e] - mean) * rstd, gg[e], bb[e]);
            }
            *reinterpret_cast<uint4*>(out + row * H + c) = make_uint4(pack_bf16x2(y[0], y[1]), pack_bf16x2(y[2], y[3]),
                                                                     pack_bf16x2(y[4], y[5]), pack_bf16x2(y[6], y[7]));
        }
    }
}

// ----------------------------------------------------------------------------------------------
// timestep embedding + time_embed MLP, fp32, warp-per-output-row dot products.  Two launches (hidden layer, output
// layer), each spread over B x row-chunks CTAs: inside the sampling loops B is 1 (all sequences share t), so a
// single-CTA formulation would stream the 1.5 MB second weight matrix through one SM.
// ----------------------------------------------------------------------------------------------
constexpr int kTmlpRowsPerCta = 32;
__global__ void __launch_bounds__(256) timestep_hidden_kernel(const float* __restrict__ t, const float* __restrict__ W0,
                                                              const float* __restrict__ b0, float* __restrict__ hid,
                                                              int t_dim, int mid_dim) {
    extern __shared__ float emb[];   // [t_dim]
    const int b = blockIdx.y;
    const int half = t_dim / 2;
    const float tv = t[b];
    for (int k = threadIdx.x; k < t_dim; k += blockDim.x) {
        float e = 0.f;
        if (k < 2 * half) {
            const int kk = (k < half) ? k : k - half;
            // freqs = exp(-log(10000) * arange(half) / half) in fp32, args = t * freqs  (network.py:121-125)
            const float freq = expf(-9.210340371976184f * (float)kk / (float)half);
            const float arg = tv * freq;
            e = (k < half) ? cosf(arg) : sinf(arg);
        }
        emb[k] = e;
    }
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int r0 = blockIdx.x * kTmlpRowsPerCta;
    for (int r = r0 + warp; r < min(r0 + kTmlpRowsPerCta, mid_dim); r += nw) {
        float acc = 0.f;
        for (int k = lane; k < t_dim; k += 32) acc = fmaf(W0[(size_t)r * t_dim + k], emb[k], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
            const float z = acc + b0[r];
            hid[(size_t)b * mid_dim + r] = z / (1.0f + expf(-z));   // SiLU
        }
    }
}
__global__ void __launch_bounds__(256) timestep_out_kernel(const float* __restrict__ hid, const float* __restrict__ W2,
                                                           const float* __restrict__ b2, float* __restrict__ out,
                                                           int mid_dim, int out_dim) {
    extern __shared__ float hs[];    // [mid_dim]
    const int b = blockIdx.y;
    for (int k = threadIdx.x; k < mid_dim; k += blockDim.x) hs[k] = hid[(size_t)b * mid_dim + k];
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int r0 = blockIdx.x * kTmlpRowsPerCta;
    for (int r = r0 + warp; r < min(r0 + kTmlpRowsPerCta, out_dim); r += nw) {
        float acc = 0.f;
        for (int k = lane; k < mid_dim; k += 32) acc = fmaf(W2[(size_t)r * mid_dim + k], hs[k], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) out[(size_t)b * out_dim + r] = acc + b2[r];
    }
}

// get_logits, logits_mode 2 (network.py:94-104): scores[m, v] = -sqrt(clamp(|E_v|^2 + |x_m|^2 - 2 x_m.E_v, 0)); the dot products
// come from the split-bf16 tensor-core GEMM, |E_v|^2 from md_embed_split.  One warp per row: |x_m|^2 by shuffle reduction.
__global__ void __launch_bounds__(256) dist_scores_kernel(const float* __restrict__ x, const float* __restrict__ dot, const float* __restrict__ esq,
                                                          float* __restrict__ out, int64_t M, int V, int dot_stride, int D) {
    const int lane = threadIdx.x & 31;
    const int64_t warp_global = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t m = warp_global; m < M; m += nwarps) {
        float q = 0.f;
        for (int d = lane; d < D; d += 32) { const float v = x[m * D + d]; q = fmaf(v, v, q); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
        for (int v = lane; v < V; v += 32) {
            const float d2 = __fsub_rn(__fadd_rn(esq[v], q), __fmul_rn(2.0f, dot[m * dot_stride + v]));
            out[m * V + v] = -sqrtf(fmaxf(d2, 0.0f));
        }
    }
}

static int ew_grid(int64_t work_items, int threads) {
    const int64_t blocks = (work_items + threads - 1) / threads;
    const int64_t cap = (int64_t)num_sms() * 8;   // 8 resident 256-thread CTAs per SM, grid-stride beyond that
    return (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}

}  // namespace md

using namespace md;

extern "C" __attribute__((visibility("default"))) const char* md_last_error(void) { return g_err; }
extern "C" __attribute__((visibility("default"))) int md_abi_version(void) { return 2; }

// Device-resident loop state for CUDA-graph replays of one reverse step: the graph is captured once and every replay reads
// its schedule index / model timestep / Philox counter from device memory.  One thread: k = *cursor;
// t_cur = t_idx[min(k, n-1)], tm_cur = t_model[min(k, n-1)], ctr_cur = ctr_base + k, *cursor = k + 1.
__global__ void step_advance_kernel(int32_t* cursor, const int32_t* t_idx, const float* t_model, int n, int32_t* t_cur,
                                    float* tm_cur, unsigned long long* ctr_cur, unsigned long long ctr_base) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const int k = *cursor;
    const int kk = k < n ? k : n - 1;
    *t_cur = t_idx[kk];
    *tm_cur = t_model[kk];
    *ctr_cur = ctr_base + (unsigned long long)k;
    *cursor = k + 1;
}
extern "C" __attribute__((visibility("default"))) int md_step_advance(int32_t* cursor, const int32_t* t_idx, const float* t_model, int n, int32_t* t_cur,
                               float* tm_cur, uint64_t* ctr_cur, uint64_t ctr_base, cudaStream_t stream) {
    if (cursor == nullptr || t_idx == nullptr || t_model == nullptr || t_cur == nullptr || tm_cur == nullptr || ctr_cur == nullptr || n <= 0) {
        set_last_error("md_step_advance: null pointer or empty schedule (n=%d)", n);
        return MD_ERR_ARG;
    }
    step_advance_kernel<<<1, 32, 0, stream>>>(cursor, t_idx, t_model, n, t_cur, tm_cur, reinterpret_cast<unsigned long long*>(ctr_cur), ctr_base);
    return check_cuda(cudaGetLastError(), "step_advance launch");
}

extern "C" __attribute__((visibility("default"))) int md_set_schedule(const float* tables, int T, cudaStream_t stream) {
    if (tables == nullptr || T <= 0) { set_last_error("md_set_schedule: bad arguments (T=%d)", T); return MD_ERR_ARG; }
    SchedState& st = sched_state();          // the calling thread's current device
    if (T > st.cap) {
        if (st.dev) cudaFree(st.dev);
        st.dev = nullptr;
        st.cap = 0;
        if (check_cuda(cudaMalloc(&st.dev, sizeof(float) * TAB_COUNT * T), "cudaMalloc(schedule)")) return MD_ERR_CUDA;
        st.cap = T;
    }
    st.T = T;
    if (check_cuda(cudaMemcpyAsync(st.dev, tables, sizeof(float) * TAB_COUNT * T, cudaMemcpyHostToDevice, stream),
                   "cudaMemcpyAsync(schedule)"))
        return MD_ERR_CUDA;
    if (T <= MD_MAX_CONST_T) {
        for (int k = 0; k < kConstTabs; ++k)
            if (check_cuda(cudaMemcpyToSymbolAsync(c_sched, tables + (size_t)k * T, sizeof(float) * T,
                                                   sizeof(float) * k * MD_MAX_CONST_T, cudaMemcpyHostToDevice, stream),
                           "cudaMemcpyToSymbolAsync(schedule)"))
                return MD_ERR_CUDA;
    }
    return check_cuda(cudaStreamSynchronize(stream), "md_set_schedule sync");
}

extern "C" __attribute__((visibility("default"))) int md_dist_scores(const float* x, const float* dot, const float* esq, float* out, int64_t M, int V,
                              int dot_stride, int D, cudaStream_t stream) {
    if (M == 0) return MD_OK;
    if (V <= 0 || D <= 0 || dot_stride < V) { set_last_error("md_dist_scores: bad sizes V=%d D=%d stride=%d", V, D, dot_stride); return MD_ERR_ARG; }
    dist_scores_kernel<<<ew_grid(M * 32, 256), 256, 0, stream>>>(x, dot, esq, out, M, V, dot_stride, D);
    return check_cuda(cudaGetLastError(), "dist_scores launch");
}

extern "C" __attribute__((visibility("default"))) int md_cast_f32_bf16(const float* in, void* out, int64_t n, cudaStream_t stream) {
    if (n % 4 != 0) { set_last_error("md_cast_f32_bf16: n must be a multiple of 4"); return MD_ERR_ARG; }
    if (n == 0) return MD_OK;
    cast_f32_bf16_kernel<<<ew_grid(n / 4, 256), 256, 0, stream>>>(in, reinterpret_cast<__nv_bfloat16*>(out), n / 4);
    return check_cuda(cudaGetLastError(), "cast launch");
}

extern "C" __attribute__((visibility("default"))) int md_cast_f32_bf16_ld(const float* in, void* out, int64_t rows, int D, int ld,
                                                                        cudaStream_t stream) {
    if (D <= 0 || D % 4 != 0 || ld < D || ld % 4 != 0) {
        set_last_error("md_cast_f32_bf16_ld: D=%d must be a positive multiple of 4, ld=%d a multiple of 4 >= D", D, ld);
        return MD_ERR_ARG;
    }
    if (rows == 0) return MD_OK;
    cast_f32_bf16_ld_kernel<<<ew_grid(rows * (D / 4), 256), 256, 0, stream>>>(in, reinterpret_cast<__nv_bfloat16*>(out), rows, D, ld);
    return check_cuda(cudaGetLastError(), "cast launch");
}

extern "C" __attribute__((visibility("default"))) int md_cast_bf16_f32(const void* in, float* out, int64_t n, cudaStream_t stream) {
    if (n % 4 != 0) { set_last_error("md_cast_bf16_f32: n must be a multiple of 4"); return MD_ERR_ARG; }
    if (n == 0) return MD_OK;
    cast_bf16_f32_kernel<<<ew_grid(n / 4, 256), 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(in), out, n / 4);
    return check_cuda(cudaGetLastError(), "cast launch");
}

extern "C" __attribute__((visibility("default"))) int md_add_pos_time(const float* x, const float* pos, const float* temb, int temb_stride, int L, int H,
                               void* out_bf16, int64_t M, cudaStream_t stream) {
    if (H % 4 != 0 || L <= 0 || M % L != 0 || pos == nullptr || temb == nullptr) {
        set_last_error("md_add_pos_time: H %% 4 == 0, L > 0 dividing M, pos and temb required (H=%d L=%d)", H, L);
        return MD_ERR_ARG;
    }
    if (M == 0) return MD_OK;
    add_pos_time_kernel<<<ew_grid(M * (H / 4), 256), 256, 0, stream>>>(x, pos, temb, temb_stride, L, H, reinterpret_cast<__nv_bfloat16*>(out_bf16), M);
    return check_cuda(cudaGetLastError(), "add_pos_time launch");
}

extern "C" __attribute__((visibility("default"))) int md_embed_gather(const float* E, const void* ids, int ids_is_i64, float* out, int64_t M, int V, int D,
                               cudaStream_t stream) {
    if (D % 4 != 0) { set_last_error("md_embed_gather: D must be a multiple of 4"); return MD_ERR_ARG; }
    if (M == 0) return MD_OK;
    const int grid = ew_grid(M * (D / 4), 256);
    if (ids_is_i64) embed_gather_kernel<int64_t><<<grid, 256, 0, stream>>>(E, (const int64_t*)ids, out, M, V, D, nullptr);
    else embed_gather_kernel<int32_t><<<grid, 256, 0, stream>>>(E, (const int32_t*)ids, out, M, V, D, nullptr);
    return check_cuda(cudaGetLastError(), "embed_gather launch");
}

extern "C" __attribute__((visibility("default"))) int md_timestep_mlp(const float* t, const float* W0, const float* b0, const float* W2, const float* b2,
                               float* out, float* hidden_ws, int B, int t_dim, int mid_dim, int out_dim, cudaStream_t stream) {
    if (B <= 0) return MD_OK;
    if (hidden_ws == nullptr) { set_last_error("md_timestep_mlp: hidden workspace [B, mid_dim] missing"); return MD_ERR_ARG; }
    dim3 g1((mid_dim + kTmlpRowsPerCta - 1) / kTmlpRowsPerCta, B), g2((out_dim + kTmlpRowsPerCta - 1) / kTmlpRowsPerCta, B);
    timestep_hidden_kernel<<<g1, 256, sizeof(float) * t_dim, stream>>>(t, W0, b0, hidden_ws, t_dim, mid_dim);
    timestep_out_kernel<<<g2, 256, sizeof(float) * mid_dim, stream>>>(hidden_ws, W2, b2, out, mid_dim, out_dim);
    return check_cuda(cudaGetLastError(), "timestep_mlp launch");
}

extern "C" __attribute__((visibility("default"))) int md_layernorm_bf16(const void* in, const void* resid, const float* gamma, const float* beta, float eps, void* out,
                                 int64_t M, int H, cudaStream_t stream) {
    if (H % 256 != 0 || H > 2048 || H <= 0) { set_last_error("md_layernorm_bf16: H=%d must be a multiple of 256, <= 2048", H); return MD_ERR_ARG; }
    if (M == 0) return MD_OK;
    const int grid = ew_grid(M * 32, 256);
    const __nv_bfloat16* i = reinterpret_cast<const __nv_bfloat16*>(in);
    __nv_bfloat16* o = reinterpret_cast<__nv_bfloat16*>(out);
    const __nv_bfloat16* r = reinterpret_cast<const __nv_bfloat16*>(resid);
    static const bool hoist = env_int("MD_LN_HOIST", 1) != 0;
    switch (H / 256) {
        case 1: layernorm_kernel<1, true><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M); break;
        case 2: layernorm_kernel<2, true><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M); break;
        case 3: if (hoist) layernorm_kernel<3, true><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M);
                else layernorm_kernel<3, false><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M);
                break;
        case 4: if (hoist) layernorm_kernel<4, true><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M);
                else layernorm_kernel<4, false><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M);
                break;
        case 5: layernorm_kernel<5, false><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M); break;
        case 6: layernorm_kernel<6, false><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M); break;
        case 7: layernorm_kernel<7, false><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M); break;
        default: layernorm_kernel<8, false><<<grid, 256, 0, stream>>>(i, r, gamma, beta, eps, o, M); break;
    }
    return check_cuda(cudaGetLastError(), "layernorm launch");
}

extern "C" __attribute__((visibility("default"))) int md_posterior_step_ld(const float* x_t, const int32_t* idx, const float* pred_in, const float* E,
                                 const float* noise, uint64_t seed, uint64_t step_counter, int64_t seq_offset,
                                 const int32_t* t, int t_stride, const int32_t* mask, int64_t mask_tok_stride,
                                 int64_t mask_d_stride, const float* x_start, float* x_out, void* out_bf16, int bf16_ld,
                                 float* pred_out, float* mean_out, int B, int L, int D, int mode, float eta, int clip,
                                 float top_p, const uint64_t* step_counter_dev, cudaStream_t stream) {
    if (sched_state().T == 0) { set_last_error("md_posterior_step: md_set_schedule has not been called on this device"); return MD_ERR_ARG; }
    if (D % 4 != 0) { set_last_error("md_posterior_step: D must be a multiple of 4"); return MD_ERR_ARG; }
    if (bf16_ld < D || bf16_ld % 4 != 0) { set_last_error("md_posterior_step: bf16_ld=%d must be a multiple of 4 >= D=%d", bf16_ld, D); return MD_ERR_ARG; }
    if ((idx == nullptr) == (pred_in == nullptr)) { set_last_error("md_posterior_step: exactly one of idx / pred_in"); return MD_ERR_ARG; }
    if (idx != nullptr && E == nullptr) { set_last_error("md_posterior_step: idx needs E"); return MD_ERR_ARG; }
    if (clip == 2 && idx == nullptr) { set_last_error("md_posterior_step: clip = 2 (pre-clamped E) needs idx"); return MD_ERR_ARG; }
    if (mask != nullptr && x_start == nullptr) { set_last_error("md_posterior_step: mask needs x_start"); return MD_ERR_ARG; }
    if (mode != MD_STEP_DDPM && mode != MD_STEP_DDIM) { set_last_error("md_posterior_step: bad mode %d", mode); return MD_ERR_ARG; }
    if ((int64_t)B * L == 0) return MD_OK;
    if ((int64_t)B * L >= (int64_t)1 << 31) { set_last_error("md_posterior_step: more than 2^31 tokens"); return MD_ERR_ARG; }
    StepArgs a;
    a.x_t = x_t; a.idx = idx; a.pred_in = pred_in; a.E = E; a.noise = noise; a.t = t; a.t_stride = t_stride ? 1 : 0;
    a.mask = mask; a.pred_out = pred_out; a.mean_out = mean_out;
    a.mask_tok_stride = mask_tok_stride; a.mask_d_stride = mask_d_stride; a.x_start = x_start; a.x_out = x_out;
    a.out_bf16 = reinterpret_cast<__nv_bfloat16*>(out_bf16); a.seq_offset = seq_offset; a.B = B; a.L = L; a.D = D;
    a.eta = eta; a.clip = clip; a.rng.init(seed, step_counter, top_p); a.sched = sched_ref(); a.vshift = vec_shift(D);
    a.bf16_ld = bf16_ld;
    a.step_dev = reinterpret_cast<const unsigned long long*>(step_counter_dev);
    const int grid = ew_grid(((int64_t)B * L * (D / 4) + kStepUnroll - 1) / kStepUnroll, 256);
    const int nz = (noise != nullptr) ? 0 : (a.rng.central ? 1 : 2);
    if (D == 128 && bf16_ld == 128 && (mask == nullptr || mask_d_stride == 0) && (int64_t)B * L < (1 << 24)) {
        const int g2 = ew_grid(((int64_t)B * L + kStepUnroll - 1) / kStepUnroll * 32, 256);
#define MD_LAUNCH_FAST(MODE_, CLIP_)                                                                              \
    do {                                                                                                          \
        if (nz == 0) posterior_step_d128_kernel<MODE_, 0, CLIP_><<<g2, 256, 0, stream>>>(a);                      \
        else if (nz == 1) posterior_step_d128_kernel<MODE_, 1, CLIP_><<<g2, 256, 0, stream>>>(a);                 \
        else posterior_step_d128_kernel<MODE_, 2, CLIP_><<<g2, 256, 0, stream>>>(a);                              \
    } while (0)
        if (mode == MD_STEP_DDPM) { if (a.clip == 1) MD_LAUNCH_FAST(MD_STEP_DDPM, true); else MD_LAUNCH_FAST(MD_STEP_DDPM, false); }
        else { if (a.clip == 1) MD_LAUNCH_FAST(MD_STEP_DDIM, true); else MD_LAUNCH_FAST(MD_STEP_DDIM, false); }
#undef MD_LAUNCH_FAST
        return check_cuda(cudaGetLastError(), "posterior_step launch");
    }
    const bool small = (int64_t)B * L * bf16_ld + (int64_t)grid * 256 * kStepUnroll * 4 < ((int64_t)1 << 31);
#define MD_LAUNCH_STEP(MODE_, NZ_)                                                                     \
    do {                                                                                               \
        if (small) posterior_step_kernel<MODE_, NZ_, int32_t><<<grid, 256, 0, stream>>>(a);            \
        else posterior_step_kernel<MODE_, NZ_, int64_t><<<grid, 256, 0, stream>>>(a);                  \
    } while (0)
    if (mode == MD_STEP_DDPM) {
        if (nz == 0) MD_LAUNCH_STEP(MD_STEP_DDPM, 0); else if (nz == 1) MD_LAUNCH_STEP(MD_STEP_DDPM, 1); else MD_LAUNCH_STEP(MD_STEP_DDPM, 2);
    } else {
        if (nz == 0) MD_LAUNCH_STEP(MD_STEP_DDIM, 0); else if (nz == 1) MD_LAUNCH_STEP(MD_STEP_DDIM, 1); else MD_LAUNCH_STEP(MD_STEP_DDIM, 2);
    }
#undef MD_LAUNCH_STEP
    return check_cuda(cudaGetLastError(), "posterior_step launch");
}

extern "C" __attribute__((visibility("default"))) int md_posterior_step(const float* x_t, const int32_t* idx, const float* pred_in, const float* E,
                                 const float* noise, uint64_t seed, uint64_t step_counter, int64_t seq_offset,
                                 const int32_t* t, int t_stride, const int32_t* mask, int64_t mask_tok_stride,
                                 int64_t mask_d_stride, const float* x_start, float* x_out, void* out_bf16,
                                 float* pred_out, float* mean_out, int B, int L, int D, int mode, float eta, int clip,
                                 float top_p, const uint64_t* step_counter_dev, cudaStream_t stream) {
    return md_posterior_step_ld(x_t, idx, pred_in, E, noise, seed, step_counter, seq_offset, t, t_stride, mask, mask_tok_stride,
                                mask_d_stride, x_start, x_out, out_bf16, D, pred_out, mean_out, B, L, D, mode, eta, clip, top_p,
                                step_counter_dev, stream);
}

extern "C" __attribute__((visibility("default"))) int md_dpm_solver_step(const float* x_t, const int32_t* idx, const float* pred_in, const float* E,
                                  float* pred_hist, const float* coef, int n_coef, const int32_t* cursor,
                                  const int32_t* mask, int64_t mask_tok_stride, int64_t mask_d_stride, const float* x_start,
                                  float* x_out, void* out_bf16, int bf16_ld, int B, int L, int D, int clip,
                                  cudaStream_t stream) {
    if (D <= 0 || D % 4 != 0) { set_last_error("md_dpm_solver_step: D=%d must be a positive multiple of 4", D); return MD_ERR_ARG; }
    if (bf16_ld < D || bf16_ld % 4 != 0) { set_last_error("md_dpm_solver_step: bf16_ld=%d must be a multiple of 4 >= D=%d", bf16_ld, D); return MD_ERR_ARG; }
    if ((idx == nullptr) == (pred_in == nullptr)) { set_last_error("md_dpm_solver_step: exactly one of idx / pred_in"); return MD_ERR_ARG; }
    if (idx != nullptr && E == nullptr) { set_last_error("md_dpm_solver_step: idx needs E"); return MD_ERR_ARG; }
    if (clip == 2 && idx == nullptr) { set_last_error("md_dpm_solver_step: clip = 2 (pre-clamped E) needs idx"); return MD_ERR_ARG; }
    if (clip < 0 || clip > 2) { set_last_error("md_dpm_solver_step: bad clip %d", clip); return MD_ERR_ARG; }
    if (mask != nullptr && x_start == nullptr) { set_last_error("md_dpm_solver_step: mask needs x_start"); return MD_ERR_ARG; }
    if (pred_hist == nullptr || coef == nullptr || n_coef <= 0 || (cursor == nullptr && n_coef != 1)) {
        set_last_error("md_dpm_solver_step: history and coefficient table required; without a cursor the table has one row (n_coef=%d)", n_coef);
        return MD_ERR_ARG;
    }
    if ((int64_t)B * L == 0) return MD_OK;
    if ((int64_t)B * L >= (int64_t)1 << 31) { set_last_error("md_dpm_solver_step: more than 2^31 tokens"); return MD_ERR_ARG; }
    DpmArgs a;
    a.x_t = x_t; a.idx = idx; a.pred_in = pred_in; a.E = E; a.hist = pred_hist; a.coef = coef; a.cursor = cursor; a.n_coef = n_coef;
    a.mask = mask; a.mask_tok_stride = mask_tok_stride; a.mask_d_stride = mask_d_stride; a.x_start = x_start; a.x_out = x_out;
    a.out_bf16 = reinterpret_cast<__nv_bfloat16*>(out_bf16); a.B = B; a.L = L; a.D = D; a.vshift = vec_shift(D);
    a.bf16_ld = bf16_ld; a.clip = clip;
    const int grid = ew_grid(((int64_t)B * L * (D / 4) + kStepUnroll - 1) / kStepUnroll, 256);
    if ((int64_t)B * L * bf16_ld + (int64_t)grid * 256 * kStepUnroll * 4 < ((int64_t)1 << 31))
        dpm_solver_step_kernel<int32_t><<<grid, 256, 0, stream>>>(a);
    else
        dpm_solver_step_kernel<int64_t><<<grid, 256, 0, stream>>>(a);
    return check_cuda(cudaGetLastError(), "dpm_solver_step launch");
}

extern "C" __attribute__((visibility("default"))) int md_xstart_from_eps(const float* x_t, const float* eps, const int32_t* t, int t_stride, float* out, int B, int L,
                                  int D, cudaStream_t stream) {
    if (sched_state().T == 0) { set_last_error("md_xstart_from_eps: md_set_schedule has not been called on this device"); return MD_ERR_ARG; }
    if (D % 4 != 0) { set_last_error("md_xstart_from_eps: D must be a multiple of 4"); return MD_ERR_ARG; }
    if ((int64_t)B * L == 0) return MD_OK;
    xstart_from_eps_kernel<<<ew_grid((int64_t)B * L * (D / 4), 256), 256, 0, stream>>>(x_t, eps, t, t_stride ? 1 : 0, out, B, L, D, vec_shift(D), sched_ref());
    return check_cuda(cudaGetLastError(), "xstart_from_eps launch");
}

extern "C" __attribute__((visibility("default"))) int md_q_sample_ld(const float* x0, const float* noise, uint64_t seed, uint64_t step_counter, int64_t seq_offset,
                           const int32_t* t, int t_stride, const int32_t* mask, int64_t mask_tok_stride,
                           int64_t mask_d_stride, float* out, void* out_bf16, int bf16_ld, int B, int L, int D, cudaStream_t stream) {
    if (t != nullptr && sched_state().T == 0) { set_last_error("md_q_sample: md_set_schedule has not been called on this device"); return MD_ERR_ARG; }
    if (D % 4 != 0) { set_last_error("md_q_sample: D must be a multiple of 4"); return MD_ERR_ARG; }
    if (bf16_ld < D || bf16_ld % 4 != 0) { set_last_error("md_q_sample: bf16_ld=%d must be a multiple of 4 >= D=%d", bf16_ld, D); return MD_ERR_ARG; }
    if ((int64_t)B * L == 0) return MD_OK;
    QSampleArgs a;
    a.x0 = x0; a.noise = noise; a.t = t; a.t_stride = t_stride ? 1 : 0; a.mask = mask; a.mask_tok_stride = mask_tok_stride; a.mask_d_stride = mask_d_stride;
    a.out = out; a.out_bf16 = reinterpret_cast<__nv_bfloat16*>(out_bf16); a.seq_offset = seq_offset; a.B = B; a.L = L; a.D = D;
    a.rng.init(seed, step_counter, 0.0f); a.sched_dev = sched_state().dev; a.T = sched_state().T; a.vshift = vec_shift(D);
    a.bf16_ld = bf16_ld;
    q_sample_kernel<<<ew_grid((int64_t)B * L * (D / 4), 256), 256, 0, stream>>>(a);
    return check_cuda(cudaGetLastError(), "q_sample launch");
}

extern "C" __attribute__((visibility("default"))) int md_q_sample(const float* x0, const float* noise, uint64_t seed, uint64_t step_counter, int64_t seq_offset,
                           const int32_t* t, int t_stride, const int32_t* mask, int64_t mask_tok_stride,
                           int64_t mask_d_stride, float* out, void* out_bf16, int B, int L, int D, cudaStream_t stream) {
    return md_q_sample_ld(x0, noise, seed, step_counter, seq_offset, t, t_stride, mask, mask_tok_stride, mask_d_stride, out, out_bf16,
                          D, B, L, D, stream);
}

extern "C" __attribute__((visibility("default"))) int md_fill_normal(float* out, int64_t n, uint64_t seed, uint64_t step_counter, int64_t elem_offset, float top_p,
                              cudaStream_t stream) {
    if (elem_offset % 4 != 0) { set_last_error("md_fill_normal: elem_offset must be a multiple of 4"); return MD_ERR_ARG; }
    if (n == 0) return MD_OK;
    NoiseGen g;
    g.init(seed, step_counter, top_p);
    fill_normal_kernel<<<ew_grid((n + 3) / 4, 256), 256, 0, stream>>>(out, n, elem_offset, g);
    return check_cuda(cudaGetLastError(), "fill_normal launch");
}
