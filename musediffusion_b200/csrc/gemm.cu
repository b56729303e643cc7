// Persistent warp-specialised tcgen05 GEMM for the denoiser's Linear layers (sm_100a).
//
//   out[M, N] = epilogue( A[M, K] (bf16, row-major)  x  W[N, K]^T (bf16, nn.Linear layout)  + bias[N] )
//
// Replaces every nn.Linear of TransformerNetModel.forward (reference MuseDiffusion/models/network.py:139-154 and
// the HF BertLayer linears called from network.py:151).  Both operands are K-major, so TMA (SWIZZLE_128B boxes of
// 64 bf16) feeds tcgen05.mma directly; fp32 accumulators live in TMEM (2 stages x BN columns) so the epilogue of
// tile i overlaps the MMAs of tile i+1.
//
// Roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM owner + single-thread MMA issuer,
// warps 2..9 = epilogue (TMEM -> registers -> bias / GELU / tanh / pos+time -> swizzled smem slab -> TMA store).
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <unordered_map>

#include "common.cuh"
#include "musediff_b200.h"

namespace md {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int UMMA_K = 16;
constexpr int kGemmThreads = 320;
constexpr int kEpiThreads = 256;

struct GemmArgs {
    int M, N, K;
    int L;                         // rows per sequence (EPI_POS_TIME)
    const float* bias;             // [N] or nullptr
    const float* pos;              // [L, N]   (MD_EPI_BIAS_POS_TIME)
    const float* temb;             // [M / L, N] (row stride temb_stride; 0 = one row shared by all sequences)
    int temb_stride;
    void* out;                     // bf16 or fp32 [M, store_cols]
    int store_cols;                // output columns kept (<= N; columns beyond are computed and dropped)
    int debug_skip;                // tuning experiments only: 1 = no TMA store, 2 = no slab write + no store
    int idle_wait;                 // bit 0: producer, bit 1: epilogue, bit 2: MMA warp wait with the try_wait suspend hint
};

template <int BN, bool kCta2 = false>
struct GemmCfg {
    static constexpr int kStages = (BN == 256 && !kCta2) ? 4 : 6;
    static constexpr int kABytes = BM * BK * 2;
    static constexpr int kBBytes = (kCta2 ? BN / 2 : BN) * BK * 2;   // a CTA pair splits the B tile: 128 W rows per CTA
    static constexpr int kStageBytes = kABytes + kBBytes;
    static constexpr int kTmemCols = 2 * BN;  // 512 or 256: power of two
    static constexpr int kSlabBytes = 32 * 128;                 // one epilogue warp's staging slab: 32 rows x 128 B
    static constexpr int kStagingBytes = 8 * kSlabBytes;
    static constexpr int kSmemBytes = 1024 /*align slack*/ + kStages * kStageBytes + kStagingBytes + 256 /*barriers*/;
};

template <int EPI>
MD_DEVINL float epi_act(float v) {
    if (EPI == MD_EPI_BIAS_GELU) return gelu_erf(v);
    if (EPI == MD_EPI_BIAS_TANH) return fast_tanh(v);
    return v;
}

// Epilogue data path: TMEM -> registers (thread = output row, 32 consecutive columns per tcgen05.ld) -> bias /
// activation -> 128B-swizzled shared-memory slab (32 rows x 128 B, one per epilogue warp) -> TMA store.  A direct
// st.global from the TMEM register layout would touch 32 different 128 B lines per warp instruction (one L1TEX
// wavefront each); the slab + cp.async.bulk.tensor store costs no LSU wavefronts and clips rows >= M / cols >= N.
// kCta2 = true: launched as clusters of two CTAs (cta_group::2).  A pair computes one 256 x 256 tile: each CTA keeps
// its own 128 A rows, its own accumulator rows (TMEM) and its own epilogue, but loads only half of the W rows — the
// UMMA reads operands from both CTAs' shared memory — which halves the per-SM shared-memory traffic of the B operand
// (the 1-CTA 128x256 mainloop needs 96 B/clk of operand reads + 96 B/clk of TMA fills against a 128 B/clk port).
template <int BN, int EPI, bool OUT_F32, bool kCta2>
MD_DEVINL void gemm_body(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const GemmArgs& p) {
    using Cfg = GemmCfg<BN, kCta2>;
    const uint32_t cta_rank = kCta2 ? cluster_ctarank() : 0u;
    const bool is_leader = (cta_rank == 0);
    const int cta_id = kCta2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;       // tile-scheduler id (pair id)
    const int n_cta = kCta2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    constexpr int BMT = kCta2 ? 2 * BM : BM;                                   // rows of one scheduled tile
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem;
    uint8_t* sB = smem + Cfg::kStages * Cfg::kABytes;
    uint8_t* sStage = smem + Cfg::kStages * Cfg::kStageBytes;          // 1024-aligned: kStageBytes is a multiple of 1024
    uint64_t* bars = reinterpret_cast<uint64_t*>(sStage + Cfg::kStagingBytes);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + Cfg::kStages;
    uint64_t* tfull_bar = bars + 2 * Cfg::kStages;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int n_tiles = (p.N + BN - 1) / BN;
    const int m_tiles = (p.M + BMT - 1) / BMT;
    const int num_tiles = n_tiles * m_tiles;
    const int num_kb = (p.K + BK - 1) / BK;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        tma_prefetch_desc(&tmC);
        for (int s = 0; s < Cfg::kStages; ++s) {
            mbar_init(&full_bar[s], kCta2 ? 2 : 1);          // pair: one arrival per CTA's producer (leader's barrier is used)
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(&tfull_bar[s], 1);
            mbar_init(&tempty_bar[s], kCta2 ? 2 * kEpiThreads : kEpiThreads);   // pair: both CTAs' epilogues release the leader
        }
        fence_barrier_init();
    }
    if (warp == 1) {
        if (kCta2) tmem_alloc_2cta<Cfg::kTmemCols>(tmem_slot);
        else tmem_alloc<Cfg::kTmemCols>(tmem_slot);
    }
    tc_fence_before();
    if (kCta2) cluster_sync_all(); else __syncthreads();     // barriers initialised in BOTH CTAs before any remote signal
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------ TMA producer (whole warp, elected issue)
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = cta_id; tile < num_tiles; tile += n_cta) {
            const int m_blk = tile / n_tiles, n_blk = tile % n_tiles;
            for (int kb = 0; kb < num_kb; ++kb) {
                if (p.idle_wait & 1) mbar_wait_idle(&empty_bar[stage], phase ^ 1); else mbar_wait(&empty_bar[stage], phase ^ 1);
                if (kCta2) {
                    // both CTAs credit the LEADER's full barrier: 2 arrivals + the bytes of all four boxes
                    if (is_leader) mbar_arrive_expect_tx_w(&full_bar[stage], 2 * Cfg::kStageBytes);
                    else mbar_arrive_remote_w(&full_bar[stage], 0);
                    tma_load_2d_2cta_w(sA + stage * Cfg::kABytes, &tmA, &full_bar[stage], kb * BK, m_blk * BMT + (int)cta_rank * BM);
                    tma_load_2d_2cta_w(sB + stage * Cfg::kBBytes, &tmB, &full_bar[stage], kb * BK, n_blk * BN + (int)cta_rank * (BN / 2));
                } else {
                    mbar_arrive_expect_tx_w(&full_bar[stage], Cfg::kStageBytes);
                    tma_load_2d_w(sA + stage * Cfg::kABytes, &tmA, &full_bar[stage], kb * BK, m_blk * BM);
                    tma_load_2d_w(sB + stage * Cfg::kBBytes, &tmB, &full_bar[stage], kb * BK, n_blk * BN);
                }
                if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------ MMA issuer (whole warp runs the loop, one elected lane issues)
        constexpr uint32_t idesc = make_idesc_bf16(BMT, BN);
        int stage = 0;
        uint32_t phase = 0;
        int acc = 0;
        uint32_t acc_phase = 0;
        if (is_leader) {        // in a pair only the leader CTA issues; its MMAs drive both tensor cores
            for (int tile = cta_id; tile < num_tiles; tile += n_cta) {
                if (p.idle_wait & 4) mbar_wait_idle(&tempty_bar[acc], acc_phase ^ 1); else mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * BN;
                for (int kb = 0; kb < num_kb; ++kb) {
                    if (p.idle_wait & 4) mbar_wait_idle(&full_bar[stage], phase); else mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint64_t a_desc = make_sdesc_sw128(smem_u32(sA + stage * Cfg::kABytes));
                    const uint64_t b_desc = make_sdesc_sw128(smem_u32(sB + stage * Cfg::kBBytes));
#pragma unroll
                    for (int k = 0; k < BK / UMMA_K; ++k) {
                        // +32 bytes per UMMA_K step inside the 128B swizzle atom  (encoded >> 4)
                        if (kCta2) umma_ss_2cta_w(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0);
                        else umma_ss_w(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0);
                    }
                    if (kCta2) tc_commit_2cta_w(&empty_bar[stage]); else tc_commit_w(&empty_bar[stage]);
                    if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
                }
                if (kCta2) tc_commit_2cta_w(&tfull_bar[acc]); else tc_commit_w(&tfull_bar[acc]);
                acc ^= 1;
                if (acc == 0) acc_phase ^= 1;
            }
        }
    } else {
        // ------------------------------------------------ epilogue (8 warps)
        const int ew = warp - 2;
        const int q = warp & 3;             // TMEM lane quadrant this warp may access
        const int hsel = ew >> 2;           // which half of the BN columns
        // Staging: each epilogue warp owns 4 KB.  bf16 output: two 2 KB half-slabs (32 rows x 64 B = 32 columns, 64B
        // swizzle) used alternately, so the TMA store of chunk c drains while chunk c+1 is produced
        // (cp.async.bulk.wait_group.read 1).  fp32 output (only the N = 128 projection): one 4 KB slab (32 rows x 128 B).
        uint8_t* slab = sStage + ew * Cfg::kSlabBytes;
        constexpr int kChunkCols = 32;
        constexpr int kChunks = (BN / 2) / kChunkCols;
        constexpr int kRowBytes = OUT_F32 ? 128 : 64;
        int acc = 0;
        uint32_t acc_phase = 0;
        uint32_t buf = 0;
        for (int tile = cta_id; tile < num_tiles; tile += n_cta) {
            const int m_blk = tile / n_tiles, n_blk = tile % n_tiles;
            const int n0 = n_blk * BN;
            if (p.idle_wait & 2) mbar_wait_idle(&tfull_bar[acc], acc_phase); else mbar_wait(&tfull_bar[acc], acc_phase);
            tc_fence_after();
            const int row0 = m_blk * BMT + (int)cta_rank * BM + q * 32;
            const int row = row0 + lane;
            int seq_b = 0, seq_l = 0;
            if (EPI == MD_EPI_BIAS_POS_TIME) {
                const int rr = row < p.M ? row : p.M - 1;
                seq_b = rr / p.L;
                seq_l = rr - seq_b * p.L;
            }
#pragma unroll 1
            for (int c = 0; c < kChunks; ++c) {
                const int col0 = hsel * (BN / 2) + c * kChunkCols;      // column inside the tile
                const int n = n0 + col0;
                if (n >= p.store_cols) break;                            // warp-uniform
                float v[kChunkCols];
                {
                    uint32_t r[32];
                    tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + col0, r);
                    tc_wait_ld();
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                }
                if (p.bias != nullptr) {
#pragma unroll
                    for (int g = 0; g < kChunkCols / 4; ++g) {
                        float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (n + g * 4 < p.N) b = __ldg(reinterpret_cast<const float4*>(p.bias + n + g * 4));
                        f2_unpack(f2_add(f2_pack(v[g * 4 + 0], v[g * 4 + 1]), f2_pack(b.x, b.y)), v[g * 4 + 0], v[g * 4 + 1]);   // FADD2
                        f2_unpack(f2_add(f2_pack(v[g * 4 + 2], v[g * 4 + 3]), f2_pack(b.z, b.w)), v[g * 4 + 2], v[g * 4 + 3]);
                    }
                }
                if (EPI == MD_EPI_BIAS_POS_TIME) {
#pragma unroll
                    for (int g = 0; g < kChunkCols / 4; ++g) {
                        if (n + g * 4 < p.N) {
                            const float4 a = *reinterpret_cast<const float4*>(p.pos + (size_t)seq_l * p.N + n + g * 4);
                            const float4 b = *reinterpret_cast<const float4*>(p.temb + (size_t)seq_b * p.temb_stride + n + g * 4);
                            v[g * 4 + 0] += a.x + b.x;
                            v[g * 4 + 1] += a.y + b.y;
                            v[g * 4 + 2] += a.z + b.z;
                            v[g * 4 + 3] += a.w + b.w;
                        }
                    }
                }
                if (EPI == MD_EPI_BIAS_GELU) {
#pragma unroll
                    for (int j = 0; j < kChunkCols; j += 2) f2_unpack(gelu_erf_x2(f2_pack(v[j], v[j + 1])), v[j], v[j + 1]);
                } else {
#pragma unroll
                    for (int j = 0; j < kChunkCols; ++j) v[j] = epi_act<EPI>(v[j]);
                }
                if (p.debug_skip == 2) continue;
                if (EPI == MD_EPI_BIAS_SPLIT) {
                    // out = bf16 [M, 2N] = [hi | lo], hi = bf16(v), lo = bf16(v - hi): the split-bf16 operand of the rounding
                    // contraction, emitted here so that the fp32 model output never makes an HBM round trip.  Two half-slab
                    // stores per chunk (columns n and N + n), the same double buffering as the plain bf16 path.
#pragma unroll
                    for (int part = 0; part < 2; ++part) {
                        uint8_t* dstp = slab + buf * 2048;
                        if (lane == 0) tma_store_wait_read<1>();
                        __syncwarp();
                        const uint32_t row_addr = smem_u32(dstp) + lane * 64;
#pragma unroll
                        for (int k = 0; k < 4; ++k) {
                            uint32_t w[4];
#pragma unroll
                            for (int e = 0; e < 4; ++e) {
                                const float a0 = v[k * 8 + 2 * e], a1 = v[k * 8 + 2 * e + 1];
                                const uint32_t hi = pack_bf16x2(a0, a1);
                                if (part == 0) w[e] = hi;
                                else { const float2 hf = unpack_bf16x2(hi); w[e] = pack_bf16x2(a0 - hf.x, a1 - hf.y); }
                            }
                            const uint32_t addr = row_addr + ((k ^ ((lane >> 1) & 3)) << 4);
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]) : "memory");
                        }
                        fence_proxy_async_smem();
                        __syncwarp();
                        if (lane == 0 && p.debug_skip == 0) {
                            tma_store_2d(&tmC, dstp, n + part * p.N, row0);
                            tma_store_commit();
                        }
                        buf ^= 1;
                    }
                    continue;
                }
                // the TMA store that last used this staging buffer must have finished READING shared memory
                uint8_t* dst = OUT_F32 ? slab : slab + buf * 2048;
                if (lane == 0) { if (OUT_F32) tma_store_wait_read<0>(); else tma_store_wait_read<1>(); }
                __syncwarp();
                const uint32_t row_addr = smem_u32(dst) + lane * kRowBytes;
                if (OUT_F32) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) {       // 8 x 16 B per 128 B row, 128B swizzle: chunk ^= row % 8
                        const uint32_t addr = row_addr + ((k ^ (lane & 7)) << 4);
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(__float_as_uint(v[k * 4 + 0])),
                                     "r"(__float_as_uint(v[k * 4 + 1])), "r"(__float_as_uint(v[k * 4 + 2])), "r"(__float_as_uint(v[k * 4 + 3]))
                                     : "memory");
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {       // 4 x 16 B per 64 B row, 64B swizzle: chunk ^= (row / 2) % 4
                        const uint32_t addr = row_addr + ((k ^ ((lane >> 1) & 3)) << 4);
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(pack_bf16x2(v[k * 8 + 0], v[k * 8 + 1])),
                                     "r"(pack_bf16x2(v[k * 8 + 2], v[k * 8 + 3])), "r"(pack_bf16x2(v[k * 8 + 4], v[k * 8 + 5])),
                                     "r"(pack_bf16x2(v[k * 8 + 6], v[k * 8 + 7]))
                                     : "memory");
                    }
                }
                fence_proxy_async_smem();           // generic-proxy writes -> visible to the async (TMA) proxy
                __syncwarp();
                if (lane == 0 && p.debug_skip == 0) {
                    tma_store_2d(&tmC, dst, n, row0);
                    tma_store_commit();
                }
                buf ^= 1;
            }
            tc_fence_before();
            if (kCta2 && !is_leader) mbar_arrive_remote(&tempty_bar[acc], 0);      // the MMA issuer lives in the leader CTA
            else mbar_arrive(&tempty_bar[acc]);
            acc ^= 1;
            if (acc == 0) acc_phase ^= 1;
        }
        if (lane == 0) tma_store_wait_read<0>();
        // global visibility of the bulk stores is guaranteed at kernel completion (stream order)
    }
    __syncwarp();
    tc_fence_before();
    if (kCta2) cluster_sync_all(); else __syncthreads();     // the peer may still read this CTA's smem / signal its barriers
    if (warp == 1) {
        if (kCta2) tmem_dealloc_2cta<Cfg::kTmemCols>(tmem_base);
        else tmem_dealloc<Cfg::kTmemCols>(tmem_base);
    }
}

template <int BN, int EPI, bool OUT_F32>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ CUtensorMap tmC, const GemmArgs p) {
    gemm_body<BN, EPI, OUT_F32, false>(tmA, tmB, tmC, p);
}

template <int EPI, bool OUT_F32>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmC, const GemmArgs p) {
    gemm_body<256, EPI, OUT_F32, true>(tmA, tmB, tmC, p);
}

// ----------------------------------------------------------------------------------------------
// host side
// ----------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (fn) return fn;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
        return nullptr;
    fn = reinterpret_cast<PFN_encodeTiled>(ptr);
    return fn;
}

// Encoded tensor maps are cached per (base pointer, geometry): the sampling loop re-issues the same ~250 (pointer, shape)
// pairs every step (fixed workspace, fixed weights), and cuTensorMapEncodeTiled costs more host time than a small-batch
// kernel takes to run.  Device pointers are unique across devices (UVA), so one process-wide table is per-device safe.
struct TmapKey {
    const void* base;
    uint64_t d[3], s[2];
    uint32_t box[2], kind;
    bool operator==(const TmapKey& o) const { return memcmp(this, &o, sizeof(TmapKey)) == 0; }
};
struct TmapKeyHash {
    size_t operator()(const TmapKey& k) const {
        const uint64_t* w = reinterpret_cast<const uint64_t*>(&k);
        uint64_t h = 0xcbf29ce484222325ull;
        for (size_t i = 0; i < sizeof(TmapKey) / 8; ++i) { h ^= w[i]; h *= 0x100000001b3ull; h ^= h >> 29; }
        return (size_t)h;
    }
};
static std::mutex g_tmap_mu;
static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> g_tmap_cache;
static bool tmap_lookup(const TmapKey& k, CUtensorMap* tm) {
    std::lock_guard<std::mutex> lock(g_tmap_mu);
    auto it = g_tmap_cache.find(k);
    if (it == g_tmap_cache.end()) return false;
    *tm = it->second;
    return true;
}
static void tmap_store(const TmapKey& k, const CUtensorMap& tm) {
    std::lock_guard<std::mutex> lock(g_tmap_mu);
    if (g_tmap_cache.size() > 16384) g_tmap_cache.clear();
    g_tmap_cache[k] = tm;
}

// 2-D row-major [rows, cols] tensor (bf16 or fp32), box = [box_rows, box_cols] with box_cols * elem = 128 B, 128B swizzle.
int make_tmap_2d(CUtensorMap* tm, const void* base, int is_f32, uint64_t rows, uint64_t cols, uint64_t row_stride_elems,
                 uint32_t box_rows, uint32_t box_cols) {
    const bool sw64 = (box_cols * (is_f32 ? 4u : 2u)) == 64u;      // 64-byte box rows use the 64B swizzle, else 128B
    TmapKey key;
    memset(&key, 0, sizeof(key));
    key.base = base; key.d[0] = cols; key.d[1] = rows; key.s[0] = row_stride_elems; key.box[0] = box_cols; key.box[1] = box_rows;
    key.kind = is_f32 ? 1u : 0u;
    if (tmap_lookup(key, tm)) return MD_OK;
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) { set_last_error("cuTensorMapEncodeTiled entry point not available"); return MD_ERR_CUDA; }
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {row_stride_elems * (is_f32 ? 4 : 2)};
    cuuint32_t box[2] = {box_cols, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(tm, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, sw64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled failed: CUresult %d (rows=%llu cols=%llu stride=%llu box=%ux%u base=%p)", (int)r,
                       (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)row_stride_elems, box_rows,
                       box_cols, base);
        return MD_ERR_CUDA;
    }
    tmap_store(key, *tm);
    return MD_OK;
}

// 3-D bf16 tensor [d2][d1][d0] (d0 contiguous), box = [1, box1, box0], 128B swizzle; rows beyond d1 read as zero.
int make_tmap_bf16_3d(CUtensorMap* tm, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t stride1_elems,
                      uint64_t stride2_elems, uint32_t box0, uint32_t box1) {
    TmapKey key;
    memset(&key, 0, sizeof(key));
    key.base = base; key.d[0] = d0; key.d[1] = d1; key.d[2] = d2; key.s[0] = stride1_elems; key.s[1] = stride2_elems;
    key.box[0] = box0; key.box[1] = box1; key.kind = 2u;
    if (tmap_lookup(key, tm)) return MD_OK;
    PFN_encodeTiled fn = get_encode_fn();
    if (!fn) { set_last_error("cuTensorMapEncodeTiled entry point not available"); return MD_ERR_CUDA; }
    cuuint64_t gdim[3] = {d0, d1, d2};
    cuuint64_t gstr[2] = {stride1_elems * 2, stride2_elems * 2};
    cuuint32_t box[3] = {box0, box1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error("cuTensorMapEncodeTiled(3d) failed: CUresult %d (dims=%llu,%llu,%llu base=%p)", (int)r,
                       (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2, base);
        return MD_ERR_CUDA;
    }
    tmap_store(key, *tm);
    return MD_OK;
}

int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}
int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0) dev = 0;
    return dev < kMaxDevices ? dev : kMaxDevices - 1;
}
static int g_num_sms[kMaxDevices] = {0};
int num_sms() {
    const int dev = current_device();
    if (g_num_sms[dev] == 0) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        n = n > 0 ? n : 148;
        static const int cap = env_int("MD_NUM_SMS", 0);     // tuning tools only (tools/clock_timeline.py leaves one SM to its probe)
        if (cap > 0 && cap < n) n = cap;
        g_num_sms[dev] = n;
    }
    return g_num_sms[dev];
}

template <int BN, int EPI, bool OUT_F32>
static int launch_gemm(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const GemmArgs& args,
                       cudaStream_t stream) {
    using Cfg = GemmCfg<BN>;
    auto kern = gemm_kernel<BN, EPI, OUT_F32>;
    static bool attr_set[kMaxDevices] = {false};
    if (ensure_dyn_smem(kern, Cfg::kSmemBytes, attr_set, "cudaFuncSetAttribute(gemm)")) return MD_ERR_CUDA;
    const int n_tiles = (args.N + BN - 1) / BN, m_tiles = (args.M + BM - 1) / BM;
    const int grid = min(n_tiles * m_tiles, num_sms());
    kern<<<grid, kGemmThreads, Cfg::kSmemBytes, stream>>>(tmA, tmB, tmC, args);
    return check_cuda(cudaGetLastError(), "gemm launch");
}

template <int EPI, bool OUT_F32>
static int launch_gemm_pair(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const GemmArgs& args,
                            cudaStream_t stream) {
    using Cfg = GemmCfg<256, true>;
    auto kern = gemm_pair_kernel<EPI, OUT_F32>;
    static bool attr_set[kMaxDevices] = {false};
    if (ensure_dyn_smem(kern, Cfg::kSmemBytes, attr_set, "cudaFuncSetAttribute(gemm pair)")) return MD_ERR_CUDA;
    const int n_tiles = (args.N + 255) / 256, m_tiles = (args.M + 255) / 256;
    int pairs = num_sms() / 2;
    if (n_tiles * m_tiles < pairs) pairs = n_tiles * m_tiles;
    kern<<<2 * pairs, kGemmThreads, Cfg::kSmemBytes, stream>>>(tmA, tmB, tmC, args);      // __cluster_dims__(2,1,1)
    return check_cuda(cudaGetLastError(), "gemm pair launch");
}

template <bool OUT_F32>
static int dispatch_epi_pair(int epi, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const GemmArgs& a,
                             cudaStream_t s) {
    switch (epi) {
        case MD_EPI_BIAS: return launch_gemm_pair<MD_EPI_BIAS, OUT_F32>(tmA, tmB, tmC, a, s);
        case MD_EPI_BIAS_GELU: return launch_gemm_pair<MD_EPI_BIAS_GELU, OUT_F32>(tmA, tmB, tmC, a, s);
        case MD_EPI_BIAS_TANH: return launch_gemm_pair<MD_EPI_BIAS_TANH, OUT_F32>(tmA, tmB, tmC, a, s);
        case MD_EPI_BIAS_POS_TIME: return launch_gemm_pair<MD_EPI_BIAS_POS_TIME, OUT_F32>(tmA, tmB, tmC, a, s);
    }
    set_last_error("md_linear_bf16: unknown epilogue %d", epi);
    return MD_ERR_ARG;
}

template <int BN, bool OUT_F32>
static int dispatch_epi(int epi, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmC, const GemmArgs& a,
                        cudaStream_t s) {
    switch (epi) {
        case MD_EPI_BIAS: return launch_gemm<BN, MD_EPI_BIAS, OUT_F32>(tmA, tmB, tmC, a, s);
        case MD_EPI_BIAS_GELU: return launch_gemm<BN, MD_EPI_BIAS_GELU, OUT_F32>(tmA, tmB, tmC, a, s);
        case MD_EPI_BIAS_TANH: return launch_gemm<BN, MD_EPI_BIAS_TANH, OUT_F32>(tmA, tmB, tmC, a, s);
        case MD_EPI_BIAS_POS_TIME: return launch_gemm<BN, MD_EPI_BIAS_POS_TIME, OUT_F32>(tmA, tmB, tmC, a, s);
        case MD_EPI_BIAS_SPLIT: return launch_gemm<BN, MD_EPI_BIAS_SPLIT, false>(tmA, tmB, tmC, a, s);
    }
    set_last_error("md_linear_bf16: unknown epilogue %d", epi);
    return MD_ERR_ARG;
}

}  // namespace md

using namespace md;

extern "C" __attribute__((visibility("default"))) int md_linear_bf16_cols(const void* A, const void* W, const float* bias, void* out, int M, int N, int K,
                                                                        int out_cols, int epilogue, int out_is_f32, const float* pos,
                                                                        const float* temb, int temb_stride, int L, cudaStream_t stream) {
    if (M <= 0 || N <= 0 || K <= 0) { set_last_error("md_linear_bf16: empty problem M=%d N=%d K=%d", M, N, K); return MD_ERR_ARG; }
    if (K % 8 != 0 || N % 8 != 0) { set_last_error("md_linear_bf16: K and N must be multiples of 8 (K=%d N=%d)", K, N); return MD_ERR_ARG; }
    // the output's row stride (out_cols elements) must be a multiple of 16 bytes for the TMA store
    if (out_cols <= 0 || out_cols > N || out_cols % (out_is_f32 ? 4 : 8) != 0) {
        set_last_error("md_linear_bf16: out_cols=%d must be <= N=%d and a multiple of %d", out_cols, N, out_is_f32 ? 4 : 8);
        return MD_ERR_ARG;
    }
    if (epilogue == MD_EPI_BIAS_POS_TIME && (pos == nullptr || temb == nullptr || L <= 0 || M % L != 0)) {
        set_last_error("md_linear_bf16: pos/time epilogue needs pos, temb and L dividing M");
        return MD_ERR_ARG;
    }
    const int BN = (N % 256 == 0 || N > 512) ? 256 : 128;
    // CTA pairs (cta_group::2) for the large regular shapes; MD_GEMM_PAIR=0 forces the single-CTA kernel
    static const int use_pair = env_int("MD_GEMM_PAIR", 1);
    const bool split = (epilogue == MD_EPI_BIAS_SPLIT);
    if (split && out_is_f32) { set_last_error("md_linear_bf16: the split epilogue writes bf16 [M, 2N]"); return MD_ERR_ARG; }
    if (split && out_cols != N) { set_last_error("md_linear_bf16: the split epilogue stores all N columns"); return MD_ERR_ARG; }
    const bool pair = use_pair && N % 256 == 0 && M >= 1024 && !out_is_f32 && !split;
    CUtensorMap tmA, tmB, tmC;
    if (int e = make_tmap_2d(&tmA, A, 0, M, K, K, BM, BK)) return e;
    if (int e = make_tmap_2d(&tmB, W, 0, N, K, K, pair ? 128 : BN, BK)) return e;
    // a tile column beyond out_cols is clipped by the TMA store
    if (int e = make_tmap_2d(&tmC, out, out_is_f32, M, split ? 2 * N : out_cols, split ? 2 * N : out_cols, 32, 32)) return e;
    GemmArgs a;
    a.M = M; a.N = N; a.K = K; a.L = L > 0 ? L : 1;
    a.bias = bias; a.pos = pos; a.temb = temb; a.temb_stride = temb_stride; a.out = out; a.store_cols = out_cols;
    static const int debug_skip = env_int("MD_GEMM_DEBUG_SKIP", 0), idle_env = env_int("MD_GEMM_IDLE", -1);
    a.debug_skip = debug_skip;
    // sleeping waits (try_wait suspend hint) for the warps that wait long: the TMA producer always, the epilogue warps when the
    // mainloop is long (K >= 2048: FFN2 +2..5 %); the epilogue-bound K = 768 shapes keep the polling wait (measured -1 % asleep)
    a.idle_wait = idle_env >= 0 ? idle_env : (K >= 2048 ? 3 : 1);
    if (pair) return dispatch_epi_pair<false>(epilogue, tmA, tmB, tmC, a, stream);
    if (BN == 256) return out_is_f32 ? dispatch_epi<256, true>(epilogue, tmA, tmB, tmC, a, stream)
                                     : dispatch_epi<256, false>(epilogue, tmA, tmB, tmC, a, stream);
    return out_is_f32 ? dispatch_epi<128, true>(epilogue, tmA, tmB, tmC, a, stream)
                      : dispatch_epi<128, false>(epilogue, tmA, tmB, tmC, a, stream);
}

extern "C" __attribute__((visibility("default"))) int md_linear_bf16(const void* A, const void* W, const float* bias, void* out, int M, int N, int K, int epilogue,
                              int out_is_f32, const float* pos, const float* temb, int temb_stride, int L,
                              cudaStream_t stream) {
    return md_linear_bf16_cols(A, W, bias, out, M, N, K, N, epilogue, out_is_f32, pos, temb, temb_stride, L, stream);
}
