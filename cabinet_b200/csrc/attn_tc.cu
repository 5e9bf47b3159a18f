// Fused global-context attention on tcgen05 (reference: src/models/cab.py:149-153):
//     ctx = softmax(Q K^T / sqrt(dk)) V       per image, query / key width dk, value width dv, L tokens
// (CABiNet: dk = dv = 128, L = H/32 * W/32 = 1024 ... 8160; a standalone ContextAggregationBlock(C, V): dk = C/2, dv = V)
// The L x L score matrix never exists in memory: one CTA owns 128 queries of one image and streams the keys in
// blocks of 128.  Two passes over the keys (QK^T is recomputed; the tensor work here is negligible):
//   pass A  S = Q K_j^T (TMEM) -> row max m (registers; no exponentials)
//   pass B  S = Q K_j^T (TMEM) -> P = exp2(S*c - m) <= 1, unnormalised (bf16, written in the K-major SWIZZLE_128B UMMA
//           layout to shared memory; row sum l of the rounded values) -> O += P V_j (TMEM accumulator over all key
//           blocks) -> ctx rows = O / l (bf16)
// so no accumulator rescaling is needed.  V must be K-major (keys contiguous) for the P V product, hence the tiny
// transpose pre-kernel v [L][dv] -> vt [dv][ceil8(L)].
// Warp roles (192 threads): warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer, warps 2-5 softmax / epilogue
// (thread = query row).  TMEM: S double-buffered (2 x 128 columns) + O (dv columns).
// Instantiated for dk in {64, 128, 256} x dv in {64, 128}; dk <= 128 double-buffers the K / Vt stages, dk = 256 runs one
// stage (the P V product of a key block is then issued before the next block's S, which reuses the stage).
#include "tc_common.cuh"

namespace {

constexpr int BQ = 128, BKEY = 128;
constexpr int TILE_BYTES = 128 * 128;  // one [128 rows x 64 elements] bf16 swizzled tile
constexpr int NUM_THREADS = 192;

// Query / key width DK, value / output width DV.  smem: Q (DK/64 tiles) | NST stages x { K (DK/64 tiles) | Vt (2 tiles of
// DV rows x 64 keys) } | P (2 tiles).  Two stages wherever they fit; at DK = 256 one stage (Q 64 KB + 2 x 96 KB + P
// 32 KB would exceed the 227 KB of shared memory).
template <int DK, int DV>
struct AttnCfg {
    static constexpr int KT = DK / 64;                   // 64-element K tiles of Q and K
    static constexpr int VT_TILE = DV * 128;             // one [DV rows x 64 keys] swizzled tile of Vt
    static constexpr int STAGE = KT * TILE_BYTES + 2 * VT_TILE;
    static constexpr int NST = DK >= 256 ? 1 : 2;
    static constexpr int SMEM = KT * TILE_BYTES + NST * STAGE + 2 * TILE_BYTES + 1024;
    static_assert(SMEM <= 227 * 1024, "attention_tc: shared memory");
    static_assert(256 + DV <= 512, "attention_tc: TMEM");
};

struct AttnParams {
    int L, nkb;
    float c;  // scale * log2(e)
    bf16* ctx;
    long long ldc;
};

template <int DK, int DV>
__global__ void __launch_bounds__(NUM_THREADS, 1)
attn_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
               const __grid_constant__ CUtensorMap tmVt, const AttnParams p) {
    using Cfg = AttnCfg<DK, DV>;
    constexpr int KT = Cfg::KT, NST = Cfg::NST, STAGE = Cfg::STAGE, VT_TILE = Cfg::VT_TILE;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t q_full, kv_full[NST], kv_empty[NST], s_full[2], s_empty[2], p_full, p_empty, o_full;
    __shared__ uint32_t tmem_base_smem;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sQ = smem;
    uint8_t* sKV = sQ + KT * TILE_BYTES;   // stage s: K at +s*STAGE, Vt at +s*STAGE + KT*TILE
    uint8_t* sP = sKV + NST * STAGE;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q0 = blockIdx.x * BQ, img = blockIdx.y;
    const int nkb = p.nkb, T = 2 * nkb;

    if (threadIdx.x == 0) {
        tc::prefetch_tmap(&tmQ);
        tc::prefetch_tmap(&tmK);
        tc::prefetch_tmap(&tmVt);
        tc::mbar_init(&q_full, 1);
        for (int s = 0; s < NST; ++s) {
            tc::mbar_init(&kv_full[s], 1);
            tc::mbar_init(&kv_empty[s], 1);
        }
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&s_full[s], 1);
            tc::mbar_init(&s_empty[s], 4);
        }
        tc::mbar_init(&p_full, 4);
        tc::mbar_init(&p_empty, 1);
        tc::mbar_init(&o_full, 1);
        tc::mbar_fence_init();
        tc::fence_proxy_async();
    }
    if (warp == 1) tc::tmem_alloc(&tmem_base_smem, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_base_smem;
    const uint32_t tmem_o = tmem + 256;

    if (warp == 0) {
        if (lane == 0) {
            // ================= TMA producer =================
            tc::mbar_expect_tx(&q_full, KT * TILE_BYTES);
#pragma unroll
            for (int kb = 0; kb < KT; ++kb) tc::tma_load_3d(sQ + kb * TILE_BYTES, &tmQ, &q_full, 64 * kb, q0, img);
            for (int t = 0; t < T; ++t) {
                const int s = t % NST;
                const uint32_t ph = (t / NST) & 1;
                const int j = t < nkb ? t : t - nkb;
                const bool pass_b = t >= nkb;
                uint8_t* stage = sKV + s * STAGE;
                tc::mbar_wait(&kv_empty[s], ph ^ 1);
                tc::mbar_expect_tx(&kv_full[s], KT * TILE_BYTES + (pass_b ? 2 * VT_TILE : 0));
#pragma unroll
                for (int kb = 0; kb < KT; ++kb)
                    tc::tma_load_3d(stage + kb * TILE_BYTES, &tmK, &kv_full[s], 64 * kb, j * BKEY, img);
                if (pass_b) {
                    tc::tma_load_3d(stage + KT * TILE_BYTES, &tmVt, &kv_full[s], j * BKEY, 0, img);
                    tc::tma_load_3d(stage + KT * TILE_BYTES + VT_TILE, &tmVt, &kv_full[s], j * BKEY + 64, 0, img);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer: warp-uniform control flow, one elected lane issues =================
        const uint32_t leader = tc::elect_one();
        const uint32_t idesc_s = tc::make_idesc_bf16(128, BKEY), idesc_o = tc::make_idesc_bf16(128, DV);
        const uint64_t q_desc = tc::make_desc_sw128(tc::smem_u32(sQ)), p_desc = tc::make_desc_sw128(tc::smem_u32(sP));
        const uint64_t kv_desc0 = tc::make_desc_sw128(tc::smem_u32(sKV));
        constexpr uint32_t TILE16 = TILE_BYTES >> 4, VT16 = VT_TILE >> 4, STAGE16 = STAGE >> 4;
        tc::mbar_wait(&q_full, 0);
        auto issue_pv = [&](int t) {  // O += P_t * V_t   (t is a pass-B index)
            const int kidx = t - nkb;
            const uint64_t v_desc = kv_desc0 + static_cast<uint64_t>((t % NST) * STAGE16 + KT * TILE16);
            tc::mbar_wait(&p_full, kidx & 1);
            tc::tc_fence_after();
#pragma unroll
            for (int kb = 0; kb < 2; ++kb)
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    tc::umma_bf16_if(leader, tmem_o, p_desc + (kb * TILE16 + 2 * k), v_desc + (kb * VT16 + 2 * k), idesc_o,
                                     (kidx | kb | k) != 0 ? 1u : 0u);
            tc::umma_commit_if(leader, &p_empty);
            tc::umma_commit_if(leader, &kv_empty[t % NST]);
        };
        for (int t = 0; t < T; ++t) {
            const int s = t % NST, sb = t & 1;
            // one stage: the previous block's P V must release the stage before the next K / Vt can land in it
            if (NST == 1 && t > nkb) issue_pv(t - 1);
            tc::mbar_wait(&kv_full[s], (t / NST) & 1);
            tc::mbar_wait(&s_empty[sb], ((t >> 1) & 1) ^ 1);
            tc::tc_fence_after();
            const uint64_t k_desc = kv_desc0 + static_cast<uint64_t>(s * STAGE16);
#pragma unroll
            for (int kb = 0; kb < KT; ++kb)
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    tc::umma_bf16_if(leader, tmem + sb * 128, q_desc + (kb * TILE16 + 2 * k), k_desc + (kb * TILE16 + 2 * k),
                                     idesc_s, (kb | k) ? 1u : 0u);
            tc::umma_commit_if(leader, &s_full[sb]);
            if (t < nkb) tc::umma_commit_if(leader, &kv_empty[s]);  // pass A: K block is free once S is computed
            else if (NST > 1 && t > nkb) issue_pv(t - 1);            // pass B: P V of the previous block, lagging one S
        }
        issue_pv(T - 1);
        tc::umma_commit_if(leader, &o_full);
        __syncwarp();
    } else {
        // ================= softmax / epilogue: thread = query row =================
        const int qd = warp & 3;
        const int row = qd * 32 + lane;
        const uint32_t lane_addr = static_cast<uint32_t>(qd * 32) << 16;
        const float c = p.c;
        // ---- pass A: row max only (c > 0, so the scale is applied to the maximum).  No exponentials here: pass B
        // writes UNNORMALISED probabilities exp2(s*c - m) <= 1, accumulates their row sum, and the output rows are
        // scaled by 1 / l at the end.
        float mraw = -INFINITY;
        for (int t = 0; t < nkb; ++t) {
            const int s = t & 1;
            tc::mbar_wait(&s_full[s], (t >> 1) & 1);
            tc::tc_fence_after();
            const uint32_t ta = tmem + s * 128 + lane_addr;
            const int nvalid = min(BKEY, p.L - t * BKEY);  // only the last key block can be partial
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
                uint32_t r[32];
                tc::tmem_ld32(ta + ch * 32, r);
                tc::tmem_ld_wait();
                if (nvalid == BKEY) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) mraw = fmaxf(mraw, __uint_as_float(r[i]));
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (ch * 32 + i < nvalid) mraw = fmaxf(mraw, __uint_as_float(r[i]));
                }
            }
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&s_empty[s]);
        }
        const float m = mraw * c;
        float l = 0.f;
        // ---- pass B: probabilities -> smem (UMMA A operand), one MUFU.EX2 per element
        for (int t = nkb; t < T; ++t) {
            const int s = t & 1;
            const int kidx = t - nkb;
            tc::mbar_wait(&s_full[s], (t >> 1) & 1);
            tc::tc_fence_after();
            tc::mbar_wait(&p_empty, (kidx & 1) ^ 1);
            const uint32_t ta = tmem + s * 128 + lane_addr;
            const int nvalid = min(BKEY, p.L - kidx * BKEY);
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) {
                uint32_t r[32];
                tc::tmem_ld32(ta + ch * 32, r);
                tc::tmem_ld_wait();
                float pv[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    float e;
                    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(fmaf(__uint_as_float(r[i]), c, -m)));
                    pv[i] = e;
                }
                if (nvalid != BKEY) {
#pragma unroll
                    for (int i = 0; i < 32; ++i)
                        if (ch * 32 + i >= nvalid) pv[i] = 0.f;
                }
#pragma unroll
                for (int g = 0; g < 4; ++g) {  // 4 chunks of 8 keys = 16 bytes each
                    Vec16<bf16> o;
                    o.pack(pv + 8 * g);
                    // the row sum is taken over the ROUNDED probabilities the tensor core will multiply with
                    float pr[8];
                    o.unpack(pr);
#pragma unroll
                    for (int i = 0; i < 8; ++i) l += pr[i];
                    const int cidx = ch * 4 + g;  // 16-byte chunk index along the 128 keys
                    tc::sts128(tc::smem_u32(sP) + (cidx >> 3) * TILE_BYTES + row * 128 + (((cidx & 7) ^ (row & 7)) << 4), o.raw);
                }
            }
            tc::fence_proxy_async();
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                tc::mbar_arrive(&p_full);
                tc::mbar_arrive(&s_empty[s]);
            }
        }
        const float inv_l = 1.f / l;
        // ---- output rows
        tc::mbar_wait(&o_full, 0);
        tc::tc_fence_after();
        const int qrow = q0 + row;
        bf16* out = p.ctx + (static_cast<long long>(img) * p.L + qrow) * p.ldc;
#pragma unroll
        for (int ch = 0; ch < DV / 32; ++ch) {
            uint32_t r[32];
            tc::tmem_ld32(tmem_o + lane_addr + ch * 32, r);
            tc::tmem_ld_wait();
            if (qrow < p.L) {
#pragma unroll
                for (int g = 0; g < 4; ++g) {
                    float f[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(r[8 * g + i]) * inv_l;
                    Vec16<bf16> o;
                    o.pack(f);
                    o.store(out + ch * 32 + g * 8);
                }
            }
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, 512);
    }
}

// v [N][L][dv] (pixel stride ldv) -> vt [N][dv][Lp], zero padded keys L..Lp-1
__global__ void __launch_bounds__(256)
transpose_v_kernel(const bf16* __restrict__ v, long long ldv, bf16* __restrict__ vt, int L, int Lp, int dv) {
    __shared__ bf16 tile[32][33];
    const int n = blockIdx.z;
    const int k0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
    const int tx = threadIdx.x % 32, ty = threadIdx.x / 32;
    for (int i = ty; i < 32; i += 8) {
        const int key = k0 + i;
        tile[i][tx] = key < L ? v[(static_cast<long long>(n) * L + key) * ldv + d0 + tx] : __float2bfloat16(0.f);
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int key = k0 + tx;
        if (key < Lp) vt[(static_cast<long long>(n) * dv + d0 + i) * Lp + key] = tile[tx][i];
    }
}

template <int DK, int DV>
int launch_attention(const CUtensorMap& tmQ, const CUtensorMap& tmK, const CUtensorMap& tmVt, const AttnParams& p, int N,
                     cudaStream_t s) {
    constexpr int SMEM = AttnCfg<DK, DV>::SMEM;
    static bool attr_done = false;
    if (!attr_done) {
        CAB_CUDA(cudaFuncSetAttribute(attn_tc_kernel<DK, DV>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
        attr_done = true;
    }
    dim3 grid((p.L + BQ - 1) / BQ, N);
    attn_tc_kernel<DK, DV><<<grid, NUM_THREADS, SMEM, s>>>(tmQ, tmK, tmVt, p);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

int attention_tc(const void* q, long long ldq, const void* k, long long ldk, const void* v, long long ldv,
                 void* vt_workspace, void* ctx, long long ldc, int N, int L, int dk, int dv, float scale,
                 cabinet_stream_t stream) {
    CAB_REQUIRE(q && k && v && vt_workspace && ctx, "attention_tc: null pointer");
    CAB_REQUIRE((dk == 64 || dk == 128 || dk == 256) && (dv == 64 || dv == 128),
                "attention_tc: key width must be 64, 128 or 256 and value width 64 or 128 (got %d, %d)", dk, dv);
    CAB_REQUIRE(N >= 0 && L > 0 && N <= 65535, "attention_tc: bad sizes");
    CAB_REQUIRE(ldq % 8 == 0 && ldk % 8 == 0 && ldc % 8 == 0 && ldq >= dk && ldk >= dk && ldv >= dv && ldc >= dv &&
                    (reinterpret_cast<uintptr_t>(q) & 15) == 0 && (reinterpret_cast<uintptr_t>(k) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(ctx) & 15) == 0 && (reinterpret_cast<uintptr_t>(vt_workspace) & 15) == 0,
                "attention_tc: 16-byte aligned rows required");
    if (N == 0) return CABINET_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int Lp = (L + 7) / 8 * 8;
    {
        dim3 grid((Lp + 31) / 32, dv / 32, N);
        transpose_v_kernel<<<grid, 256, 0, s>>>(reinterpret_cast<const bf16*>(v), ldv, reinterpret_cast<bf16*>(vt_workspace),
                                                L, Lp, dv);
        CAB_LAUNCH_CHECK();
    }
    CUtensorMap tmQ, tmK, tmVt;
    {
        const uint32_t box[3] = {64, 128, 1};
        const uint64_t dims[3] = {(uint64_t)dk, (uint64_t)L, (uint64_t)N};
        const uint64_t sq[2] = {(uint64_t)ldq * 2, (uint64_t)ldq * 2 * L};
        const uint64_t sk[2] = {(uint64_t)ldk * 2, (uint64_t)ldk * 2 * L};
        int rc = cab_make_tmap_bf16(&tmQ, q, 3, dims, sq, box);
        if (rc) return rc;
        rc = cab_make_tmap_bf16(&tmK, k, 3, dims, sk, box);
        if (rc) return rc;
        const uint32_t vbox[3] = {64, (uint32_t)dv, 1};
        const uint64_t dvt[3] = {(uint64_t)Lp, (uint64_t)dv, (uint64_t)N};
        const uint64_t sv[2] = {(uint64_t)Lp * 2, (uint64_t)Lp * 2 * dv};
        rc = cab_make_tmap_bf16(&tmVt, vt_workspace, 3, dvt, sv, vbox);
        if (rc) return rc;
    }
    AttnParams p;
    p.L = L;
    p.nkb = (L + BKEY - 1) / BKEY;
    p.c = scale * 1.4426950408889634f;
    p.ctx = reinterpret_cast<bf16*>(ctx);
    p.ldc = ldc;
    switch (dk * 1000 + dv) {
        case 64064: return launch_attention<64, 64>(tmQ, tmK, tmVt, p, N, s);
        case 64128: return launch_attention<64, 128>(tmQ, tmK, tmVt, p, N, s);
        case 128064: return launch_attention<128, 64>(tmQ, tmK, tmVt, p, N, s);
        case 128128: return launch_attention<128, 128>(tmQ, tmK, tmVt, p, N, s);
        case 256064: return launch_attention<256, 64>(tmQ, tmK, tmVt, p, N, s);
        default: return launch_attention<256, 128>(tmQ, tmK, tmVt, p, N, s);
    }
}

}  // namespace

extern "C" int cabinet_attention_tc(const void* q, long long ldq, const void* k, long long ldk, const void* v,
                                    long long ldv, void* vt_workspace, void* ctx, long long ldc, int N, int L, int d,
                                    float scale, cabinet_stream_t stream) {
    CAB_REQUIRE(d == 128, "attention_tc: head dim must be 128 (got %d)", d);
    return attention_tc(q, ldq, k, ldk, v, ldv, vt_workspace, ctx, ldc, N, L, 128, 128, scale, stream);
}

extern "C" int cabinet_attention_tc_dkdv(const void* q, long long ldq, const void* k, long long ldk, const void* v,
                                         long long ldv, void* vt_workspace, void* ctx, long long ldc, int N, int L, int dk,
                                         int dv, float scale, cabinet_stream_t stream) {
    return attention_tc(q, ldq, k, ldk, v, ldv, vt_workspace, ctx, ldc, N, L, dk, dv, scale, stream);
}
