// Fused network stems, second formulation: NO im2col.  Same contract as stem_tc.cu -- both convolutions that read the
// fp32 NCHW input image
//   sb.conv1      7x7 s2 p3, 3 -> 64, BN, ReLU       (src/models/cabinet.py:111, 19-44)
//   mobile stem   3x3 s2 p1, 3 -> 16, BN, HardSwish  (src/models/mobilenetv3.py:86-91,173)
// as ONE GEMM D[128 px x 80] = A[128 x 224] * W[80 x 224]^T (the 3x3 filter sits in the centre of a 7x7 one) -- but the
// A operand is never built.  stem_tc.cu spends its time writing a 48 KB im2col tile per 128 pixels (it is bound by
// shared-memory bandwidth, 0.55 of the HBM roofline).  Here the converter warps only turn the fp32 NCHW window into a
// pixel-interleaved bf16 copy, 4 channels (r, g, b, 1.0) = 8 bytes per pixel, and the tensor core reads the im2col
// view straight out of it through the shared-memory matrix descriptor:
//
//   tap row ky, output pixel (oy, ox) of a 16 x 8 patch:  A[m = oy*8 + ox][k = kx*4 + c] = copy[2 oy + ky][2 ox + kx][c]
//   = byte (2 oy + ky) * PITCH + 16 ox + 2 k of the copy: consecutive A rows are 16 bytes apart and OVERLAP (a stride-2
//   conv over 8-byte pixels).  That is exactly the no-swizzle K-major UMMA layout (core matrix = 8 rows x 16 bytes, rows
//   16 bytes apart) with LBO = 16 (next 8 k: the same rows shifted by two pixels) and SBO = 2 PITCH (next oy).
//
// K = 7 tap rows x (8 pixels x 4 channels): 14 MMAs of M128 N80 K16 per tile; the pixel at kx = 0 and the channel c = 3
// have zero weights, except that the bias rides on the constant-1 channel of the centre pixel (bf16 hi + lo parts).
// Shared-memory traffic per 128 pixels drops from ~230 KB to ~110 KB; the kernel becomes output-write (HBM) bound.
//
// Persistent, warp specialised like stem_tc.cu: warp 0 TMA producer (weights once by one bulk copy; per tile one 3-D
// fp32 box {24 cols, 37 rows, 3 ch}), warp 1 MMA issuer, warps 2-9 converters, warps 10-13 epilogue (two TMA stores).
#include "tc_common.cuh"

namespace {

constexpr int TH = 16, TW = 8;               // output patch = 128 pixels, m = oy * 8 + ox
constexpr int WIN_H = 37, WIN_W = 24;        // input window rows / cols
constexpr int WIN_BYTES = 3 * WIN_H * WIN_W * 4;     // 10656
constexpr int WIN_STRIDE = 10752;
constexpr int WIN_STAGES = 3;
constexpr int PITCH = WIN_W * 8;             // bytes per row of the bf16 x 4 copy (192)
constexpr int WINB_BYTES = WIN_H * PITCH;    // 7104
constexpr int WINB_STRIDE = 7168;
constexpr int WINB_STAGES = 3;
constexpr int NMMA = 14;                     // 7 tap rows x 2 K halves
// NOUT = 80: sb.conv1 (64) + the backbone stem (16), CABiNet's fused stems; NOUT = 64: sb.conv1 alone
template <int NOUT>
struct Stem2Shape {
    static constexpr int W_MMA_BYTES = 2 * (NOUT / 8) * 128;  // one [NOUT x 16] bf16 operand (80: 2 x 10 core matrices)
    static constexpr int W_BYTES = NMMA * W_MMA_BYTES;        // 80: 35840 (<= the 36 KB reserved), 64: 28672
    static constexpr int ACC_COLS = NOUT > 64 ? 128 : 64;     // TMEM columns per accumulator stage (a power of 2)
};
constexpr int ACC_STAGES = 2;
constexpr int CONV_WARPS = 8, CONV_THREADS = 32 * CONV_WARPS;
constexpr int EPI_WARP0 = 2 + CONV_WARPS;
constexpr int NUM_THREADS = 64 + CONV_THREADS + 128;
constexpr int CSB_BYTES = 128 * 128, CST_BYTES = 128 * 32;
constexpr int SMEM_BYTES = 36864 + WIN_STAGES * WIN_STRIDE + WINB_STAGES * WINB_STRIDE + 2 * (CSB_BYTES + CST_BYTES) + 1024;

struct Stem2Params {
    int N, OH, OW, tiles_w, tiles_h, num_tiles;
    const void* w;
};

// K-major operand without swizzle: 8-row x 16-byte core matrices; LBO = bytes between core matrices adjacent in K,
// SBO = bytes between core matrices adjacent in M / N.
__device__ __forceinline__ uint64_t make_desc_nosw(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>(lbo >> 4) << 16;
    d |= static_cast<uint64_t>(sbo >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    return d;
}

__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
    __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&h);
}

// NOUT = 64 stores the sb tile only (tmYst is not read).
template <int NOUT>
__global__ void __launch_bounds__(NUM_THREADS, 1)
stem_tc2_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmYsb,
                const __grid_constant__ CUtensorMap tmYst, const Stem2Params p) {
    constexpr int W_MMA_BYTES = Stem2Shape<NOUT>::W_MMA_BYTES, W_BYTES = Stem2Shape<NOUT>::W_BYTES;
    constexpr int ACC_COLS = Stem2Shape<NOUT>::ACC_COLS;
    constexpr bool kStem = NOUT == 80;
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t w_bar, win_full[WIN_STAGES], win_empty[WIN_STAGES], a_full[WINB_STAGES],
        a_empty[WINB_STAGES], acc_full[ACC_STAGES], acc_empty[ACC_STAGES];
    __shared__ uint32_t tmem_base_smem;

    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sW = smem;                                   // 14 x [80 x 16] bf16 core-matrix tiles (36 KB reserved)
    uint8_t* sCsb = sW + 36864;                           // 2 x staged sb output (swizzled: 1024-aligned)
    uint8_t* sCst = sCsb + 2 * CSB_BYTES;                 // 2 x staged stem output
    uint8_t* sWin = sCst + 2 * CST_BYTES;                 // 3 x [3][37][24] fp32 (128-aligned TMA destinations)
    uint8_t* sWinB = sWin + WIN_STAGES * WIN_STRIDE;      // 3 x [37][24][4] bf16: the A operand of all 14 MMAs

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        tc::prefetch_tmap(&tmX);
        tc::prefetch_tmap(&tmYsb);
        if constexpr (kStem) tc::prefetch_tmap(&tmYst);
        tc::mbar_init(&w_bar, 1);
        for (int s = 0; s < WIN_STAGES; ++s) {
            tc::mbar_init(&win_full[s], 1);
            tc::mbar_init(&win_empty[s], CONV_WARPS);
        }
        for (int s = 0; s < WINB_STAGES; ++s) {
            tc::mbar_init(&a_full[s], CONV_WARPS);
            tc::mbar_init(&a_empty[s], 1);
        }
        for (int s = 0; s < ACC_STAGES; ++s) {
            tc::mbar_init(&acc_full[s], 1);
            tc::mbar_init(&acc_empty[s], 4);
        }
        tc::mbar_fence_init();
        tc::fence_proxy_async();
    }
    if (warp == 1) tc::tmem_alloc(&tmem_base_smem, ACC_STAGES * ACC_COLS);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_base_smem;
    const int tiles_per_img = p.tiles_w * p.tiles_h;

    if (warp == 0) {
        if (lane == 0) {
            // ================= TMA producer =================
            tc::mbar_expect_tx(&w_bar, W_BYTES);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             tc::smem_u32(sW)),
                         "l"(reinterpret_cast<uint64_t>(p.w)), "r"(W_BYTES), "r"(tc::smem_u32(&w_bar))
                         : "memory");
            int it = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
                const int s = it % WIN_STAGES;
                const uint32_t ph = (it / WIN_STAGES) & 1;
                const int img = tile / tiles_per_img, r = tile - img * tiles_per_img;
                const int oh0 = (r / p.tiles_w) * TH, ow0 = (r % p.tiles_w) * TW;
                tc::mbar_wait(&win_empty[s], ph ^ 1);
                tc::mbar_expect_tx(&win_full[s], WIN_BYTES);
                // the innermost TMA coordinate must be 16-byte aligned: start one column left of the 7x7 footprint
                tc::tma_load_3d(sWin + s * WIN_STRIDE, &tmX, &win_full[s], 2 * ow0 - 4, 2 * oh0 - 3, 3 * img);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer =================
        const uint32_t leader = tc::elect_one();
        const uint32_t idesc = tc::make_idesc_bf16(128, NOUT);
        tc::mbar_wait(&w_bar, 0);
        int it = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const int as = it % WINB_STAGES, cs = it % ACC_STAGES;
            const uint32_t aph = (it / WINB_STAGES) & 1, cph = (it / ACC_STAGES) & 1;
            tc::mbar_wait(&acc_empty[cs], cph ^ 1);
            tc::mbar_wait(&a_full[as], aph);
            tc::tc_fence_after();
            const uint32_t a0 = tc::smem_u32(sWinB) + as * WINB_STRIDE;
            const uint32_t d = tmem + cs * ACC_COLS;
#pragma unroll
            for (int j = 0; j < NMMA; ++j) {  // j = ky * 2 + K half
                const uint64_t a_desc = make_desc_nosw(a0 + (j >> 1) * PITCH + (j & 1) * 32, 16, 2 * PITCH);
                const uint64_t w_desc = make_desc_nosw(tc::smem_u32(sW) + j * W_MMA_BYTES, (NOUT / 8) * 128, 128);
                tc::umma_bf16_if(leader, d, a_desc, w_desc, idesc, j ? 1u : 0u);
            }
            tc::umma_commit_if(leader, &a_empty[as]);
            tc::umma_commit_if(leader, &acc_full[cs]);
        }
        __syncwarp();
    } else if (warp < EPI_WARP0) {
        // ================= converters: fp32 planar window -> (r, g, b, 1.0) bf16 pixels =================
        const int ct = threadIdx.x - 64;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const int ws = it % WIN_STAGES, as = it % WINB_STAGES;
            const uint32_t wph = (it / WIN_STAGES) & 1, aph = (it / WINB_STAGES) & 1;
            tc::mbar_wait(&win_full[ws], wph);
            tc::mbar_wait(&a_empty[as], aph ^ 1);  // the MMAs that read this copy three tiles ago are done
            const uint32_t win = tc::smem_u32(sWin) + ws * WIN_STRIDE;
            const uint32_t winb = tc::smem_u32(sWinB) + as * WINB_STRIDE;
#pragma unroll
            for (int k = 0; k < (WIN_H * WIN_W + CONV_THREADS - 1) / CONV_THREADS; ++k) {
                const int pidx = ct + CONV_THREADS * k;  // = row * 24 + col: planar index and pixel index coincide
                if (pidx < WIN_H * WIN_W) {
                    float f0, f1, f2;
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(f0) : "r"(win + pidx * 4));
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(f1) : "r"(win + (WIN_H * WIN_W + pidx) * 4));
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(f2) : "r"(win + (2 * WIN_H * WIN_W + pidx) * 4));
                    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(winb + pidx * 8), "r"(pack2(f0, f1)), "r"(pack2(f2, 1.0f))
                                 : "memory");
                }
            }
            tc::fence_proxy_async();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
            __syncwarp();
            if (lane == 0) {
                tc::mbar_arrive(&win_empty[ws]);
                tc::mbar_arrive(&a_full[as]);
            }
        }
    } else {
        // ================= epilogue (as stem_tc.cu; patch rows are m = oy * 8 + ox) =================
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const bool leader = warp == EPI_WARP0 && lane == 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const int cs = it % ACC_STAGES;
            const uint32_t cph = (it / ACC_STAGES) & 1;
            const int img = tile / tiles_per_img, rr = tile - img * tiles_per_img;
            const int oh0 = (rr / p.tiles_w) * TH, ow0 = (rr % p.tiles_w) * TW;
            uint8_t* bsb = sCsb + (it & 1) * CSB_BYTES;
            uint8_t* bst = sCst + (it & 1) * CST_BYTES;
            tc::mbar_wait(&acc_full[cs], cph);
            tc::tc_fence_after();
            const uint32_t taddr = tmem + cs * ACC_COLS + (static_cast<uint32_t>(q * 32) << 16);
            uint32_t a0[32], a1[32], a2[16];
            tc::tmem_ld32(taddr, a0);
            tc::tmem_ld32(taddr + 32, a1);
            if constexpr (kStem) tc::tmem_ld16(taddr + 64, a2);
            tc::tmem_ld_wait();
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&acc_empty[cs]);
            if (leader) tc::bulk_wait_read<1>();
            tc::named_bar_sync(1, 128);
            const uint32_t rowp = tc::smem_u32(bsb) + r * 128;
#pragma unroll
            for (int g = 0; g < 8; ++g) {
                uint32_t w[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float lo = __uint_as_float(g < 4 ? a0[8 * g + 2 * j] : a1[8 * (g - 4) + 2 * j]);
                    const float hi = __uint_as_float(g < 4 ? a0[8 * g + 2 * j + 1] : a1[8 * (g - 4) + 2 * j + 1]);
                    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(w[j]) : "f"(hi), "f"(lo));
                }
                tc::sts128(rowp + ((g ^ (r & 7)) << 4), make_uint4(w[0], w[1], w[2], w[3]));
            }
            if constexpr (kStem) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    float v[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float t = __uint_as_float(a2[8 * g + j]);
                        v[j] = t * __saturatef(fmaf(t, 1.f / 6.f, 0.5f));
                    }
                    Vec16<bf16> o;
                    o.pack(v);
                    tc::sts128(tc::smem_u32(bst) + r * 32 + g * 16, o.raw);
                }
            }
            tc::fence_proxy_async();
            tc::named_bar_sync(1, 128);
            if (leader) {
                tc::tma_store_4d(&tmYsb, bsb, 0, ow0, oh0, img);
                if constexpr (kStem) tc::tma_store_4d(&tmYst, bst, 0, ow0, oh0, img);
                tc::bulk_commit();
            }
        }
        if (leader) tc::bulk_wait_read<0>();
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, ACC_STAGES * ACC_COLS);
    }
}

template <int NOUT>
int g_attr_set2 = 0;

// Host side of both instantiations.  y_stem == nullptr: NOUT = 64, sb.conv1 alone.
template <int NOUT>
int launch_stem2(const char* name, const float* x, int N, int H, int W, const void* w_packed, void* y_sb, long long ld_sb,
                 void* y_stem, long long ld_stem, int OH, int OW, cabinet_stream_t stream) {
    constexpr bool kStem = NOUT == 80;
    CAB_REQUIRE(x && w_packed && y_sb && (y_stem || !kStem), "%s: null pointer", name);
    CAB_REQUIRE(N >= 0 && H > 0 && W > 0 && W % 4 == 0, "%s: W must be a multiple of 4 (TMA row pitch)", name);
    CAB_REQUIRE(OH == (H - 1) / 2 + 1 && OW == (W - 1) / 2 + 1, "%s: inconsistent output size", name);
    CAB_REQUIRE(ld_sb >= 64 && ld_sb % 8 == 0 && (!kStem || (ld_stem >= 16 && ld_stem % 8 == 0)) &&
                    (reinterpret_cast<uintptr_t>(y_sb) & 15) == 0 && (reinterpret_cast<uintptr_t>(y_stem) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_packed) & 15) == 0,
                kStem ? "%s: alignment" : "%s: alignment (ld_y a multiple of 8 >= 64, 16-byte aligned pointers)", name);
    if (N == 0) return CABINET_OK;
    cab_encode_tiled_fn enc = cab_get_encode_tiled();
    CAB_REQUIRE(enc != nullptr, "%s: cuTensorMapEncodeTiled unavailable", name);
    CUtensorMap tmX;
    {
        cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)3 * N};
        cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4};
        cuuint32_t box[3] = {WIN_W, WIN_H, 3};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&tmX, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(x), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            cabinet_set_error("%s: input tensor map encode failed (CUresult %d)", name, (int)r);
            return CABINET_ERR_CUDA;
        }
    }
    Stem2Params p;
    p.N = N; p.OH = OH; p.OW = OW; p.w = w_packed;
    p.tiles_w = (OW + TW - 1) / TW;
    p.tiles_h = (OH + TH - 1) / TH;
    const long long nt = static_cast<long long>(N) * p.tiles_w * p.tiles_h;
    CAB_REQUIRE(nt < (1LL << 31), "%s: too many tiles", name);
    p.num_tiles = static_cast<int>(nt);
    CUtensorMap tmYsb, tmYst;
    {
        const uint64_t dsb[4] = {64, (uint64_t)OW, (uint64_t)OH, (uint64_t)N};
        const uint64_t ssb[3] = {(uint64_t)ld_sb * 2, (uint64_t)ld_sb * 2 * OW, (uint64_t)ld_sb * 2 * OW * OH};
        const uint32_t bsb[4] = {64, TW, TH, 1};
        int rc = cab_make_tmap_bf16(&tmYsb, y_sb, 4, dsb, ssb, bsb);
        if (rc) return rc;
        if (kStem) {
            const uint64_t dst[4] = {16, (uint64_t)OW, (uint64_t)OH, (uint64_t)N};
            const uint64_t sst[3] = {(uint64_t)ld_stem * 2, (uint64_t)ld_stem * 2 * OW, (uint64_t)ld_stem * 2 * OW * OH};
            const uint32_t bst[4] = {16, TW, TH, 1};
            rc = cab_make_tmap_bf16(&tmYst, y_stem, 4, dst, sst, bst, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                    CU_TENSOR_MAP_SWIZZLE_NONE);
            if (rc) return rc;
        } else {
            tmYst = tmYsb;  // not read by the NOUT = 64 kernel
        }
    }
    if (!g_attr_set2<NOUT>) {
        CAB_CUDA(cudaFuncSetAttribute(stem_tc2_kernel<NOUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        g_attr_set2<NOUT> = 1;
    }
    int dev = 0, sms = 148;
    CAB_CUDA(cudaGetDevice(&dev));
    CAB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int grid = static_cast<int>(std::min<long long>(nt, sms));
    stem_tc2_kernel<NOUT><<<grid, NUM_THREADS, SMEM_BYTES, static_cast<cudaStream_t>(stream)>>>(tmX, tmYsb, tmYst, p);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

}  // namespace

extern "C" int cabinet_stem_tc2(const float* x, int N, int H, int W, const void* w_packed2, void* y_sb, long long ld_sb,
                                void* y_stem, long long ld_stem, int OH, int OW, cabinet_stream_t stream) {
    return launch_stem2<80>("stem_tc2", x, N, H, W, w_packed2, y_sb, ld_sb, y_stem, ld_stem, OH, OW, stream);
}

// sb.conv1 alone (a standalone SpatialBranch): the N = 64 instantiation, one TMA store per tile.
extern "C" int cabinet_stem7_tc(const float* x, int N, int H, int W, const void* w_packed7, void* y, long long ld_y, int OH,
                                int OW, cabinet_stream_t stream) {
    return launch_stem2<64>("stem7_tc", x, N, H, W, w_packed7, y, ld_y, nullptr, 0, OH, OW, stream);
}

// ===================================================================================================================
// The backbone stem alone (a standalone MobileNetV3): 3x3 s2 p1, 3 -> 16, BN folded, HardSwish, in the formulation
// above.  The window starts one aligned pixel group left of the footprint (input column 2 ow0 - 4), so tap row ky of
// output (oy, ox) reads the copy at pixels 2 ox + 2 .. 2 ox + 5: slot 0 carries no weight (its constant-1 channel carries
// the bias), slots 1..3 are kx = 0..2.  That is ONE K16 slice per tap row: 3 MMAs of M128 N16 K16 per 128 pixels, over a
// 33 x 20 window.  Per tile the kernel moves ~8 KB in and 4 KB out against 6 tiny MMAs, so it keeps more windows in
// flight (6 stages) than the fused kernel.
namespace {
namespace s3 {

constexpr int TH = 16, TW = 8;
constexpr int WIN_H = 2 * TH + 1, WIN_W = 20;       // rows 2 oh0 - 1 .. 2 oh0 + 31, cols 2 ow0 - 4 .. 2 ow0 + 15
constexpr int WIN_BYTES = 3 * WIN_H * WIN_W * 4;    // 7920
constexpr int WIN_STRIDE = 7936;
constexpr int WIN_STAGES = 6;
constexpr int PITCH = WIN_W * 8;                    // 160
constexpr int WINB_STRIDE = 5376;                   // >= WIN_H * PITCH = 5280
constexpr int WINB_STAGES = 3;
constexpr int NOUT = 16;
constexpr int NMMA = 3;                             // one K16 slice per tap row
constexpr int W_MMA_BYTES = 2 * (NOUT / 8) * 128;   // 512
constexpr int W_BYTES = NMMA * W_MMA_BYTES;         // 1536
constexpr int ACC_STAGES = 2, ACC_COLS = 32;
constexpr int CONV_WARPS = 8, CONV_THREADS = 32 * CONV_WARPS;
constexpr int EPI_WARP0 = 2 + CONV_WARPS;
constexpr int NUM_THREADS = 64 + CONV_THREADS + 128;
constexpr int CST_BYTES = 128 * 32;
constexpr int W_RESERVE = 2048;
constexpr int SMEM_BYTES = W_RESERVE + 2 * CST_BYTES + WIN_STAGES * WIN_STRIDE + WINB_STAGES * WINB_STRIDE + 1024;

__global__ void __launch_bounds__(NUM_THREADS, 1)
stem3_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY, const Stem2Params p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t w_bar, win_full[WIN_STAGES], win_empty[WIN_STAGES], a_full[WINB_STAGES],
        a_empty[WINB_STAGES], acc_full[ACC_STAGES], acc_empty[ACC_STAGES];
    __shared__ uint32_t tmem_base_smem;

    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sW = smem;                                   // 3 x [16 x 16] bf16 core-matrix tiles
    uint8_t* sCst = sW + W_RESERVE;                       // 2 x staged output tile [128 px][16]
    uint8_t* sWin = sCst + 2 * CST_BYTES;                 // 6 x [3][33][20] fp32
    uint8_t* sWinB = sWin + WIN_STAGES * WIN_STRIDE;      // 3 x [33][20][4] bf16: the A operand of the 3 MMAs

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        tc::prefetch_tmap(&tmX);
        tc::prefetch_tmap(&tmY);
        tc::mbar_init(&w_bar, 1);
        for (int s = 0; s < WIN_STAGES; ++s) {
            tc::mbar_init(&win_full[s], 1);
            tc::mbar_init(&win_empty[s], CONV_WARPS);
        }
        for (int s = 0; s < WINB_STAGES; ++s) {
            tc::mbar_init(&a_full[s], CONV_WARPS);
            tc::mbar_init(&a_empty[s], 1);
        }
        for (int s = 0; s < ACC_STAGES; ++s) {
            tc::mbar_init(&acc_full[s], 1);
            tc::mbar_init(&acc_empty[s], 4);
        }
        tc::mbar_fence_init();
        tc::fence_proxy_async();
    }
    if (warp == 1) tc::tmem_alloc(&tmem_base_smem, ACC_STAGES * ACC_COLS);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_base_smem;
    const int tiles_per_img = p.tiles_w * p.tiles_h;

    if (warp == 0) {
        if (lane == 0) {
            // ================= TMA producer =================
            tc::mbar_expect_tx(&w_bar, W_BYTES);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             tc::smem_u32(sW)),
                         "l"(reinterpret_cast<uint64_t>(p.w)), "r"(W_BYTES), "r"(tc::smem_u32(&w_bar))
                         : "memory");
            int it = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
                const int s = it % WIN_STAGES;
                const uint32_t ph = (it / WIN_STAGES) & 1;
                const int img = tile / tiles_per_img, r = tile - img * tiles_per_img;
                const int oh0 = (r / p.tiles_w) * TH, ow0 = (r % p.tiles_w) * TW;
                tc::mbar_wait(&win_empty[s], ph ^ 1);
                tc::mbar_expect_tx(&win_full[s], WIN_BYTES);
                tc::tma_load_3d(sWin + s * WIN_STRIDE, &tmX, &win_full[s], 2 * ow0 - 4, 2 * oh0 - 1, 3 * img);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer =================
        const uint32_t leader = tc::elect_one();
        const uint32_t idesc = tc::make_idesc_bf16(128, NOUT);
        tc::mbar_wait(&w_bar, 0);
        int it = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const int as = it % WINB_STAGES, cs = it % ACC_STAGES;
            const uint32_t aph = (it / WINB_STAGES) & 1, cph = (it / ACC_STAGES) & 1;
            tc::mbar_wait(&acc_empty[cs], cph ^ 1);
            tc::mbar_wait(&a_full[as], aph);
            tc::tc_fence_after();
            const uint32_t a0 = tc::smem_u32(sWinB) + as * WINB_STRIDE;
            const uint32_t d = tmem + cs * ACC_COLS;
#pragma unroll
            for (int ky = 0; ky < NMMA; ++ky) {  // A row (oy, ox) of tap row ky: copy row 2 oy + ky, pixel 2 ox + 2
                const uint64_t a_desc = make_desc_nosw(a0 + ky * PITCH + 16, 16, 2 * PITCH);
                const uint64_t w_desc = make_desc_nosw(tc::smem_u32(sW) + ky * W_MMA_BYTES, (NOUT / 8) * 128, 128);
                tc::umma_bf16_if(leader, d, a_desc, w_desc, idesc, ky ? 1u : 0u);
            }
            tc::umma_commit_if(leader, &a_empty[as]);
            tc::umma_commit_if(leader, &acc_full[cs]);
        }
        __syncwarp();
    } else if (warp < EPI_WARP0) {
        // ================= converters: fp32 planar window -> (r, g, b, 1.0) bf16 pixels =================
        const int ct = threadIdx.x - 64;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const int ws = it % WIN_STAGES, as = it % WINB_STAGES;
            const uint32_t wph = (it / WIN_STAGES) & 1, aph = (it / WINB_STAGES) & 1;
            tc::mbar_wait(&win_full[ws], wph);
            tc::mbar_wait(&a_empty[as], aph ^ 1);
            const uint32_t win = tc::smem_u32(sWin) + ws * WIN_STRIDE;
            const uint32_t winb = tc::smem_u32(sWinB) + as * WINB_STRIDE;
#pragma unroll
            for (int k = 0; k < (WIN_H * WIN_W + CONV_THREADS - 1) / CONV_THREADS; ++k) {
                const int pidx = ct + CONV_THREADS * k;
                if (pidx < WIN_H * WIN_W) {
                    float f0, f1, f2;
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(f0) : "r"(win + pidx * 4));
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(f1) : "r"(win + (WIN_H * WIN_W + pidx) * 4));
                    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(f2) : "r"(win + (2 * WIN_H * WIN_W + pidx) * 4));
                    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(winb + pidx * 8), "r"(pack2(f0, f1)), "r"(pack2(f2, 1.0f))
                                 : "memory");
                }
            }
            tc::fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                tc::mbar_arrive(&win_empty[ws]);
                tc::mbar_arrive(&a_full[as]);
            }
        }
    } else {
        // ================= epilogue: HardSwish, one 16 x 8 x 16 TMA store per tile =================
        const int q = warp & 3;
        const int r = q * 32 + lane;
        const bool leader = warp == EPI_WARP0 && lane == 0;
        int it = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const int cs = it % ACC_STAGES;
            const uint32_t cph = (it / ACC_STAGES) & 1;
            const int img = tile / tiles_per_img, rr = tile - img * tiles_per_img;
            const int oh0 = (rr / p.tiles_w) * TH, ow0 = (rr % p.tiles_w) * TW;
            uint8_t* bst = sCst + (it & 1) * CST_BYTES;
            tc::mbar_wait(&acc_full[cs], cph);
            tc::tc_fence_after();
            uint32_t a[16];
            tc::tmem_ld16(tmem + cs * ACC_COLS + (static_cast<uint32_t>(q * 32) << 16), a);
            tc::tmem_ld_wait();
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&acc_empty[cs]);
            if (leader) tc::bulk_wait_read<1>();  // the store that read this staging buffer two tiles ago is done
            tc::named_bar_sync(1, 128);
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                float v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float t = __uint_as_float(a[8 * g + j]);
                    v[j] = t * __saturatef(fmaf(t, 1.f / 6.f, 0.5f));
                }
                Vec16<bf16> o;
                o.pack(v);
                tc::sts128(tc::smem_u32(bst) + r * 32 + g * 16, o.raw);
            }
            tc::fence_proxy_async();
            tc::named_bar_sync(1, 128);
            if (leader) {
                tc::tma_store_4d(&tmY, bst, 0, ow0, oh0, img);
                tc::bulk_commit();
            }
        }
        if (leader) tc::bulk_wait_read<0>();
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, ACC_STAGES * ACC_COLS);
    }
}

int g_attr_set3 = 0;

int launch(const float* x, int N, int H, int W, const void* w_packed3, void* y, long long ld_y, int OH, int OW,
           cabinet_stream_t stream) {
    CAB_REQUIRE(x && w_packed3 && y, "stem3_tc: null pointer");
    CAB_REQUIRE(N >= 0 && H > 0 && W > 0 && W % 4 == 0, "stem3_tc: W must be a multiple of 4 (TMA row pitch)");
    CAB_REQUIRE(OH == (H - 1) / 2 + 1 && OW == (W - 1) / 2 + 1, "stem3_tc: inconsistent output size");
    CAB_REQUIRE(ld_y >= 16 && ld_y % 8 == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(w_packed3) & 15) == 0,
                "stem3_tc: alignment (ld_y a multiple of 8 >= 16, 16-byte aligned pointers)");
    if (N == 0) return CABINET_OK;
    cab_encode_tiled_fn enc = cab_get_encode_tiled();
    CAB_REQUIRE(enc != nullptr, "stem3_tc: cuTensorMapEncodeTiled unavailable");
    CUtensorMap tmX;
    {
        cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)3 * N};
        cuuint64_t strides[2] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4};
        cuuint32_t box[3] = {WIN_W, WIN_H, 3};
        cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&tmX, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(x), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) {
            cabinet_set_error("stem3_tc: input tensor map encode failed (CUresult %d)", (int)r);
            return CABINET_ERR_CUDA;
        }
    }
    Stem2Params p;
    p.N = N; p.OH = OH; p.OW = OW; p.w = w_packed3;
    p.tiles_w = (OW + TW - 1) / TW;
    p.tiles_h = (OH + TH - 1) / TH;
    const long long nt = static_cast<long long>(N) * p.tiles_w * p.tiles_h;
    CAB_REQUIRE(nt < (1LL << 31), "stem3_tc: too many tiles");
    p.num_tiles = static_cast<int>(nt);
    CUtensorMap tmY;
    {
        const uint64_t d[4] = {16, (uint64_t)OW, (uint64_t)OH, (uint64_t)N};
        const uint64_t s[3] = {(uint64_t)ld_y * 2, (uint64_t)ld_y * 2 * OW, (uint64_t)ld_y * 2 * OW * OH};
        const uint32_t b[4] = {16, TW, TH, 1};
        int rc = cab_make_tmap_bf16(&tmY, y, 4, d, s, b, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_SWIZZLE_NONE);
        if (rc) return rc;
    }
    if (!g_attr_set3) {
        CAB_CUDA(cudaFuncSetAttribute(stem3_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
        g_attr_set3 = 1;
    }
    int dev = 0, sms = 148;
    CAB_CUDA(cudaGetDevice(&dev));
    CAB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int grid = static_cast<int>(std::min<long long>(nt, sms));
    stem3_tc_kernel<<<grid, NUM_THREADS, SMEM_BYTES, static_cast<cudaStream_t>(stream)>>>(tmX, tmY, p);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

}  // namespace s3
}  // namespace

extern "C" int cabinet_stem3_tc(const float* x, int N, int H, int W, const void* w_packed3, void* y, long long ld_y, int OH,
                                int OW, cabinet_stream_t stream) {
    return s3::launch(x, N, H, W, w_packed3, y, ld_y, OH, OW, stream);
}
