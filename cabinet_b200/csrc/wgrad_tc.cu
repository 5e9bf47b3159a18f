// Weight gradient of a stride-1 "same" (or any stride-2) convolution on the 5th-gen tensor cores (tcgen05.mma, fp32 accumulation in TMEM):
//
//     dW[co][ky][kx][ci] = sum over pixels (n, oy, ox)  dy[n][oy][ox][co] * x[n][oy + ky - pad][ox + kx - pad][ci]
//
// (reference: the autograd backward of every nn.Conv2d on the training path, src/scripts/train.py:436).  Per filter tap
// it is a GEMM whose reduction dimension is the PIXEL index: D[128 co x NB ci] += A^T B with A = dy tile [K pixels][co],
// B = x tile [K pixels][ci].  In NHWC both operands have the reduction index as their ROW and the M / N index contiguous,
// i.e. they are MN-major UMMA operands: a TMA box {64 channels, TW, TH, 1} lands as K rows of 128 bytes in the
// 128-byte-swizzled layout, which is exactly the canonical MN-major SWIZZLE_128B atom (64 MN elements x 8 K rows);
// descriptors: LBO = bytes between 64-channel blocks, SBO = 1024 (8 K rows), instruction descriptor a_major = b_major = 1.
// No transposition pass, no im2col: the tap shift is a shifted box coordinate and the zero padding TMA's out-of-bounds fill.
// Stride 2: one tensor map per input parity (py, px): map(py,px)[h][w] = x[2h+py][2w+px]; tap (ky, kx) reads the map of
// parity ((ky - pad) & 1, (kx - pad) & 1) at the box shifted by (ky - pad) >> 1 -- again a plain box.
//
// Grid: (cout tiles of 128, taps x cin tiles of NB, pixel splits).  Warp 0 = TMA producer, warp 1 = TMEM allocator +
// MMA issuer, warps 2-5 = epilogue (TMEM -> fp32 partial[split][co][tap * Cin + ci]).  The splits are added in index
// order by wgrad_finalize (deterministic), which also scatters into the OIHW gradient.
#include "tc_common.cuh"

namespace {

constexpr int KT = 64;                 // pixels per pipeline stage (4 MMAs of K = 16)
constexpr int BOX_BYTES = KT * 128;    // one {64 channels x KT pixels} box
constexpr int WG_THREADS = 192;
constexpr int WG_MAX_STAGES = 8;

struct WgParams {
    int Cin, Cout, taps, KW, pad, stride;
    int TW, TH, tiles_w, tiles_h, n_k_tiles, tiles_per_split, flat;
    int NB, n_blocks, n_tiles, stages, stage_bytes;
    float* partial;
};

// MN-major SWIZZLE_128B operand: start>>4 | LBO>>4 [16,30) | SBO>>4 [32,46) | version 1 [46,48) | layout 2 [61,64)
__device__ __forceinline__ uint64_t make_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;
    d |= static_cast<uint64_t>(1024 >> 4) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}

template <typename T>  // operand type: bf16 or f16
__global__ void __launch_bounds__(WG_THREADS, 2)
conv_wgrad_tc_kernel(const __grid_constant__ CUtensorMap tmDY, const __grid_constant__ CUtensorMap tmX,
                     const __grid_constant__ CUtensorMap tmX1, const __grid_constant__ CUtensorMap tmX2,
                     const __grid_constant__ CUtensorMap tmX3, const WgParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[WG_MAX_STAGES], empty_bar[WG_MAX_STAGES], acc_bar;
    __shared__ uint32_t tmem_base_smem;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int co0 = blockIdx.x * 128;
    const int tap = blockIdx.y / p.n_tiles, nt = blockIdx.y - tap * p.n_tiles;
    const int ci0 = nt * p.NB;
    const int ky = tap / p.KW, kx = tap - ky * p.KW;
    const int t0 = blockIdx.z * p.tiles_per_split;
    const int t1 = min(t0 + p.tiles_per_split, p.n_k_tiles);

    if (threadIdx.x == 0) {
        tc::prefetch_tmap(&tmDY);
        tc::prefetch_tmap(&tmX);
        if (p.stride == 2) {
            tc::prefetch_tmap(&tmX1);
            tc::prefetch_tmap(&tmX2);
            tc::prefetch_tmap(&tmX3);
        }
        for (int s = 0; s < p.stages; ++s) {
            tc::mbar_init(&full_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
        }
        tc::mbar_init(&acc_bar, 1);
        tc::mbar_fence_init();
        tc::fence_proxy_async();
    }
    if (warp == 1) tc::tmem_alloc(&tmem_base_smem, static_cast<uint32_t>(p.NB < 32 ? 32 : p.NB));
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_base_smem;

    if (warp == 0) {
        // ---------------- TMA producer
        if (lane == 0) {
            // stride 2: this tap's input parity map and box shift
            const int dy_ = ky - p.pad, dx_ = kx - p.pad;
            const int par = p.stride == 2 ? ((dy_ & 1) * 2 + (dx_ & 1)) : 0;
            const int shy = p.stride == 2 ? (dy_ - (dy_ & 1)) / 2 : dy_, shx = p.stride == 2 ? (dx_ - (dx_ & 1)) / 2 : dx_;
            const CUtensorMap* tmx = par == 0 ? &tmX : (par == 1 ? &tmX1 : (par == 2 ? &tmX2 : &tmX3));
            for (int t = t0; t < t1; ++t) {
                const int it = t - t0, s = it % p.stages;
                if (it >= p.stages) tc::mbar_wait(&empty_bar[s], ((it / p.stages) - 1) & 1);
                int c1, c2, c3;  // box origin (x, y, image) of pixel tile t
                if (p.flat) {
                    c1 = t * KT; c2 = 0; c3 = 0;
                } else {
                    const int tw = t % p.tiles_w, r = t / p.tiles_w;
                    c1 = tw * p.TW; c2 = (r % p.tiles_h) * p.TH; c3 = r / p.tiles_h;
                }
                uint8_t* st = smem + static_cast<size_t>(s) * p.stage_bytes;
                tc::mbar_expect_tx(&full_bar[s], static_cast<uint32_t>(p.stage_bytes));
                tc::tma_load_4d(st, &tmDY, &full_bar[s], co0, c1, c2, c3);
                tc::tma_load_4d(st + BOX_BYTES, &tmDY, &full_bar[s], co0 + 64, c1, c2, c3);
                const int xs = p.flat ? c1 : c1 + shx, ys = p.flat ? 0 : c2 + shy;
                for (int j = 0; j < p.n_blocks; ++j)
                    tc::tma_load_4d(st + (2 + j) * BOX_BYTES, tmx, &full_bar[s], ci0 + 64 * j, xs, ys, c3);
            }
        }
    } else if (warp == 1) {
        // ---------------- MMA issuer: D[128 x NB] += A^T B over the pixel tiles of this split
        const uint32_t leader = tc::elect_one();
        // kind::f16, D fp32, A/B bf16 or f16, BOTH MN-major (bits 15, 16), N >> 3 at [17,23), M >> 4 at [24,29)
        const uint32_t idesc = tc::make_idesc<T>(128, p.NB) | (1u << 15) | (1u << 16);
        for (int t = t0; t < t1; ++t) {
            const int it = t - t0, s = it % p.stages;
            tc::mbar_wait(&full_bar[s], (it / p.stages) & 1);
            tc::tc_fence_after();
            const uint32_t sa = tc::smem_u32(smem + static_cast<size_t>(s) * p.stage_bytes);
            const uint64_t ad = make_desc_mn_sw128(sa, BOX_BYTES);
            const uint64_t bd = make_desc_mn_sw128(sa + 2 * BOX_BYTES, BOX_BYTES);
#pragma unroll
            for (int kk = 0; kk < KT / 16; ++kk)  // 16 pixel rows = 2048 bytes per K step
                tc::umma_bf16_if(leader, tmem, ad + static_cast<uint64_t>(kk * (2048 >> 4)), bd + static_cast<uint64_t>(kk * (2048 >> 4)),
                                 idesc, (it > 0 || kk > 0) ? 1u : 0u);
            tc::umma_commit_if(leader, &empty_bar[s]);
        }
        tc::umma_commit_if(leader, &acc_bar);
        __syncwarp();
    } else {
        // ---------------- epilogue: TMEM lane = output channel row, 32 input-channel columns per round trip
        const int q = warp & 3;
        const int co = co0 + q * 32 + lane;
        const long long Kn = static_cast<long long>(p.taps) * p.Cin;
        float* out = p.partial + (static_cast<long long>(blockIdx.z) * p.Cout + co) * Kn + static_cast<long long>(tap) * p.Cin;
        tc::mbar_wait(&acc_bar, 0);
        tc::tc_fence_after();
        for (int c = 0; c < p.NB; c += 32) {
            if (ci0 + c >= p.Cin) break;  // warp-uniform
            uint32_t v[32];
            tc::tmem_ld32(tmem + c + (static_cast<uint32_t>(q * 32) << 16), v);
            tc::tmem_ld_wait();
            if (co < p.Cout) {
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (ci0 + c + j < p.Cin) out[ci0 + c + j] = __uint_as_float(v[j]);
            }
        }
        tc::tc_fence_before();
    }
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, static_cast<uint32_t>(p.NB < 32 ? 32 : p.NB));
    }
}

// dW (OIHW) += sum over splits of partial[z][co][tap*Cin + ci]
__global__ void wgrad_tc_finalize_kernel(const float* __restrict__ partial, int splits, int Cout, int Cin, int taps,
                                         float* __restrict__ dw) {
    const long long total = static_cast<long long>(Cout) * Cin * taps;
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int ci = static_cast<int>(i % Cin);
    const long long t = i / Cin;
    const int tap = static_cast<int>(t % taps), co = static_cast<int>(t / taps);
    float sum = 0.f;
    for (int z = 0; z < splits; ++z) sum += partial[static_cast<long long>(z) * total + i];
    dw[(static_cast<long long>(co) * Cin + ci) * taps + tap] += sum;
}

// The same for many splits (small weight matrices cut over up to 296 pixel ranges): 8 warps of a block walk 8 interleaved
// split subsets of 32 consecutive outputs (coalesced), then warp 0 adds the 8 sums in order -- a thread per output
// would walk all splits alone, one dependent L2 round trip after the other (30 us for 4 KB of output).
constexpr int FZ = 8;
__global__ void __launch_bounds__(32 * FZ)
wgrad_tc_finalize_par_kernel(const float* __restrict__ partial, int splits, int Cout, int Cin, int taps, float* __restrict__ dw) {
    __shared__ float s_sum[FZ][32];
    const int ti = threadIdx.x & 31, zg = threadIdx.x >> 5;
    const long long total = static_cast<long long>(Cout) * Cin * taps;
    const long long i = static_cast<long long>(blockIdx.x) * 32 + ti;
    float sum = 0.f;
    if (i < total)
        for (int z = zg; z < splits; z += FZ) sum += partial[static_cast<long long>(z) * total + i];
    s_sum[zg][ti] = sum;
    __syncthreads();
    if (zg != 0 || i >= total) return;
#pragma unroll
    for (int g = 1; g < FZ; ++g) sum += s_sum[g][ti];
    const int ci = static_cast<int>(i % Cin);
    const long long t = i / Cin;
    const int tap = static_cast<int>(t % taps), co = static_cast<int>(t / taps);
    dw[(static_cast<long long>(co) * Cin + ci) * taps + tap] += sum;
}

struct WgPlan {
    int TW, TH, tiles_w, tiles_h, flat, NB, n_tiles, m_tiles, splits, tiles_per_split;
    long long n_k_tiles;
};

WgPlan wg_plan(int N, int H, int W, int Cin, int Cout, int KH, int KW, int stride = 1) {
    // H, W: the OUTPUT (dy) grid
    WgPlan g;
    g.flat = (KH == 1 && KW == 1 && stride == 1) ? 1 : 0;
    if (g.flat) {
        g.TW = KT; g.TH = 1; g.tiles_h = 1;
        g.n_k_tiles = cab_ceil_div(static_cast<long long>(N) * H * W, KT);
        g.tiles_w = static_cast<int>(g.n_k_tiles);
    } else {
        long long best = -1;
        for (int tw = KT; tw >= 2; tw >>= 1) {  // the TH x TW = 64 patch that wastes the fewest pixels (ties: wider)
            const int th = KT / tw;
            const long long cover = cab_ceil_div(W, tw) * tw * cab_ceil_div(H, th) * th;
            if (best < 0 || cover < best) { best = cover; g.TW = tw; g.TH = th; }
        }
        g.tiles_w = static_cast<int>(cab_ceil_div(W, g.TW));
        g.tiles_h = static_cast<int>(cab_ceil_div(H, g.TH));
        g.n_k_tiles = static_cast<long long>(N) * g.tiles_w * g.tiles_h;
    }
    g.NB = Cin <= 64 ? 64 : (Cin <= 128 ? 128 : 256);
    g.n_tiles = static_cast<int>(cab_ceil_div(Cin, g.NB));
    g.m_tiles = static_cast<int>(cab_ceil_div(Cout, 128));
    // ONE wave: NB <= 128 leaves room for two CTAs per SM (<= 100 KB of pipeline stages, 2 x NB <= 512 TMEM columns),
    // NB = 256 runs one CTA per SM with a deeper ring; the pixel range is cut so that the grid does not exceed that
    const long long base = static_cast<long long>(g.m_tiles) * g.n_tiles * KH * KW;
    const long long slots = 148LL * (g.NB <= 128 ? 2 : 1);
    long long splits = std::max<long long>(1, std::min<long long>(slots / base, g.n_k_tiles));
    splits = std::min<long long>(splits, 1024);
    g.tiles_per_split = static_cast<int>(cab_ceil_div(g.n_k_tiles, splits));
    g.splits = static_cast<int>(cab_ceil_div(g.n_k_tiles, g.tiles_per_split));  // <= splits
    return g;
}

}  // namespace

extern "C" long long cabinet_conv_wgrad_tc_scratch_floats(int N, int H, int W, int Cin, int Cout, int KH, int KW, int stride,
                                                          int pad) {
    const int OH = (H + 2 * pad - KH) / stride + 1, OW = (W + 2 * pad - KW) / stride + 1;
    const WgPlan g = wg_plan(N, OH, OW, Cin, Cout, KH, KW, stride);
    return static_cast<long long>(g.splits) * Cout * KH * KW * Cin;
}

// per_image: 1x1 only; one pixel split per image and the "partials" ARE the result: out[n][co][ci] (no second level)
static int wgrad_tc_impl(const void* dy, long long lddy, const void* x, long long ldx, float* dw_oihw, int N, int H, int W,
                         int Cin, int Cout, int KH, int KW, int stride, int pad, float* scratch, int op_dtype,
                         cabinet_stream_t stream, bool per_image) {
    CAB_REQUIRE_DTYPE("conv_wgrad_tc", op_dtype, CAB_DT_BF16 | CAB_DT_F16);
    CAB_REQUIRE(dy && x && dw_oihw && scratch, "conv_wgrad_tc: null pointer");
    CAB_REQUIRE(N > 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0 && KH > 0 && KW > 0 && KH == KW && pad >= 0 &&
                    ((stride == 1 && 2 * pad == KH - 1) || (stride == 2 && H >= 2 && W >= 2)),
                "conv_wgrad_tc: stride-1 'same' (2 * pad == k - 1) or stride-2 convolutions only");
    const int OH = (H + 2 * pad - KH) / stride + 1, OW = (W + 2 * pad - KW) / stride + 1;
    CAB_REQUIRE(lddy % 8 == 0 && ldx % 8 == 0 && lddy >= Cout && ldx >= Cin && (reinterpret_cast<uintptr_t>(dy) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(x) & 15) == 0,
                "conv_wgrad_tc: pixel strides must be multiples of 8 and the bases 16-byte aligned");
    WgPlan g = wg_plan(N, OH, OW, Cin, Cout, KH, KW, stride);
    CAB_REQUIRE(g.n_k_tiles < (1LL << 31) && static_cast<long long>(N) * H * W < (1LL << 31), "conv_wgrad_tc: too many pixels");
    if (per_image) {
        CAB_REQUIRE(g.flat && (static_cast<long long>(H) * W) % KT == 0 && N <= 65535,
                    "conv_wgrad_tc_batched: 1x1, H * W a multiple of 64, at most 65535 images");
        g.tiles_per_split = H * W / KT;
        g.splits = N;
    }
    WgParams p;
    p.Cin = Cin; p.Cout = Cout; p.taps = KH * KW; p.KW = KW; p.pad = pad; p.stride = stride;
    p.TW = g.TW; p.TH = g.TH; p.tiles_w = g.tiles_w; p.tiles_h = g.tiles_h; p.n_k_tiles = static_cast<int>(g.n_k_tiles);
    p.tiles_per_split = g.tiles_per_split; p.flat = g.flat;
    p.NB = g.NB; p.n_blocks = g.NB / 64; p.n_tiles = g.n_tiles;
    p.stage_bytes = (2 + p.n_blocks) * BOX_BYTES;
    p.stages = std::max(2, std::min(WG_MAX_STAGES, ((p.NB <= 128 ? 100 : 200) * 1024) / p.stage_bytes));
    p.partial = scratch;
    CUtensorMap tmDY, tmX[4];
    const uint64_t es = 2;
    if (g.flat) {
        const uint64_t P = static_cast<uint64_t>(N) * H * W;
        const uint32_t box[4] = {64, KT, 1, 1};
        for (int which = 0; which < 2; ++which) {
            const long long ld = which ? ldx : lddy;
            const uint64_t dims[4] = {(uint64_t)(which ? Cin : Cout), P, 1, 1};
            const uint64_t strides[3] = {(uint64_t)ld * es, (uint64_t)ld * es * P, (uint64_t)ld * es * P};
            int rc = cab_make_tmap_2b(which ? &tmX[0] : &tmDY, op_dtype, which ? x : dy, 4, dims, strides, box);
            if (rc) return rc;
        }
        tmX[1] = tmX[2] = tmX[3] = tmX[0];
    } else {
        const uint32_t box[4] = {64, (uint32_t)g.TW, (uint32_t)g.TH, 1};
        {
            const uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)OW, (uint64_t)OH, (uint64_t)N};
            const uint64_t strides[3] = {(uint64_t)lddy * es, (uint64_t)lddy * es * OW, (uint64_t)lddy * es * OW * OH};
            int rc = cab_make_tmap_2b(&tmDY, op_dtype, dy, 4, dims, strides, box);
            if (rc) return rc;
        }
        const uint16_t* xb = reinterpret_cast<const uint16_t*>(x);  // 2-byte elements of either type
        for (int py = 0; py < stride; ++py)
            for (int px = 0; px < stride; ++px) {
                const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)((W - px + stride - 1) / stride),
                                          (uint64_t)((H - py + stride - 1) / stride), (uint64_t)N};
                const uint64_t strides[3] = {(uint64_t)ldx * es * stride, (uint64_t)ldx * es * W * stride,
                                             (uint64_t)ldx * es * W * H};
                int rc = cab_make_tmap_2b(&tmX[py * stride + px], op_dtype, xb + (static_cast<long long>(py) * W + px) * ldx, 4, dims,
                                            strides, box);
                if (rc) return rc;
            }
        if (stride == 1) tmX[1] = tmX[2] = tmX[3] = tmX[0];
    }
    const size_t smem = static_cast<size_t>(p.stages) * p.stage_bytes + 1024;
    static bool attr_done = false;
    if (!attr_done) {
        CAB_CUDA(cudaFuncSetAttribute(conv_wgrad_tc_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        CAB_CUDA(cudaFuncSetAttribute(conv_wgrad_tc_kernel<f16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        attr_done = true;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    dim3 grid(g.m_tiles, p.taps * g.n_tiles, g.splits);
    CAB_DISPATCH_DT_HALF(op_dtype, T, conv_wgrad_tc_kernel<T><<<grid, WG_THREADS, smem, s>>>(tmDY, tmX[0], tmX[1], tmX[2], tmX[3], p));
    CAB_LAUNCH_CHECK();
    const long long total = static_cast<long long>(Cout) * Cin * p.taps;
    if (per_image) return CABINET_OK;
    // many splits of a small matrix: 8 warps per 32 outputs; otherwise one thread per output has parallelism enough
    if (g.splits >= 8 * FZ || (g.splits >= 2 * FZ && total <= 65536))
        wgrad_tc_finalize_par_kernel<<<static_cast<unsigned>(cab_ceil_div(total, 32)), 32 * FZ, 0, s>>>(scratch, g.splits, Cout, Cin,
                                                                                                       p.taps, dw_oihw);
    else
        wgrad_tc_finalize_kernel<<<static_cast<unsigned>(cab_ceil_div(total, 256)), 256, 0, s>>>(scratch, g.splits, Cout, Cin, p.taps,
                                                                                                dw_oihw);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_conv_wgrad_tc(const void* dy, long long lddy, const void* x, long long ldx, float* dw_oihw, int N,
                                     int H, int W, int Cin, int Cout, int KH, int KW, int stride, int pad, float* scratch,
                                     cabinet_stream_t stream) {
    return cabinet_conv_wgrad_tc_dt(dy, lddy, x, ldx, dw_oihw, N, H, W, Cin, Cout, KH, KW, stride, pad, scratch, CABINET_BF16,
                                    stream);
}

extern "C" int cabinet_conv_wgrad_tc_dt(const void* dy, long long lddy, const void* x, long long ldx, float* dw_oihw, int N,
                                        int H, int W, int Cin, int Cout, int KH, int KW, int stride, int pad, float* scratch,
                                        int op_dtype, cabinet_stream_t stream) {
    return wgrad_tc_impl(dy, lddy, x, ldx, dw_oihw, N, H, W, Cin, Cout, KH, KW, stride, pad, scratch, op_dtype, stream, false);
}

extern "C" int cabinet_conv_wgrad_tc_batched(const void* a, long long lda, const void* x, long long ldx, float* out, int N,
                                             int H, int W, int Cin, int Cout, cabinet_stream_t stream) {
    return cabinet_conv_wgrad_tc_batched_dt(a, lda, x, ldx, out, N, H, W, Cin, Cout, CABINET_BF16, stream);
}

extern "C" int cabinet_conv_wgrad_tc_batched_dt(const void* a, long long lda, const void* x, long long ldx, float* out, int N,
                                                int H, int W, int Cin, int Cout, int op_dtype, cabinet_stream_t stream) {
    CAB_REQUIRE(out != nullptr, "conv_wgrad_tc_batched: null pointer");
    return wgrad_tc_impl(a, lda, x, ldx, out, N, H, W, Cin, Cout, 1, 1, 1, 0, out, op_dtype, stream, true);
}
