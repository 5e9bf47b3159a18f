// Depthwise k x k convolution, bf16 (or fp16) NHWC, shared-memory halo staging by TMA.
//
// One CTA = one 8 x 16 output patch of one image for one chunk of <= 64 channels.  A single 4-D TMA box
// {CB channels, (16-1)*S+K cols, (8-1)*S+K rows, 1} brings the input patch INCLUDING its halo into shared memory;
// the zero padding of the convolution is the TMA out-of-bounds fill, so the compute loop has no bounds checks and no
// global loads.  Several CTAs are resident per SM, so the TMA
// fetch of one overlaps the FMAs / stores of the others.  Outputs are written with 16-byte stores that cover whole
// 128-byte lines (8 lanes = the 64 channels of one pixel).
// Epilogue: + folded-BN bias, activation, optional per-(image, channel) partial sums for the SE / GAP consumers.
// HBM-bound: algorithmic bytes = input + output (+ weights); halo re-reads are served by L2.
#include "tc_common.cuh"

namespace {

constexpr int TH = 8, TW = 16, RUN = 4;

struct DwParams {
    int C, OH, OW, CB, act, reverse;  // reverse: blocks walk (tile, image) back to front (CABINET_CONV_REVERSE_TILES)
    const float* w;
    const float* bias;
    void* y;                 // the operand type T of the kernel (bf16 / f16)
    long long ldy;
    long long* gap_sum;      // [N][C] fixed-point (2^-24) pooling sums of the written values (SE consumers), or nullptr
};

// Warp = one output row of the 8 x 16 patch; lane = (column group, channel PAIR): one 32-bit word of the staged NHWC
// pixel per lane, so a warp-wide LDS.32 of a full 64-channel chunk is one conflict-free 128-byte wavefront.  A chunk
// narrower than 64 channels packs 16/COLS column groups into the warp (COLS = columns per lane) to keep lanes busy.
// The thread keeps all K*K taps of its two channels in registers for its whole lifetime (loaded while the TMA is in
// flight) and slides over its COLS output columns: ((COLS-1)*S + K) loads per filter row feed COLS*K*2 FMAs, no weight
// traffic and no bounds checks in the loop.
template <int K, int S, int COLS, typename T>
__device__ __forceinline__ void dw_row(const DwParams& p, const uint8_t* tile, uint64_t* bar, float* s_gap, int cw,
                                       int chunk, int n, int oh0, int ow0) {
    constexpr int IWT = (TW - 1) * S + K;
    constexpr int SPAN = (COLS - 1) * S + K;
    const int row = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lanes_px = cw >> 1;               // lanes per pixel (channel pairs of this chunk)
    const int grp = lane / lanes_px, cl = lane - grp * lanes_px;
    const int c0 = chunk * p.CB + cl * 2;
    const bool active = grp < TW / COLS;
    const int col0 = grp * COLS;

    // 3x3: all nine taps live in registers for the whole thread.  5x5: one filter row (5 taps) at a time, fetched one
    // row ahead -- 25 resident taps cost 50 registers and halve the number of resident CTAs (the kernel is bound by
    // the TMA round trip per CTA, so residency matters more than the 20 extra L1 loads).
    constexpr bool ROWTAPS = K > 3;
    float2 w[ROWTAPS ? K : K * K];
    float2 wn[K];
    float2 acc[COLS];
    if (active) {
        if constexpr (!ROWTAPS) {
#pragma unroll
            for (int t = 0; t < K * K; ++t) w[t] = __ldg(reinterpret_cast<const float2*>(p.w + t * p.C + c0));
        } else {
#pragma unroll
            for (int t = 0; t < K; ++t) wn[t] = __ldg(reinterpret_cast<const float2*>(p.w + t * p.C + c0));
        }
        const float2 b = __ldg(reinterpret_cast<const float2*>(p.bias + c0));
#pragma unroll
        for (int r = 0; r < COLS; ++r) acc[r] = b;
    }
    tc::mbar_wait(bar, 0);
    if (active) {
        constexpr int pitch = 128;  // bytes per staged pixel (64-channel TMA box; narrower chunks are zero filled)
        const uint32_t base = tc::smem_u32(tile) + ((row * S) * IWT + col0 * S) * pitch + cl * 4;
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
            if constexpr (ROWTAPS) {
#pragma unroll
                for (int t = 0; t < K; ++t) w[t] = wn[t];
                if (ky + 1 < K) {
#pragma unroll
                    for (int t = 0; t < K; ++t)
                        wn[t] = __ldg(reinterpret_cast<const float2*>(p.w + ((ky + 1) * K + t) * p.C + c0));
                }
            }
            const uint32_t rowp = base + ky * IWT * pitch;
#pragma unroll
            for (int sx = 0; sx < SPAN; ++sx) {
                uint32_t raw;
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(raw) : "r"(rowp + sx * pitch));
                const float2 xv = cab_unpack2<T>(raw);
#pragma unroll
                for (int r = 0; r < COLS; ++r) {
                    const int kx = sx - r * S;  // compile-time after unrolling
                    if (kx >= 0 && kx < K) cab_ffma2(acc[r], xv, w[ROWTAPS ? kx : ky * K + kx]);
                }
            }
        }
        cab_act_vec<2 * COLS>(&acc[0].x, p.act);
        const int oh = oh0 + row;
        float g0 = 0.f, g1 = 0.f;
        if (oh < p.OH) {
            T* yout = reinterpret_cast<T*>(p.y) + ((static_cast<long long>(n) * p.OH + oh) * p.OW + ow0 + col0) * p.ldy + c0;
#pragma unroll
            for (int r = 0; r < COLS; ++r) {
                if (ow0 + col0 + r < p.OW) {
                    g0 += acc[r].x;
                    g1 += acc[r].y;
                    *reinterpret_cast<uint32_t*>(yout + static_cast<long long>(r) * p.ldy) = cab_pack2<T>(acc[r].x, acc[r].y);
                }
            }
        }
        if (p.gap_sum) {  // this warp's row, this lane's channel pair: summed in a fixed order by the caller
            s_gap[row * 64 + lane * 2] = g0;
            s_gap[row * 64 + lane * 2 + 1] = g1;
        }
    }
}

template <int K, int S, typename T>
__global__ void __launch_bounds__(256, K > 3 ? 3 : 4)
dwconv_tma_kernel(const __grid_constant__ CUtensorMap tmX, const DwParams p) {
    constexpr int PAD = (K - 1) / 2;
    constexpr int IWT = (TW - 1) * S + K, IHT = (TH - 1) * S + K;
    extern __shared__ __align__(128) uint8_t smem_dw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ float s_gap[TH * 64];  // [output row = warp][lane][2]

    const int tiles_w = (p.OW + TW - 1) / TW;
    const int bx = p.reverse ? gridDim.x - 1 - blockIdx.x : blockIdx.x;
    const int ow0 = (bx % tiles_w) * TW, oh0 = (bx / tiles_w) * TH;
    const int chunk = blockIdx.y, n = p.reverse ? gridDim.z - 1 - blockIdx.z : blockIdx.z;
    uint8_t* tile = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dw) + 127) & ~uintptr_t(127));

    if (threadIdx.x == 0) {
        tc::mbar_init(&bar, 1);
        tc::mbar_fence_init();
        tc::fence_proxy_async();
        tc::mbar_expect_tx(&bar, static_cast<uint32_t>(IWT * IHT * 128));
        tc::tma_load_4d(tile, &tmX, &bar, chunk * p.CB, ow0 * S - PAD, oh0 * S - PAD, n);
    }
    if (p.gap_sum) {
        s_gap[threadIdx.x] = 0.f;
        s_gap[threadIdx.x + 256] = 0.f;
    }
    __syncthreads();

    const int cw = min(p.CB, p.C - chunk * p.CB);  // channels of this chunk (multiple of 8)
    // columns per lane: as many column groups as fit into the 32 lanes (power of two)
    if (cw > 32) dw_row<K, S, 16, T>(p, tile, &bar, s_gap, cw, chunk, n, oh0, ow0);
    else if (cw > 16) dw_row<K, S, 8, T>(p, tile, &bar, s_gap, cw, chunk, n, oh0, ow0);
    else if (cw > 8) dw_row<K, S, 4, T>(p, tile, &bar, s_gap, cw, chunk, n, oh0, ow0);
    else dw_row<K, S, 2, T>(p, tile, &bar, s_gap, cw, chunk, n, oh0, ow0);

    if (p.gap_sum) {
        // Deterministic pooling sums: fixed-order fp32 sum over the rows / column groups of this CTA, then ONE 64-bit
        // INTEGER atomic per channel (fixed point, 2^-24): integer addition is associative, so the total does not depend
        // on the order in which the CTAs arrive -- bit-reproducible without tickets, fences or a second pass.
        __syncthreads();
        if (threadIdx.x < cw) {
            const int lanes_px = cw >> 1, ng = cw > 32 ? 1 : cw > 16 ? 2 : cw > 8 ? 4 : 8;
            const int cl = threadIdx.x >> 1, hi = threadIdx.x & 1;
            float sum = 0.f;
            for (int r = 0; r < TH; ++r)
                for (int g = 0; g < ng; ++g) sum += s_gap[r * 64 + (g * lanes_px + cl) * 2 + hi];
            atomicAdd(reinterpret_cast<unsigned long long*>(p.gap_sum + static_cast<long long>(n) * p.C + chunk * p.CB + threadIdx.x),
                      static_cast<unsigned long long>(__float2ll_rn(sum * CABINET_GAP_FIXED_ONE)));
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Fused no-expand inverted-residual block (reference: src/models/mobilenetv3.py:110-125,154-159 with inp == hidden,
// no SE, stride 1, identity): y = x + W2 * act(dw3x3(x) + b1) + b2 for C <= 32 channels (Large f1: C = 16 at 1/2
// resolution, the two largest-area tensors of the backbone).  The input patch (+halo) is staged once by TMA; the
// depthwise result stays in shared memory (fp32), the tiny C x C pointwise runs on the CUDA cores and the residual
// comes from the centre of the staged patch: one HBM read + one HBM write instead of five tensor passes.
struct Mb1Params {
    int C, OH, OW, act;
    const float* w_dw;   // [9][C]
    const float* b_dw;   // [C]
    const float* w_pw;   // [C][C] (cout, cin)
    const float* b_pw;   // [C]
    bf16* y;
    long long ldy;
};

constexpr int MB_TH = 16, MB_TW = 32;  // output patch of the fused block kernel (512 pixels)

template <int C>
__global__ void __launch_bounds__(256)
mbconv1_fused_kernel(const __grid_constant__ CUtensorMap tmX, const Mb1Params p) {
    constexpr int K = 3, PAD = 1;
    constexpr int IWT = MB_TW + 2, IHT = MB_TH + 2;
    constexpr int PITCH = C * 2;            // staged pixel pitch in bytes (TMA box = exactly C channels)
    constexpr int LANES_PX = C / 2;         // lanes per pixel (channel pairs)
    extern __shared__ __align__(128) uint8_t smem_dw[];
    __shared__ __align__(8) uint64_t bar;
    const int tiles_w = (p.OW + MB_TW - 1) / MB_TW;
    const int ow0 = (blockIdx.x % tiles_w) * MB_TW, oh0 = (blockIdx.x / tiles_w) * MB_TH;
    const int n = blockIdx.z;
    uint8_t* tile = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_dw) + 127) & ~uintptr_t(127));
    constexpr bool MMA = C >= 16;  // pointwise on mma.sync (bf16 hidden tile) / on the CUDA cores (fp32 hidden tile)
    uint8_t* hs_raw = tile + ((IWT * IHT * PITCH + 127) & ~127);
    float* hs = reinterpret_cast<float*>(hs_raw);  // [512 px][C] depthwise output

    if (threadIdx.x == 0) {
        tc::mbar_init(&bar, 1);
        tc::mbar_fence_init();
        tc::fence_proxy_async();
        tc::mbar_expect_tx(&bar, static_cast<uint32_t>(IWT * IHT * PITCH));
        tc::tma_load_4d(tile, &tmX, &bar, 0, ow0 - PAD, oh0 - PAD, n);
    }
    __syncthreads();
    // ---- phase 1: depthwise 3x3 + bias + act.  A warp covers CW = 32 / LANES_PX adjacent columns x all channel pairs
    // (one contiguous 128-byte line of the staged patch per LDS: conflict-free; column GROUPS side by side in a warp
    // would sit 256 B apart = the same banks, a 4-way conflict) and slides DOWN 8 output rows: 10 x 3 loads feed
    // 8 x 9 packed FMAs per thread.
    {
        constexpr int CW = 32 / LANES_PX;            // columns per warp
        constexpr int CGROUPS = MB_TW / CW;          // column groups per tile row
        constexpr int ROWS = 8;                      // output rows per thread
        constexpr int WITEMS = CGROUPS * (MB_TH / ROWS);
        static_assert(MB_TW % CW == 0 && MB_TH % ROWS == 0, "tile shape");
        float2 w[K * K];
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const int cl = lane % LANES_PX, j = lane / LANES_PX;
        const int c0 = cl * 2;
#pragma unroll
        for (int t = 0; t < K * K; ++t) w[t] = __ldg(reinterpret_cast<const float2*>(p.w_dw + t * C + c0));
        const float2 b = __ldg(reinterpret_cast<const float2*>(p.b_dw + c0));
        tc::mbar_wait(&bar, 0);
        for (int wi = warp; wi < WITEMS; wi += 8) {
            const int col = (wi % CGROUPS) * CW + j, row0 = (wi / CGROUPS) * ROWS;
            float2 acc[ROWS];
#pragma unroll
            for (int r = 0; r < ROWS; ++r) acc[r] = b;
            const uint32_t base = tc::smem_u32(tile) + (row0 * IWT + col) * PITCH + cl * 4;
#pragma unroll
            for (int sy = 0; sy < ROWS + K - 1; ++sy)
#pragma unroll
                for (int kx = 0; kx < K; ++kx) {
                    uint32_t raw;
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(raw) : "r"(base + (sy * IWT + kx) * PITCH));
                    const float2 xv = cab_unpack2<bf16>(raw);
#pragma unroll
                    for (int r = 0; r < ROWS; ++r) {
                        const int ky = sy - r;
                        if (ky >= 0 && ky < K) cab_ffma2(acc[r], xv, w[ky * K + kx]);
                    }
                }
            cab_act_vec<2 * ROWS>(&acc[0].x, p.act);
            if constexpr (MMA) {
                const uint32_t hb = tc::smem_u32(hs_raw) + ((row0 * MB_TW + col) * C + c0) * 2;
#pragma unroll
                for (int r = 0; r < ROWS; ++r) {
                    const __nv_bfloat162 hv = __floats2bfloat162_rn(acc[r].x, acc[r].y);
                    asm volatile("st.shared.u32 [%0], %1;" ::"r"(hb + r * MB_TW * C * 2), "r"(*reinterpret_cast<const uint32_t*>(&hv)) : "memory");
                }
            } else {
#pragma unroll
                for (int r = 0; r < ROWS; ++r)
                    *reinterpret_cast<float2*>(hs + ((row0 + r) * MB_TW + col) * C + c0) = acc[r];
            }
        }
    }
    __syncthreads();
    // ---- phase 2: pointwise C -> C (+ bias + residual)
    if constexpr (MMA) {
        // warp-level tensor-core GEMM (mma.sync.m16n8k16, bf16 -> fp32): per 16 pixels one ldmatrix.x4 per 16 input
        // channels and C/8 MMAs; the weight fragments live in registers for the whole CTA.  A TMEM round trip
        // (tcgen05) does not pay for K = C = 16.
        constexpr int KS = C / 16, NT = C / 8;
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const int gq = lane >> 2, tq = lane & 3;  // fragment row group / column pair
        uint32_t bfrag[KS][NT][2];
#pragma unroll
        for (int ks = 0; ks < KS; ++ks)
#pragma unroll
            for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const float* wp = p.w_pw + (nt * 8 + gq) * C + ks * 16 + hh * 8 + tq * 2;  // B[k][n] = W[n][k]
                    const __nv_bfloat162 wv = __floats2bfloat162_rn(__ldg(wp), __ldg(wp + 1));
                    bfrag[ks][nt][hh] = *reinterpret_cast<const uint32_t*>(&wv);
                }
        float2 bias[NT];
#pragma unroll
        for (int nt = 0; nt < NT; ++nt) bias[nt] = __ldg(reinterpret_cast<const float2*>(p.b_pw + nt * 8 + tq * 2));
        const uint32_t hbase = tc::smem_u32(hs_raw);
        // ldmatrix.x4: lane -> (matrix = lane / 8, row = lane % 8); matrices: rows 0-7 / 8-15 x k 0-7 / 8-15
        const uint32_t lm_off = ((lane & 7) + ((lane >> 3) & 1) * 8) * (C * 2) + (lane >> 4) * 16;
        for (int mt = warp; mt < MB_TH * MB_TW / 16; mt += 8) {
            const int px0 = mt * 16;  // 16 consecutive pixels of one tile row (MB_TW is a multiple of 16)
            float acc[NT][4];
#pragma unroll
            for (int nt = 0; nt < NT; ++nt) {
                acc[nt][0] = bias[nt].x; acc[nt][1] = bias[nt].y; acc[nt][2] = bias[nt].x; acc[nt][3] = bias[nt].y;
            }
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                uint32_t a0, a1, a2, a3;
                asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
                             : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3)
                             : "r"(hbase + px0 * (C * 2) + lm_off + ks * 32));
#pragma unroll
                for (int nt = 0; nt < NT; ++nt)
                    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                                 : "+f"(acc[nt][0]), "+f"(acc[nt][1]), "+f"(acc[nt][2]), "+f"(acc[nt][3])
                                 : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(bfrag[ks][nt][0]), "r"(bfrag[ks][nt][1]));
            }
            const int row = px0 / MB_TW, colb = px0 % MB_TW;
            const int oh = oh0 + row;
            if (oh >= p.OH) continue;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {  // fragment rows gq and gq + 8
                const int col = colb + gq + hh * 8;
                if (ow0 + col >= p.OW) continue;
                const uint32_t res = tc::smem_u32(tile) + ((row + PAD) * IWT + col + PAD) * PITCH + tq * 4;
                bf16* yp = p.y + ((static_cast<long long>(n) * p.OH + oh) * p.OW + ow0 + col) * p.ldy + tq * 2;
#pragma unroll
                for (int nt = 0; nt < NT; ++nt) {
                    uint32_t raw;  // residual: the block input at the same pixel (centre of the staged patch)
                    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(raw) : "r"(res + nt * 16));
                    const float2 rv = cab_unpack2<bf16>(raw);
                    const float o0 = acc[nt][2 * hh] + rv.x;
                    const float o1 = acc[nt][2 * hh + 1] + rv.y;
                    *reinterpret_cast<__nv_bfloat162*>(yp + nt * 8) = __floats2bfloat162_rn(o0, o1);
                }
            }
        }
    } else {
        // CUDA-core pointwise; work item = (pixel, cout pair)
        constexpr int PAIRS = C / 2;
        const int cp = threadIdx.x % PAIRS;
        const int co = cp * 2;
        float w0[C], w1[C];
#pragma unroll
        for (int ci = 0; ci < C; ++ci) {
            w0[ci] = __ldg(p.w_pw + co * C + ci);
            w1[ci] = __ldg(p.w_pw + (co + 1) * C + ci);
        }
        const float2 b = __ldg(reinterpret_cast<const float2*>(p.b_pw + co));
        for (int px = threadIdx.x / PAIRS; px < MB_TH * MB_TW; px += 256 / PAIRS) {
            const int row = px / MB_TW, col = px % MB_TW;
            const int oh = oh0 + row, ow = ow0 + col;
            if (oh >= p.OH || ow >= p.OW) continue;
            const float* h = hs + px * C;
            float o0 = b.x, o1 = b.y;
#pragma unroll
            for (int ci = 0; ci < C; ci += 4) {
                const float4 hv = *reinterpret_cast<const float4*>(h + ci);
                o0 = fmaf(hv.x, w0[ci], o0); o0 = fmaf(hv.y, w0[ci + 1], o0);
                o0 = fmaf(hv.z, w0[ci + 2], o0); o0 = fmaf(hv.w, w0[ci + 3], o0);
                o1 = fmaf(hv.x, w1[ci], o1); o1 = fmaf(hv.y, w1[ci + 1], o1);
                o1 = fmaf(hv.z, w1[ci + 2], o1); o1 = fmaf(hv.w, w1[ci + 3], o1);
            }
            uint32_t raw;  // residual: the block input at the same pixel (centre of the staged patch)
            asm volatile("ld.shared.u32 %0, [%1];"
                         : "=r"(raw)
                         : "r"(tc::smem_u32(tile) + ((row + PAD) * IWT + col + PAD) * PITCH + co * 2));
            const float2 rv = cab_unpack2<bf16>(raw);
            o0 += rv.x;
            o1 += rv.y;
            *reinterpret_cast<__nv_bfloat162*>(p.y + ((static_cast<long long>(n) * p.OH + oh) * p.OW + ow) * p.ldy + co) =
                __floats2bfloat162_rn(o0, o1);
        }
    }
}

template <int K, int S, typename T>
int launch(const CUtensorMap& tm, const DwParams& p, int N, int n_chunks, cudaStream_t s) {
    constexpr int IWT = (TW - 1) * S + K, IHT = (TH - 1) * S + K;
    const size_t smem = static_cast<size_t>(IWT) * IHT * 128 + 128;
    static bool attr_set = false;
    if (!attr_set) {
        CAB_CUDA(cudaFuncSetAttribute(dwconv_tma_kernel<K, S, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
        attr_set = true;
    }
    const int tiles = ((p.OW + TW - 1) / TW) * ((p.OH + TH - 1) / TH);
    dim3 grid(tiles, n_chunks, N);
    dwconv_tma_kernel<K, S, T><<<grid, 32 * TH, smem, s>>>(tm, p);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

}  // namespace

extern "C" int cabinet_mbconv_noexpand_fused(const void* x, long long ldx, const float* w_dw, const float* b_dw,
                                             const float* w_pw, const float* b_pw, void* y, long long ldy, int N,
                                             int H, int W, int C, int act, cabinet_stream_t stream) {
    CAB_REQUIRE(x && w_dw && b_dw && w_pw && b_pw && y, "mbconv_noexpand_fused: null pointer");
    CAB_REQUIRE(C >= 8 && C <= 32 && (C & (C - 1)) == 0, "mbconv_noexpand_fused: C must be 8, 16 or 32 (got %d)", C);
    CAB_REQUIRE(ldx % 8 == 0 && ldy % 8 == 0 && ldx >= C && ldy >= C && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(y) & 3) == 0 && N <= 65535,
                "mbconv_noexpand_fused: alignment");
    if (N == 0) return CABINET_OK;
    CUtensorMap tm;
    const uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    const uint64_t strides[3] = {(uint64_t)ldx * 2, (uint64_t)ldx * 2 * W, (uint64_t)ldx * 2 * W * H};
    const uint32_t box[4] = {(uint32_t)C, (uint32_t)(MB_TW + 2), (uint32_t)(MB_TH + 2), 1};
    int rc = cab_make_tmap_bf16(&tm, x, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    Mb1Params p;
    p.C = C; p.OH = H; p.OW = W; p.act = act; p.w_dw = w_dw; p.b_dw = b_dw; p.w_pw = w_pw; p.b_pw = b_pw;
    p.y = reinterpret_cast<bf16*>(y); p.ldy = ldy;
    const size_t smem = static_cast<size_t>(MB_TW + 2) * (MB_TH + 2) * C * 2 + 128 +
                        static_cast<size_t>(MB_TH) * MB_TW * C * (C >= 16 ? 2 : 4) + 128;  // bf16 / fp32 hidden tile
    const int tiles = ((W + MB_TW - 1) / MB_TW) * ((H + MB_TH - 1) / MB_TH);
    dim3 grid(tiles, 1, N);
    static bool attr_done = false;
    if (!attr_done) {
        CAB_CUDA(cudaFuncSetAttribute(mbconv1_fused_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
        CAB_CUDA(cudaFuncSetAttribute(mbconv1_fused_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
        CAB_CUDA(cudaFuncSetAttribute(mbconv1_fused_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
        attr_done = true;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (C == 8) mbconv1_fused_kernel<8><<<grid, 256, smem, st>>>(tm, p);
    else if (C == 16) mbconv1_fused_kernel<16><<<grid, 256, smem, st>>>(tm, p);
    else mbconv1_fused_kernel<32><<<grid, 256, smem, st>>>(tm, p);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_dwconv_tma(const void* x, long long ldx, const float* w, const float* bias, void* y,
                                  long long ldy, int N, int H, int W, int C, int k, int stride, int OH, int OW, int act,
                                  long long* gap_sum, cabinet_stream_t stream) {
    return cabinet_dwconv_tma_dt(x, ldx, w, bias, y, ldy, N, H, W, C, k, stride, OH, OW, act, gap_sum, CABINET_BF16, stream);
}

extern "C" int cabinet_dwconv_tma_dt(const void* x, long long ldx, const float* w, const float* bias, void* y,
                                     long long ldy, int N, int H, int W, int C, int k, int stride, int OH, int OW, int act,
                                     long long* gap_sum, int op_dtype, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("dwconv_tma", op_dtype, CAB_DT_BF16 | CAB_DT_F16);
    CAB_REQUIRE(x && w && bias && y, "dwconv_tma: null pointer");
    const int reverse = (act & CABINET_CONV_REVERSE_TILES) ? 1 : 0;
    act &= ~CABINET_CONV_REVERSE_TILES;
    CAB_REQUIRE((k == 3 || k == 5) && (stride == 1 || stride == 2), "dwconv_tma: k must be 3|5 and stride 1|2");
    CAB_REQUIRE(C > 0 && C % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && ldx >= C && ldy >= C &&
                    (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(w) & 15) == 0 && (reinterpret_cast<uintptr_t>(bias) & 15) == 0,
                "dwconv_tma: C/ldx/ldy must be multiples of 8 and pointers 16-byte aligned");
    CAB_REQUIRE(OH == (H + 2 * ((k - 1) / 2) - k) / stride + 1 && OW == (W + 2 * ((k - 1) / 2) - k) / stride + 1,
                "dwconv_tma: inconsistent output size");
    CAB_REQUIRE(N <= 65535, "dwconv_tma: N exceeds grid limits");
    if (N == 0) return CABINET_OK;
    DwParams p;
    const int n_chunks = (C + 63) / 64;
    p.C = C; p.OH = OH; p.OW = OW; p.act = act; p.w = w; p.bias = bias; p.reverse = reverse;
    // balanced chunks (multiples of 8 channels, <= 64): 72 -> 40 + 32, 200 -> 56 + 56 + 56 + 32.  A ragged 8-channel
    // tail would pack 8 column groups into a warp whose rows sit a multiple of 128 B apart: an 8-way bank conflict
    // that makes the tail cost more than a full chunk.  The TMA box stays 64 channels wide.
    p.CB = ((C + n_chunks - 1) / n_chunks + 7) / 8 * 8;
    p.y = y; p.ldy = ldy; p.gap_sum = gap_sum;
    const int IWT = (TW - 1) * stride + k, IHT = (TH - 1) * stride + k;
    CUtensorMap tm;
    const uint64_t dims[4] = {(uint64_t)C, (uint64_t)W, (uint64_t)H, (uint64_t)N};
    const uint64_t strides[3] = {(uint64_t)ldx * 2, (uint64_t)ldx * 2 * W, (uint64_t)ldx * 2 * W * H};
    const uint32_t box[4] = {64, (uint32_t)IWT, (uint32_t)IHT, 1};
    int rc = cab_make_tmap_2b(&tm, op_dtype, x, 4, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                              CU_TENSOR_MAP_SWIZZLE_NONE);
    if (rc) return rc;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CAB_DISPATCH_DT_HALF(op_dtype, T,
                         if (k == 3 && stride == 1) return launch<3, 1, T>(tm, p, N, n_chunks, s);
                         if (k == 3 && stride == 2) return launch<3, 2, T>(tm, p, N, n_chunks, s);
                         if (k == 5 && stride == 1) return launch<5, 1, T>(tm, p, N, n_chunks, s);
                         return launch<5, 2, T>(tm, p, N, n_chunks, s));
    return CABINET_OK;
}
