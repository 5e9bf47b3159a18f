// Data gradient of the two stride-2 stems into the fp32 NCHW network input (cabinet_stem_dgrad):
//   dx[n][c][iy][ix] = sum over both stems of sum_{co, ky, kx} dy[n][oy][ox][co] * w[co][c][ky][kx],  iy = 2 oy - pad + ky
// for sb.conv1 (7x7 / pad 3, 64 outputs) and mobile.features.0.0 (3x3 / pad 1, 16 outputs).
//
// Input pixel (iy, ix) = (2 ay + py, 2 ax + px) reads dy[ay + vy][ax + vx] through the tap ky = py + pad - 2 vy,
// kx = px + pad - 2 vx: the four parity classes (py, px) of one "class pixel" (ay, ax) read the SAME dy pixels, each
// with its own tap.  So for a dy view (vy, vx) -- 4 x 4 of them for the 7x7 stem, vy, vx in -1..2, and 2 x 2 for the 3x3
// stem, vy, vx in 0..1 -- one GEMM serves all four classes:
//   D[class pixels][cls * 3 + c] += A_view[class pixels][co] * B_view[cls * 3 + c][co],  B = w[co][c][ky][kx] (0 where
//   the class has no tap at that view)
// 2-byte dy: on the tensor cores (tcgen05.mma kind::f16, M = 128 class pixels of one class row, N = 16 = 4 classes x 3
// channels + 4 zero rows, K = 64 (7x7, four K = 16 steps) or 16 (3x3, one step) per view): 68 MMAs per tile, both stems
// into ONE TMEM accumulator, so dx is written once, without atomics and in a fixed order (bit-reproducible).
// A persistent CTA walks a column strip of 128 class columns down its rows.  Tile row ay reads dy rows ay - 1 .. ay + 2,
// kept in a ring of six shared-memory row slots (132 pixels: the strip and its halo, both stems' channels): each tile
// loads ONE new row, two tiles ahead (cp.async, zero fill outside the map), under the MMAs of the tiles before it, and every view is a shifted
// no-swizzle descriptor into a slot (A rows = consecutive pixels 16 bytes apart).  The filters are read and rounded to the
// operand type once per CTA and call (34 KB of B), so a replayed graph sees the weights the optimizer just wrote.  The
// epilogue writes both column parities of a class pixel, so a warp's stores cover whole lines.
// fp32 dy (the parity mode): the same sums on the CUDA cores.
#include "tc_common.cuh"

namespace {

constexpr int SD_THREADS = 128;             // 4 warps: warp w reads TMEM lanes 32w .. 32w + 31 = tile columns
constexpr int SD_M = 128;                   // class columns per tile (one class row)
constexpr int SD_N = 16;                    // 4 parity classes x 3 input channels, zero padded
constexpr int HALO = SD_M + 4;              // slot pixels: class columns ax0 - 1 .. ax0 + 130
constexpr int CH_STRIDE = HALO * 16;        // bytes between the 8-channel chunks of a slot (the descriptor's LBO)
constexpr int SLOT7 = 8 * CH_STRIDE;        // 64 channels of the 7x7 stem's dy
constexpr int SLOT_BYTES = SLOT7 + 2 * CH_STRIDE;   // + 16 channels of the 3x3 stem's dy
constexpr int NSLOTS = 6;                   // rows ay - 1 .. ay + 2 in use, ay + 3 and ay + 4 loading
constexpr int B7_VIEW = 8 * 256, B3_VIEW = 2 * 256;   // [chunk][16 rows][16 B] per view
constexpr int B_BYTES = 16 * B7_VIEW + 4 * B3_VIEW;
constexpr int SD_SMEM = NSLOTS * SLOT_BYTES + B_BYTES + 128;
constexpr int C7 = 64, C3 = 16;             // output channels of the two stems

struct StemDgradParams {
    const void* dy7;
    const void* dy3;
    long long ld7, ld3;
    const float* w7;   // [64][3][7][7]
    const float* w3;   // [16][3][3][3]
    float* dx;         // [N][3][H][W]
    int N, H, W, OH, OW;
    int strips;        // column strips of 128 class columns per image
    int rows_per_cta;  // consecutive (strip, class row) tiles of one CTA
    long long tiles;   // N * strips * OH
};

// K-major operand without swizzle: 8-row x 16-byte core matrices; LBO = bytes between core matrices adjacent in K,
// SBO = bytes between core matrices adjacent in M / N.
__device__ __forceinline__ uint64_t desc_nosw(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
    return static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4) | (static_cast<uint64_t>(lbo >> 4) << 16) |
           (static_cast<uint64_t>(sbo >> 4) << 32) | (static_cast<uint64_t>(1) << 46);
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_but_newest() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

__device__ __forceinline__ int slot_of(int y) { return ((y % NSLOTS) + NSLOTS) % NSLOTS; }

// dy row y (both stems) of image n, class columns ax0 - 1 .. ax0 + 130 -> its ring slot; zero outside the map.  One
// cp.async group per call, empty without ``load``: a tile waits for all groups but the newest.
template <typename T>
__device__ __forceinline__ void load_row(const StemDgradParams& p, uint32_t slots, int n, int y, int ax0, bool load = true) {
    const uint32_t dst0 = slots + slot_of(y) * SLOT_BYTES;
    const bool row_ok = y >= 0 && y < p.OH;
    const long long row = (static_cast<long long>(n) * p.OH + (row_ok ? y : 0)) * p.OW;
    for (int i = threadIdx.x; load && i < HALO * 10; i += SD_THREADS) {
        const bool big = i < HALO * 8;
        const int q = big ? i : i - HALO * 8;
        const int c = big ? q >> 3 : q >> 1, j = big ? q & 7 : q & 1;   // pixel-major: a warp reads whole pixels
        const int x = ax0 - 1 + c;
        const void* base = big ? p.dy7 : p.dy3;
        const bool ok = base && row_ok && x >= 0 && x < p.OW;
        const T* src = reinterpret_cast<const T*>(base ? base : p.dx) +
                       (ok ? (row + x) * (big ? p.ld7 : p.ld3) + j * 8 : 0);
        cp_async16(dst0 + (big ? 0 : SLOT7) + j * CH_STRIDE + c * 16, src, ok ? 16u : 0u);
    }
    cp_async_commit();
}

template <typename T>
__global__ void __launch_bounds__(SD_THREADS, 1) stem_dgrad_tc_kernel(const __grid_constant__ StemDgradParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t acc_bar[2];
    __shared__ uint32_t tmem_slot;

    const uint32_t slots = (tc::smem_u32(smem_raw) + 127) & ~127u;
    const uint32_t sB = slots + NSLOTS * SLOT_BYTES;
    const int tid = threadIdx.x, warp = tid >> 5;

    if (tid == 0) {
        tc::mbar_init(&acc_bar[0], 1);
        tc::mbar_init(&acc_bar[1], 1);
        tc::mbar_fence_init();
    }
    __syncwarp();
    if (warp == 0) tc::tmem_alloc(&tmem_slot, 32);

    // B: per view, rows n = cls * 3 + c (cls = py * 2 + px) of w[co][c][ky][kx], ky = py + pad - 2 vy (0 where the class
    // has no tap there), the filters rounded to T on every call
    for (int i = tid; i < 16 * 16 * 8 + 4 * 16 * 2; i += SD_THREADS) {
        const bool big = i < 16 * 16 * 8;
        const int q = big ? i : i - 16 * 16 * 8;
        const int v = big ? q >> 7 : q >> 5, r = q & 15, j = big ? (q >> 4) & 7 : (q >> 4) & 1;
        const int k = big ? 7 : 3, pad = big ? 3 : 1, nv = big ? 4 : 2, v0 = big ? -1 : 0;
        const int cls = r / 3, c = r - cls * 3;
        const int ky = (cls >> 1) + pad - 2 * (v / nv + v0), kx = (cls & 1) + pad - 2 * (v % nv + v0);
        const float* w = big ? p.w7 : p.w3;
        const bool ok = r < 12 && (big ? p.dy7 : p.dy3) && ky >= 0 && ky < k && kx >= 0 && kx < k;
        float f[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) f[e] = ok ? __ldg(w + (((j * 8 + e) * 3 + c) * k + ky) * k + kx) : 0.f;
        Vec16<T> vv;
        vv.pack(f);
        tc::sts128(sB + (big ? v * B7_VIEW : 16 * B7_VIEW + v * B3_VIEW) + j * 256 + (r >> 3) * 128 + (r & 7) * 16, vv.raw);
    }
    tc::fence_proxy_async();
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t idesc = tc::make_idesc<T>(SD_M, SD_N);
    const long long plane = static_cast<long long>(p.H) * p.W;

    // epilogue of one tile: TMEM row tid = class column ax0 + tid -> 4 classes x 3 channels of dx
    auto epilogue = [&](uint32_t t, int n, int ay, int ax0) {
        tc::mbar_wait(&acc_bar[t & 1], (t >> 1) & 1);
        tc::tc_fence_after();
        uint32_t r[16];
        tc::tmem_ld16(tmem + (t & 1) * SD_N + (static_cast<uint32_t>(warp * 32) << 16), r);
        tc::tmem_ld_wait();
        tc::tc_fence_before();
        const int ax = ax0 + tid;
        float* o = p.dx + static_cast<long long>(n) * 3 * plane;
#pragma unroll
        for (int cls = 0; cls < 4; ++cls) {
            const int iy = 2 * ay + (cls >> 1), ix = 2 * ax + (cls & 1);
            if (iy < p.H && ix < p.W) {
#pragma unroll
                for (int c = 0; c < 3; ++c) o[c * plane + static_cast<long long>(iy) * p.W + ix] = __uint_as_float(r[cls * 3 + c]);
            }
        }
    };

    uint32_t t = 0;   // tiles of this CTA: accumulator stage t & 1
    long long g = static_cast<long long>(blockIdx.x) * p.rows_per_cta;
    const long long g_end = min(g + p.rows_per_cta, p.tiles);
    while (g < g_end) {
        // a segment: consecutive class rows ay0 .. ay1 - 1 of one column strip
        const long long strip = g / p.OH;
        const int ay0 = static_cast<int>(g - strip * p.OH);
        const int ay1 = static_cast<int>(min(static_cast<long long>(p.OH), ay0 + (g_end - g)));
        const int n = static_cast<int>(strip / p.strips), ax0 = static_cast<int>(strip % p.strips) * SD_M;
        for (int y = ay0 - 1; y <= ay0 + 3; ++y) load_row<T>(p, slots, n, y, ax0);
        for (int ay = ay0; ay < ay1; ++ay, ++t) {
            cp_async_wait_but_newest();   // rows up to ay + 2 are in; ay + 3 may still be arriving
            tc::fence_proxy_async();
            __syncthreads();
            if (tid == 0) {
                tc::tc_fence_after();
                const uint32_t d = tmem + (t & 1) * SD_N;
                uint32_t acc = 0;
                if (p.dy7) {
                    for (int v = 0; v < 16; ++v) {
                        const uint32_t a = slots + slot_of(ay + (v >> 2) - 1) * SLOT_BYTES + (v & 3) * 16;
                        const uint32_t b = sB + v * B7_VIEW;
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk, acc = 1)
                            tc::umma_bf16(d, desc_nosw(a + 2 * kk * CH_STRIDE, CH_STRIDE, 128), desc_nosw(b + kk * 512, 256, 128),
                                          idesc, acc);
                    }
                }
                if (p.dy3) {
                    for (int v = 0; v < 4; ++v, acc = 1) {
                        const uint32_t a = slots + slot_of(ay + (v >> 1)) * SLOT_BYTES + SLOT7 + ((v & 1) + 1) * 16;
                        tc::umma_bf16(d, desc_nosw(a, CH_STRIDE, 128), desc_nosw(sB + 16 * B7_VIEW + v * B3_VIEW, 256, 128), idesc,
                                      acc);
                    }
                }
                tc::umma_commit(&acc_bar[t & 1]);
            }
            if (ay > ay0) epilogue(t - 1, n, ay - 1, ax0);   // under this tile's MMAs; frees the slot of row ay - 2
            load_row<T>(p, slots, n, ay + 4, ax0, ay + 2 < ay1);
        }
        epilogue(t - 1, n, ay1 - 1, ax0);
        g += ay1 - ay0;
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, 32);
    }
}

// fp32 dy: one thread per input pixel, the taps of its parity class (7x7 stem, then 3x3), channels in ascending
// order within a tap.  Filters in shared memory as [tap][co][3].
__global__ void __launch_bounds__(256) stem_dgrad_f32_kernel(const __grid_constant__ StemDgradParams p) {
    __shared__ float s7[49 * C7 * 3];
    __shared__ float s3[9 * C3 * 3];
    for (int i = threadIdx.x; i < 49 * C7 * 3; i += blockDim.x) {
        const int c = i % 3, co = (i / 3) % C7, tap = i / (3 * C7);
        s7[i] = p.dy7 ? p.w7[(co * 3 + c) * 49 + tap] : 0.f;
    }
    for (int i = threadIdx.x; i < 9 * C3 * 3; i += blockDim.x) {
        const int c = i % 3, co = (i / 3) % C3, tap = i / (3 * C3);
        s3[i] = p.dy3 ? p.w3[(co * 3 + c) * 9 + tap] : 0.f;
    }
    __syncthreads();
    const long long plane = static_cast<long long>(p.H) * p.W;
    const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= p.N * plane) return;
    const int n = static_cast<int>(q / plane);
    const int rem = static_cast<int>(q - n * plane);
    const int iy = rem / p.W, ix = rem % p.W;
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f;
    for (int stem = 0; stem < 2; ++stem) {
        const float* dy = reinterpret_cast<const float*>(stem == 0 ? p.dy7 : p.dy3);
        if (!dy) continue;
        const int k = stem == 0 ? 7 : 3, pad = stem == 0 ? 3 : 1, cout = stem == 0 ? C7 : C3;
        const long long ld = stem == 0 ? p.ld7 : p.ld3;
        const float* sw = stem == 0 ? s7 : s3;
        for (int ky = (iy + pad) & 1; ky < k; ky += 2) {
            const int oy = (iy + pad - ky) >> 1;
            if (oy < 0 || oy >= p.OH) continue;
            for (int kx = (ix + pad) & 1; kx < k; kx += 2) {
                const int ox = (ix + pad - kx) >> 1;
                if (ox < 0 || ox >= p.OW) continue;
                const float4* d = reinterpret_cast<const float4*>(dy + ((static_cast<long long>(n) * p.OH + oy) * p.OW + ox) * ld);
                const float* w = sw + (ky * k + kx) * cout * 3;
                for (int c4 = 0; c4 < cout / 4; ++c4) {
                    const float4 v = __ldg(d + c4);
                    const float* we = w + c4 * 12;
                    acc0 = fmaf(v.x, we[0], acc0); acc1 = fmaf(v.x, we[1], acc1); acc2 = fmaf(v.x, we[2], acc2);
                    acc0 = fmaf(v.y, we[3], acc0); acc1 = fmaf(v.y, we[4], acc1); acc2 = fmaf(v.y, we[5], acc2);
                    acc0 = fmaf(v.z, we[6], acc0); acc1 = fmaf(v.z, we[7], acc1); acc2 = fmaf(v.z, we[8], acc2);
                    acc0 = fmaf(v.w, we[9], acc0); acc1 = fmaf(v.w, we[10], acc1); acc2 = fmaf(v.w, we[11], acc2);
                }
            }
        }
    }
    float* o = p.dx + static_cast<long long>(n) * 3 * plane + rem;
    o[0] = acc0;
    o[plane] = acc1;
    o[2 * plane] = acc2;
}

}  // namespace

extern "C" int cabinet_stem_dgrad(const void* dy7, long long ld7, const void* dy3, long long ld3, int dtype, const float* w7,
                                  const float* w3, float* dx, int N, int H, int W, int OH, int OW, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("stem_dgrad", dtype, CAB_DT_ALL);
    CAB_REQUIRE(dy7 || dy3, "stem_dgrad: both output gradients are NULL");
    CAB_REQUIRE(dx, "stem_dgrad: NULL dx");
    CAB_REQUIRE(N >= 0 && H >= 1 && W >= 1 && OH == (H - 1) / 2 + 1 && OW == (W - 1) / 2 + 1,
                "stem_dgrad: bad sizes (N %d, H %d, W %d, OH %d, OW %d: OH = (H - 1) / 2 + 1 and OW = (W - 1) / 2 + 1)", N, H,
                W, OH, OW);
    const int vec = 16 / cab_dtype_size(dtype);
    CAB_REQUIRE(!dy7 || (w7 && ld7 >= C7 && ld7 % vec == 0 && (reinterpret_cast<uintptr_t>(dy7) & 15) == 0),
                "stem_dgrad: the 7x7 stem's gradient needs its filter, ld >= 64, 16-byte aligned pixels");
    CAB_REQUIRE(!dy3 || (w3 && ld3 >= C3 && ld3 % vec == 0 && (reinterpret_cast<uintptr_t>(dy3) & 15) == 0),
                "stem_dgrad: the 3x3 stem's gradient needs its filter, ld >= 16, 16-byte aligned pixels");
    if (N == 0) return CABINET_OK;
    CAB_REQUIRE(static_cast<long long>(N) * 3 * H * W < (1LL << 40), "stem_dgrad: too many pixels");

    StemDgradParams p;
    p.dy7 = dy7; p.dy3 = dy3; p.ld7 = ld7; p.ld3 = ld3; p.w7 = w7; p.w3 = w3; p.dx = dx;
    p.N = N; p.H = H; p.W = W; p.OH = OH; p.OW = OW;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == CABINET_F32) {
        const long long total = static_cast<long long>(N) * H * W;
        CAB_REQUIRE(cab_ceil_div(total, 256) < (1LL << 31), "stem_dgrad: too many pixels");
        stem_dgrad_f32_kernel<<<static_cast<unsigned>(cab_ceil_div(total, 256)), 256, 0, st>>>(p);
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    p.strips = static_cast<int>(cab_ceil_div((W + 1) / 2, SD_M));
    p.tiles = static_cast<long long>(N) * p.strips * OH;
    int dev = 0, sms = 148;
    CAB_CUDA(cudaGetDevice(&dev));
    CAB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const long long per = cab_ceil_div(p.tiles, sms);   // equal shares of tile rows, split at strip ends
    CAB_REQUIRE(per < (1LL << 31), "stem_dgrad: too many pixels");
    p.rows_per_cta = static_cast<int>(per);
    const int grid = static_cast<int>(cab_ceil_div(p.tiles, per));
#define CAB_SD_LAUNCH(T_)                                                                                                 \
    do {                                                                                                                  \
        static bool attr_done = false;                                                                                    \
        if (!attr_done) {                                                                                                 \
            CAB_CUDA(cudaFuncSetAttribute(stem_dgrad_tc_kernel<T_>, cudaFuncAttributeMaxDynamicSharedMemorySize, SD_SMEM)); \
            attr_done = true;                                                                                             \
        }                                                                                                                 \
        stem_dgrad_tc_kernel<T_><<<grid, SD_THREADS, SD_SMEM, st>>>(p);                                                   \
    } while (0)
    if (dtype == CABINET_F16) CAB_SD_LAUNCH(f16);
    else CAB_SD_LAUNCH(bf16);
#undef CAB_SD_LAUNCH
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}
