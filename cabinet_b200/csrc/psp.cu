// Pyramid pooling pieces (src/models/cab.py:46-76): adaptive average pools (1,3,6,8) and the
// [x, up(pool_s)...] 5C-channel concat that feeds the 1x1 `project` GEMM.  The maps here are 1/32 resolution
// (<= 8160 pixels, 128 channels): negligible bytes next to the high-resolution layers.
#include "common.cuh"

namespace {

__device__ __constant__ int kPspSize[4] = {1, 3, 6, 8};
__device__ __constant__ int kPspOffset[4] = {0, 1, 10, 46};  // bin offsets inside the 110-entry table
constexpr int kPspBins = 110;

// Work table of the pooling kernel: large bins (the 1x1 and 3x3 levels) are split into parts of <= `chunk` pixels so
// that every block is short; the parts of one bin go to a scratch area and the part that arrives last (per-bin ticket)
// adds them in part order -- deterministic, no floating-point atomics.
struct PspWork {
    unsigned short bin[256];
    unsigned char part[256], parts[256];
    int n, chunk;
};

__host__ __device__ inline void psp_bin_rect(int bin, int H, int W, int& h0, int& h1, int& w0, int& w1) {
    const int size[4] = {1, 3, 6, 8}, offset[4] = {0, 1, 10, 46};
    int si = 3;
    if (bin < 1) si = 0; else if (bin < 10) si = 1; else if (bin < 46) si = 2;
    const int s = size[si];
    const int local = bin - offset[si];
    const int by = local / s, bx = local % s;
    // ATen adaptive_avg_pool2d bins: [floor(i*H/s), ceil((i+1)*H/s))
    h0 = (by * H) / s; h1 = ((by + 1) * H + s - 1) / s;
    w0 = (bx * W) / s; w1 = ((bx + 1) * W + s - 1) / s;
}

// grid (work items, N); 128 threads = (C / VPT channel vectors) x (pixel lanes), 16-byte loads, four loads in flight
// per thread, shared-memory tree over the pixel lanes.
template <typename T>
__global__ void __launch_bounds__(128)
psp_pool_kernel(const T* __restrict__ x, long long ldx, float* __restrict__ pooled, int H, int W, int C,
                const __grid_constant__ PspWork wk, float* __restrict__ partial, unsigned int* __restrict__ tickets) {
    constexpr int VPT = Vec16<T>::N;  // channels per thread: 8 (bf16) or 4 (fp32)
    extern __shared__ float red[];    // [blockDim.x][VPT]
    const int bin = wk.bin[blockIdx.x], part = wk.part[blockIdx.x], parts = wk.parts[blockIdx.x];
    const int n = blockIdx.y;
    int h0, h1, w0, w1;
    psp_bin_rect(bin, H, W, h0, h1, w0, w1);
    const int bw = w1 - w0, npix = (h1 - h0) * bw;
    const int per = (npix + parts - 1) / parts;
    const int i_beg = part * per, i_end = min(npix, i_beg + per);
    const int CQ = C / VPT;
    const int lanes = blockDim.x / CQ;       // pixel lanes
    const int cq = threadIdx.x % CQ, pl = threadIdx.x / CQ;
    const T* base = x + static_cast<long long>(n) * H * W * ldx + cq * VPT;
    float acc[VPT];
#pragma unroll
    for (int j = 0; j < VPT; ++j) acc[j] = 0.f;
    if (pl < lanes) {
        for (int i0 = i_beg + pl; i0 < i_end; i0 += 4 * lanes) {
            Vec16<T> v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * lanes;
                if (i < i_end) v[u].load(base + (static_cast<long long>(h0 + i / bw) * W + (w0 + i % bw)) * ldx);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (i0 + u * lanes < i_end) {
                    float f[VPT];
                    v[u].unpack(f);
#pragma unroll
                    for (int j = 0; j < VPT; ++j) acc[j] += f[j];
                }
            }
        }
    }
    float* mine = red + threadIdx.x * VPT;
    int span = 1;
    while (span < lanes) span <<= 1;
    for (int off = span >> 1; off >= 1; off >>= 1) {
#pragma unroll
        for (int j = 0; j < VPT; ++j) mine[j] = acc[j];
        __syncthreads();
        if (pl < off && pl + off < lanes) {
            const float* o = red + ((pl + off) * CQ + cq) * VPT;
#pragma unroll
            for (int j = 0; j < VPT; ++j) acc[j] += o[j];
        }
        __syncthreads();
    }
    const float inv = 1.f / static_cast<float>(npix);
    float* out = pooled + (static_cast<long long>(n) * kPspBins + bin) * C + cq * VPT;
    if (parts == 1) {
        if (pl == 0) {
#pragma unroll
            for (int j = 0; j < VPT; ++j) out[j] = acc[j] * inv;
        }
        return;
    }
    // split bin: park this part, the last part to arrive adds all of them in part order
    __shared__ bool s_last;
    float* parked = partial + (static_cast<long long>(n) * wk.n + blockIdx.x) * C + cq * VPT;
    if (pl == 0) {
#pragma unroll
        for (int j = 0; j < VPT; ++j) parked[j] = acc[j];
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&tickets[n * kPspBins + bin], 1u) == static_cast<unsigned>(parts - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (pl == 0) {
        const float* first = partial + (static_cast<long long>(n) * wk.n + (blockIdx.x - part)) * C + cq * VPT;
        float sum[VPT];
#pragma unroll
        for (int j = 0; j < VPT; ++j) sum[j] = 0.f;
        for (int q = 0; q < parts; ++q)
#pragma unroll
            for (int j = 0; j < VPT; ++j) sum[j] += __ldcg(first + static_cast<long long>(q) * C + j);
#pragma unroll
        for (int j = 0; j < VPT; ++j) out[j] = sum[j] * inv;
    }
    if (threadIdx.x == 0) tickets[n * kPspBins + bin] = 0;  // ready for the next launch
}

// grid (ceil(W*CQ/256), H, N); thread per (column, channel vector): out[pix][0:C] = x, out[pix][C*(1+si) + c] =
// bilinear(pooled_si)(pix, c), 16-byte loads and stores.  Row taps are per-block constants.
template <typename T>
__global__ void __launch_bounds__(256)
psp_concat_kernel(const T* __restrict__ x, long long ldx, const float* __restrict__ pooled, T* __restrict__ out,
                  long long ldo, int H, int W, int C) {
    constexpr int VPT = Vec16<T>::N;
    const int CQ = C / VPT;
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= static_cast<unsigned>(W) * CQ) return;
    const int w = idx / CQ, c = (idx - w * CQ) * VPT;
    const int h = blockIdx.y, n = blockIdx.z;
    const long long pix = (static_cast<long long>(n) * H + h) * W + w;
    T* o = out + pix * ldo;
    Vec16<T> xv;
    xv.load(x + pix * ldx + c);
    xv.store(o + c);
    const float* pn = pooled + static_cast<long long>(n) * kPspBins * C + c;
#pragma unroll
    for (int si = 0; si < 4; ++si) {
        const int s = kPspSize[si];
        const float* ps = pn + static_cast<long long>(kPspOffset[si]) * C;
        int y0, y1, x0, x1;
        float wy, wx;
        cab_bilinear_tap(h, static_cast<float>(s) / static_cast<float>(H), s, y0, y1, wy);
        cab_bilinear_tap(w, static_cast<float>(s) / static_cast<float>(W), s, x0, x1, wx);
        const float* p00 = ps + (y0 * s + x0) * C;
        const float* p01 = ps + (y0 * s + x1) * C;
        const float* p10 = ps + (y1 * s + x0) * C;
        const float* p11 = ps + (y1 * s + x1) * C;
        float f[VPT];
#pragma unroll
        for (int j = 0; j < VPT; j += 4) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(p00 + j)), b = __ldg(reinterpret_cast<const float4*>(p01 + j));
            const float4 cc = __ldg(reinterpret_cast<const float4*>(p10 + j)), d = __ldg(reinterpret_cast<const float4*>(p11 + j));
            f[j + 0] = (1.f - wy) * ((1.f - wx) * a.x + wx * b.x) + wy * ((1.f - wx) * cc.x + wx * d.x);
            f[j + 1] = (1.f - wy) * ((1.f - wx) * a.y + wx * b.y) + wy * ((1.f - wx) * cc.y + wx * d.y);
            f[j + 2] = (1.f - wy) * ((1.f - wx) * a.z + wx * b.z) + wy * ((1.f - wx) * cc.z + wx * d.z);
            f[j + 3] = (1.f - wy) * ((1.f - wx) * a.w + wx * b.w) + wy * ((1.f - wx) * cc.w + wx * d.w);
        }
        Vec16<T> ov;
        ov.pack(f);
        ov.store(o + static_cast<long long>(C) * (1 + si) + c);
    }
}

}  // namespace

extern "C" int cabinet_psp_pool(const void* x, long long ldx, int dtype, float* pooled, int N, int H, int W, int C,
                                float* scratch, long long scratch_bytes, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("psp_pool", dtype, CAB_DT_F32 | CAB_DT_BF16);
    const int vpt = dtype == CABINET_BF16 ? 8 : 4;
    CAB_REQUIRE(x && pooled && H > 0 && W > 0 && C > 0 && ldx >= C && C % vpt == 0 && C <= 1024 && ldx % vpt == 0 &&
                    (reinterpret_cast<uintptr_t>(x) & 15) == 0,
                "psp_pool: bad arguments (C and ldx must be multiples of 16 bytes, C <= 1024, x 16-byte aligned)");
    if (N == 0) return CABINET_OK;
    CAB_REQUIRE(C / vpt <= 128 && N <= 65535, "psp_pool: C / N too large");
    // split bins larger than `chunk` pixels; at most 256 work items
    PspWork wk;
    for (wk.chunk = 128;; wk.chunk *= 2) {
        wk.n = 0;
        bool fits = true;
        for (int bin = 0; bin < kPspBins && fits; ++bin) {
            int h0, h1, w0, w1;
            psp_bin_rect(bin, H, W, h0, h1, w0, w1);
            const int npix = (h1 - h0) * (w1 - w0);
            const int parts = std::min(255, (npix + wk.chunk - 1) / wk.chunk);
            for (int pt = 0; pt < parts && fits; ++pt) {
                if (wk.n == 256) { fits = false; break; }
                wk.bin[wk.n] = static_cast<unsigned short>(bin);
                wk.part[wk.n] = static_cast<unsigned char>(pt);
                wk.parts[wk.n] = static_cast<unsigned char>(parts);
                ++wk.n;
            }
        }
        if (fits) break;
    }
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    // scratch: [N][110] tickets (uint32; zero before the first launch, left at zero) then [N][work items][C] partial sums
    const size_t off = (static_cast<size_t>(N) * kPspBins * sizeof(unsigned int) + 255) & ~size_t(255);
    const size_t need = off + static_cast<size_t>(N) * wk.n * C * sizeof(float);
    CAB_REQUIRE(scratch && static_cast<size_t>(scratch_bytes) >= need, "psp_pool: scratch needs %zu bytes", need);
    unsigned int* tickets = reinterpret_cast<unsigned int*>(scratch);
    float* partial = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(scratch) + off);
    dim3 grid(wk.n, N);
    const int cq = C / vpt;
    const int threads = std::max(cq, 128 / cq * cq);  // a multiple of the channel-vector count close to 128
    const size_t smem = static_cast<size_t>(threads) * vpt * sizeof(float);
    if (dtype == CABINET_BF16)
        psp_pool_kernel<bf16><<<grid, threads, smem, s>>>(reinterpret_cast<const bf16*>(x), ldx, pooled, H, W, C, wk, partial, tickets);
    else
        psp_pool_kernel<float><<<grid, threads, smem, s>>>(reinterpret_cast<const float*>(x), ldx, pooled, H, W, C, wk, partial, tickets);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_psp_concat(const void* x, long long ldx, const float* pooled, void* out, long long ldo,
                                  int dtype, int N, int H, int W, int C, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("psp_concat", dtype, CAB_DT_F32 | CAB_DT_BF16);
    const int vpt = dtype == CABINET_BF16 ? 8 : 4;
    CAB_REQUIRE(x && pooled && out && H > 0 && W > 0 && C > 0 && ldx >= C && ldo >= 5LL * C, "psp_concat: bad arguments");
    CAB_REQUIRE(C % vpt == 0 && ldx % vpt == 0 && ldo % vpt == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(out) & 15) == 0 && (reinterpret_cast<uintptr_t>(pooled) & 15) == 0,
                "psp_concat: C / ldx / ldo must be multiples of 16 bytes and the pointers 16-byte aligned");
    if (N == 0) return CABINET_OK;
    CAB_REQUIRE(H <= 65535 && N <= 65535, "psp_concat: H/N exceed grid limits");
    dim3 grid(static_cast<unsigned>(cab_ceil_div(static_cast<long long>(W) * (C / vpt), 256)), H, N);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (dtype == CABINET_BF16)
        psp_concat_kernel<bf16><<<grid, 256, 0, s>>>(reinterpret_cast<const bf16*>(x), ldx, pooled,
                                                    reinterpret_cast<bf16*>(out), ldo, H, W, C);
    else
        psp_concat_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(x), ldx, pooled,
                                                     reinterpret_cast<float*>(out), ldo, H, W, C);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}
