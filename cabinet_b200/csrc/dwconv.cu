// Depthwise k x k convolution (+ folded BN bias, activation, optional GAP partial sums), NHWC.
// HBM-bound: every thread owns one 16-byte channel vector (8 bf16 / 4 fp32) of a short run of output
// pixels along W, so the k x (k + run - 1) input window is loaded once into registers and re-used;
// neighbouring rows/threads hit L1.  Algorithmic bytes per launch = in + out activations + weights.
#include "common.cuh"

namespace {

template <typename T, int K, int S, int RUN>
__global__ void __launch_bounds__(256)
dwconv_kernel(const T* __restrict__ x, long long ldx, const float* __restrict__ w, const float* __restrict__ bias,
              T* __restrict__ y, long long ldy, int H, int W, int C, int OH, int OW, int act,
              float* __restrict__ gap_sum) {
    constexpr int V = Vec16<T>::N;
    constexpr int PAD = (K - 1) / 2;
    constexpr int SPAN = (RUN - 1) * S + K;  // input columns needed by RUN outputs
    extern __shared__ float s_gap[];         // [C] when gap_sum != nullptr

    const int n = blockIdx.y;
    const int CG = C / V;
    const int runs_w = (OW + RUN - 1) / RUN;
    const long long total = static_cast<long long>(OH) * runs_w * CG;
    if (gap_sum) {
        for (int i = threadIdx.x; i < C; i += blockDim.x) s_gap[i] = 0.f;
        __syncthreads();
    }
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx < total) {
        const int cg = static_cast<int>(idx % CG);
        long long t = idx / CG;
        const int rw = static_cast<int>(t % runs_w);
        const int oh = static_cast<int>(t / runs_w);
        const int c0 = cg * V;
        const int ow0 = rw * RUN;
        const int iw0 = ow0 * S - PAD;
        const int ih0 = oh * S - PAD;

        float acc[RUN][V];
        float bv[V];
#pragma unroll
        for (int v = 0; v < V; ++v) bv[v] = bias[c0 + v];
#pragma unroll
        for (int r = 0; r < RUN; ++r)
#pragma unroll
            for (int v = 0; v < V; ++v) acc[r][v] = bv[v];

        const T* xin = x + static_cast<long long>(n) * H * W * ldx + c0;
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
            const int ih = ih0 + ky;
            if (ih < 0 || ih >= H) continue;
            float wk[K][V];
#pragma unroll
            for (int kx = 0; kx < K; ++kx) {
                if constexpr (V == 8) {
                    float4 w0 = __ldg(reinterpret_cast<const float4*>(w + (ky * K + kx) * C + c0));
                    float4 w1 = __ldg(reinterpret_cast<const float4*>(w + (ky * K + kx) * C + c0 + 4));
                    wk[kx][0] = w0.x; wk[kx][1] = w0.y; wk[kx][2] = w0.z; wk[kx][3] = w0.w;
                    wk[kx][4] = w1.x; wk[kx][5] = w1.y; wk[kx][6] = w1.z; wk[kx][7] = w1.w;
                } else {
                    float4 w0 = __ldg(reinterpret_cast<const float4*>(w + (ky * K + kx) * C + c0));
                    wk[kx][0] = w0.x; wk[kx][1] = w0.y; wk[kx][2] = w0.z; wk[kx][3] = w0.w;
                }
            }
            const T* row = xin + static_cast<long long>(ih) * W * ldx;
#pragma unroll
            for (int sx = 0; sx < SPAN; ++sx) {
                const int iw = iw0 + sx;
                if (iw < 0 || iw >= W) continue;
                Vec16<T> xv;
                xv.load(row + static_cast<long long>(iw) * ldx);
                float xf[V];
                xv.unpack(xf);
#pragma unroll
                for (int r = 0; r < RUN; ++r) {
                    const int kx = sx - r * S;  // compile-time after unrolling
                    if (kx >= 0 && kx < K) {
#pragma unroll
                        for (int v = 0; v < V; ++v) acc[r][v] = fmaf(xf[v], wk[kx][v], acc[r][v]);
                    }
                }
            }
        }

        float gsum[V];
#pragma unroll
        for (int v = 0; v < V; ++v) gsum[v] = 0.f;
        T* yout = y + (static_cast<long long>(n) * OH + oh) * OW * ldy + c0;
#pragma unroll
        for (int r = 0; r < RUN; ++r) {
            const int ow = ow0 + r;
            if (ow >= OW) continue;
            cab_act_vec<V>(acc[r], act);
#pragma unroll
            for (int v = 0; v < V; ++v) gsum[v] += acc[r][v];
            Vec16<T> ov;
            ov.pack(acc[r]);
            ov.store(yout + static_cast<long long>(ow) * ldy);
        }
        if (gap_sum) {
#pragma unroll
            for (int v = 0; v < V; ++v) atomicAdd(&s_gap[c0 + v], gsum[v]);
        }
    }
    if (gap_sum) {
        __syncthreads();
        for (int i = threadIdx.x; i < C; i += blockDim.x) {
            float v = s_gap[i];
            if (v != 0.f) atomicAdd(&gap_sum[static_cast<long long>(n) * C + i], v);
        }
    }
}

template <typename T, int K, int S>
int launch(const void* x, long long ldx, const float* w, const float* bias, void* y, long long ldy, int N, int H,
           int W, int C, int OH, int OW, int act, float* gap_sum, cudaStream_t s) {
    constexpr int RUN = 4;
    constexpr int V = Vec16<T>::N;
    const int runs_w = (OW + RUN - 1) / RUN;
    const long long total = static_cast<long long>(OH) * runs_w * (C / V);
    dim3 grid(static_cast<unsigned>(cab_ceil_div(total, 256)), N);
    size_t smem = gap_sum ? sizeof(float) * C : 0;
    dwconv_kernel<T, K, S, RUN><<<grid, 256, smem, s>>>(reinterpret_cast<const T*>(x), ldx, w, bias,
                                                        reinterpret_cast<T*>(y), ldy, H, W, C, OH, OW, act, gap_sum);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

}  // namespace

extern "C" int cabinet_dwconv(const void* x, long long ldx, const float* w, const float* bias, void* y,
                              long long ldy, int dtype, int N, int H, int W, int C, int k, int stride, int OH, int OW,
                              int act, float* gap_sum, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("dwconv", dtype, CAB_DT_F32 | CAB_DT_BF16);
    CAB_REQUIRE(x && w && bias && y, "dwconv: null pointer");
    CAB_REQUIRE((k == 3 || k == 5) && (stride == 1 || stride == 2), "dwconv: k must be 3|5 and stride 1|2 (got %d,%d)",
                k, stride);
    const int V = dtype == CABINET_F32 ? 4 : 8;
    CAB_REQUIRE(C > 0 && C % V == 0 && ldx % V == 0 && ldy % V == 0 && ldx >= C && ldy >= C,
                "dwconv: C/ldx/ldy must be multiples of %d (C=%d ldx=%lld ldy=%lld)", V, C, ldx, ldy);
    CAB_REQUIRE(OH == (H + 2 * ((k - 1) / 2) - k) / stride + 1 && OW == (W + 2 * ((k - 1) / 2) - k) / stride + 1,
                "dwconv: inconsistent output size");
    if (N == 0) return CABINET_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define CAB_DW(T, KK, SS) return launch<T, KK, SS>(x, ldx, w, bias, y, ldy, N, H, W, C, OH, OW, act, gap_sum, s)
    if (dtype == CABINET_BF16) {
        if (k == 3 && stride == 1) CAB_DW(bf16, 3, 1);
        if (k == 3 && stride == 2) CAB_DW(bf16, 3, 2);
        if (k == 5 && stride == 1) CAB_DW(bf16, 5, 1);
        CAB_DW(bf16, 5, 2);
    } else {
        if (k == 3 && stride == 1) CAB_DW(float, 3, 1);
        if (k == 3 && stride == 2) CAB_DW(float, 3, 2);
        if (k == 5 && stride == 1) CAB_DW(float, 5, 1);
        CAB_DW(float, 5, 2);
    }
#undef CAB_DW
}
