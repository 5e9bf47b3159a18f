// CUDA-core implicit-GEMM convolution / batched GEMM (fp32 accumulate).
// This is the fp32 parity path of the whole network and the Cin=3 stem path of the bf16 network;
// the bf16 GEMM-shaped layers run on tcgen05 (gemm_tc.cu).
#include "common.cuh"

namespace {

struct ConvArgs {
    const void* x; long long sxn, sxh, sxw, sxc, xbs;
    const void* w; long long w_sco, w_sk, wbs;
    const float* bias;
    const void* res; long long ldres;
    void* y; long long ldy, ybs;
    int N, H, W, Cin, Cout, KH, KW, stride, pad, OH, OW, act;
    float alpha;
    long long M;  // N*OH*OW
    int K;        // KH*KW*Cin
};

constexpr int BM = 64, BN = 64, BK = 16, THREADS = 256;

template <typename TX, typename TW, typename TY>
__global__ void __launch_bounds__(THREADS) conv_simt_kernel(ConvArgs a) {
    __shared__ __align__(16) float As[BK][BM];
    __shared__ __align__(16) float Bs[BK][BN + 4];
    __shared__ long long pix_base[BM];
    __shared__ int pix_ih0[BM], pix_iw0[BM];

    const int tid = threadIdx.x;
    const int b = blockIdx.z;
    const long long m0 = static_cast<long long>(blockIdx.x) * BM;
    const int n0 = blockIdx.y * BN;
    const TX* __restrict__ x = reinterpret_cast<const TX*>(a.x) + b * a.xbs;
    const TW* __restrict__ w = reinterpret_cast<const TW*>(a.w) + b * a.wbs;

    if (tid < BM) {
        long long m = m0 + tid;
        if (m < a.M) {
            int ow = static_cast<int>(m % a.OW);
            long long t = m / a.OW;
            int oh = static_cast<int>(t % a.OH);
            int n = static_cast<int>(t / a.OH);
            int ih0 = oh * a.stride - a.pad, iw0 = ow * a.stride - a.pad;
            pix_ih0[tid] = ih0;
            pix_iw0[tid] = iw0;
            pix_base[tid] = n * a.sxn + ih0 * a.sxh + iw0 * a.sxw;
        } else {
            pix_ih0[tid] = -(1 << 28);  // forces every tap out of bounds -> zeros
            pix_iw0[tid] = -(1 << 28);
            pix_base[tid] = 0;
        }
    }
    __syncthreads();

    const int ty = tid / 16, tx = tid % 16;
    float acc[4][4] = {};

    const int a_pix = tid % BM, a_kq = tid / BM;  // A loader: pixel, k-quad (0..3)
    const int b_co = tid / 4, b_kq = tid % 4;     // B loader
    const long long abase = pix_base[a_pix];
    const int aih0 = pix_ih0[a_pix], aiw0 = pix_iw0[a_pix];

    for (int k0 = 0; k0 < a.K; k0 += BK) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int k = k0 + a_kq * 4 + j;
            float v = 0.f;
            if (k < a.K) {
                int tap = k / a.Cin, c = k - tap * a.Cin;
                int ky = tap / a.KW, kx = tap - ky * a.KW;
                int ih = aih0 + ky, iw = aiw0 + kx;
                if (ih >= 0 && ih < a.H && iw >= 0 && iw < a.W)
                    v = to_f32<TX>(x[abase + ky * a.sxh + kx * a.sxw + c * a.sxc]);
            }
            As[a_kq * 4 + j][a_pix] = v;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int k = k0 + b_kq * 4 + j;
            int co = n0 + b_co;
            float v = 0.f;
            if (k < a.K && co < a.Cout) v = to_f32<TW>(w[co * a.w_sco + k * a.w_sk]);
            Bs[b_kq * 4 + j][b_co] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float af[4] = {av.x, av.y, av.z, av.w};
            const float bf[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(af[i], bf[j], acc[i][j]);
        }
        __syncthreads();
    }

    TY* __restrict__ y = reinterpret_cast<TY*>(a.y) + b * a.ybs;
    const TY* __restrict__ res = a.res ? reinterpret_cast<const TY*>(a.res) + b * a.ybs : nullptr;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        long long m = m0 + ty * 4 + i;
        if (m >= a.M) continue;
        float v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = n0 + tx * 4 + j;
            v[j] = acc[i][j] * a.alpha + ((a.bias && co < a.Cout) ? a.bias[co] : 0.f);
        }
        cab_act_vec<4>(v, a.act);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = n0 + tx * 4 + j;
            if (co >= a.Cout) continue;
            if (res) v[j] += to_f32<TY>(res[m * a.ldres + co]);
            y[m * a.ldy + co] = from_f32<TY>(v[j]);
        }
    }
}

template <typename TX, typename TW, typename TY>
int launch(const ConvArgs& a, int batches, cudaStream_t s) {
    dim3 grid(static_cast<unsigned>(cab_ceil_div(a.M, BM)), static_cast<unsigned>(cab_ceil_div(a.Cout, BN)), batches);
    conv_simt_kernel<TX, TW, TY><<<grid, THREADS, 0, s>>>(a);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

}  // namespace

extern "C" int cabinet_conv2d_simt(const void* x, int x_dtype, long long sxn, long long sxh, long long sxw,
                                   long long sxc, long long x_batch_stride, const void* w, int w_dtype,
                                   long long w_sco, long long w_sk, long long w_batch_stride, const float* bias,
                                   const void* res, long long ldres, void* y, int y_dtype, long long ldy,
                                   long long y_batch_stride, int batches, int N, int H, int W, int Cin, int Cout,
                                   int KH, int KW, int stride, int pad, int OH, int OW, int act, float alpha,
                                   cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("conv2d_simt", x_dtype, CAB_DT_ALL);
    CAB_REQUIRE_DTYPE("conv2d_simt", w_dtype, CAB_DT_ALL);
    CAB_REQUIRE_DTYPE("conv2d_simt", y_dtype, CAB_DT_ALL);
    CAB_REQUIRE(x && w && y, "conv2d_simt: null pointer");
    CAB_REQUIRE(batches >= 1 && N >= 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0 && KH > 0 && KW > 0,
                "conv2d_simt: bad sizes");
    CAB_REQUIRE(stride >= 1 && pad >= 0 && OH > 0 && OW > 0, "conv2d_simt: bad stride/pad/output size");
    CAB_REQUIRE(ldy >= Cout, "conv2d_simt: ldy < Cout");
    ConvArgs a;
    a.x = x; a.sxn = sxn; a.sxh = sxh; a.sxw = sxw; a.sxc = sxc; a.xbs = x_batch_stride;
    a.w = w; a.w_sco = w_sco; a.w_sk = w_sk; a.wbs = w_batch_stride;
    a.bias = bias; a.res = res; a.ldres = ldres; a.y = y; a.ldy = ldy; a.ybs = y_batch_stride;
    a.N = N; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.KH = KH; a.KW = KW; a.stride = stride; a.pad = pad;
    a.OH = OH; a.OW = OW; a.act = act; a.alpha = alpha;
    a.M = static_cast<long long>(N) * OH * OW;
    a.K = KH * KW * Cin;
    if (a.M == 0) return CABINET_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool has_f16 = x_dtype == CABINET_F16 || w_dtype == CABINET_F16 || y_dtype == CABINET_F16;
    if (has_f16) {  // fp16 training mode: each operand fp32 or fp16
        CAB_REQUIRE(x_dtype != CABINET_BF16 && w_dtype != CABINET_BF16 && y_dtype != CABINET_BF16,
                    "conv2d_simt: bf16 and fp16 operands do not mix");
        switch ((x_dtype == CABINET_F16) * 4 + (w_dtype == CABINET_F16) * 2 + (y_dtype == CABINET_F16)) {
            case 1: return launch<float, float, f16>(a, batches, s);
            case 2: return launch<float, f16, float>(a, batches, s);
            case 3: return launch<float, f16, f16>(a, batches, s);
            case 4: return launch<f16, float, float>(a, batches, s);
            case 5: return launch<f16, float, f16>(a, batches, s);
            case 6: return launch<f16, f16, float>(a, batches, s);
            case 7: return launch<f16, f16, f16>(a, batches, s);
        }
    }
    const int key = x_dtype * 4 + w_dtype * 2 + y_dtype;
    switch (key) {
        case 0: return launch<float, float, float>(a, batches, s);
        case 1: return launch<float, float, bf16>(a, batches, s);
        case 2: return launch<float, bf16, float>(a, batches, s);
        case 3: return launch<float, bf16, bf16>(a, batches, s);
        case 4: return launch<bf16, float, float>(a, batches, s);
        case 5: return launch<bf16, float, bf16>(a, batches, s);
        case 6: return launch<bf16, bf16, float>(a, batches, s);
        case 7: return launch<bf16, bf16, bf16>(a, batches, s);
    }
    cabinet_set_error("conv2d_simt: unsupported dtype combination %d/%d/%d", x_dtype, w_dtype, y_dtype);
    return CABINET_ERR_INVALID;
}
