// Bilinear resampling (align_corners=False) and the fused output tail:
//   bilinear_nhwc          1/32 -> 1/8 feature / aux-logit upsample (src/models/cabinet.py:228-233)
//   upsample_logits_nchw   x8 logits upsample written as the NCHW tensors CABiNet.forward returns (:240-245)
//   upsample_argmax        the same upsample fused with argmax (+ confusion matrix), logits never reach HBM
//   confusion_hist         hist[pred, label] (src/scripts/evaluate.py:162-191)
// All HBM-bound on their OUTPUT bytes: the sources are <= 1/64 of the output and stay in L1/L2.
#include "common.cuh"

namespace {

// ---------------------------------------------------------------------------------- NHWC -> NHWC
template <typename TI, typename TO>
__global__ void __launch_bounds__(256)
bilinear_nhwc_kernel(const TI* __restrict__ x, long long ldx, TO* __restrict__ y, long long ldy, int IH, int IW, int C,
                     int OH, int OW, long long total, float sh, float sw) {
    // thread per (output pixel, group of 4 channels)
    const int CG = (C + 3) / 4;
    const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const int cg = static_cast<int>(idx % CG);
    long long t = idx / CG;
    const int ow = static_cast<int>(t % OW);
    t /= OW;
    const int oh = static_cast<int>(t % OH);
    const int n = static_cast<int>(t / OH);
    int y0, y1, x0, x1;
    float wy, wx;
    cab_bilinear_tap(oh, sh, IH, y0, y1, wy);
    cab_bilinear_tap(ow, sw, IW, x0, x1, wx);
    const TI* b = x + static_cast<long long>(n) * IH * IW * ldx + cg * 4;
    const TI* p00 = b + (static_cast<long long>(y0) * IW + x0) * ldx;
    const TI* p01 = b + (static_cast<long long>(y0) * IW + x1) * ldx;
    const TI* p10 = b + (static_cast<long long>(y1) * IW + x0) * ldx;
    const TI* p11 = b + (static_cast<long long>(y1) * IW + x1) * ldx;
    TO* o = y + ((static_cast<long long>(n) * OH + oh) * OW + ow) * ldy + cg * 4;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        if (cg * 4 + c >= C) break;
        const float v = (1.f - wy) * ((1.f - wx) * to_f32<TI>(p00[c]) + wx * to_f32<TI>(p01[c])) +
                        wy * ((1.f - wx) * to_f32<TI>(p10[c]) + wx * to_f32<TI>(p11[c]));
        o[c] = from_f32<TO>(v);
    }
}

// bf16 -> bf16, C % 8 == 0: grid (x-chunks, OH, N); one thread = one output pixel x 8 channels (four 16-byte loads, one
// 16-byte store); row taps are per-block constants, 32-bit index arithmetic only.
__global__ void __launch_bounds__(256)
bilinear_nhwc_bf16x8_kernel(const bf16* __restrict__ x, long long ldx, bf16* __restrict__ y, long long ldy, int IH,
                            int IW, int C, int OH, int OW, float sh, float sw) {
    const int CG = C >> 3;
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= static_cast<unsigned>(OW) * CG) return;
    const int ow = idx / CG, cg = idx - ow * CG;
    const int oh = blockIdx.y, n = blockIdx.z;
    int y0, y1, x0, x1;
    float wy, wx;
    cab_bilinear_tap(oh, sh, IH, y0, y1, wy);
    cab_bilinear_tap(ow, sw, IW, x0, x1, wx);
    const bf16* b = x + static_cast<long long>(n) * IH * IW * ldx + cg * 8;
    Vec16<bf16> v00, v01, v10, v11, o;
    v00.load(b + (static_cast<long long>(y0) * IW + x0) * ldx);
    v01.load(b + (static_cast<long long>(y0) * IW + x1) * ldx);
    v10.load(b + (static_cast<long long>(y1) * IW + x0) * ldx);
    v11.load(b + (static_cast<long long>(y1) * IW + x1) * ldx);
    float f00[8], f01[8], f10[8], f11[8], r[8];
    v00.unpack(f00); v01.unpack(f01); v10.unpack(f10); v11.unpack(f11);
#pragma unroll
    for (int c = 0; c < 8; ++c)
        r[c] = (1.f - wy) * ((1.f - wx) * f00[c] + wx * f01[c]) + wy * ((1.f - wx) * f10[c] + wx * f11[c]);
    o.pack(r);
    o.store(y + ((static_cast<long long>(n) * OH + oh) * OW + ow) * ldy + cg * 8);
}

// bf16 -> bf16, exact x4 (OH = 4*IH, OW = 4*IW: the 1/32 -> 1/8 feature upsample whenever H, W are multiples of 32):
// one thread = one SOURCE pixel x 8 channels -> its 4 x 4 output pixels.  Output column 4g+j reads source columns
// (g-1, g) with weight {0.625, 0.875} for j = 0, 1 and (g, g+1) with {0.125, 0.375} for j = 2, 3 (same for rows), so
// nine 16-byte loads feed sixteen 16-byte stores (the per-pixel kernel needs 64 loads for them).  At the borders the
// clamped neighbour equals the centre, which makes ATen's clamped source index and the static weight agree.
__global__ void __launch_bounds__(256)
bilinear_x4_bf16_kernel(const bf16* __restrict__ x, long long ldx, bf16* __restrict__ y, long long ldy, int IH, int IW,
                        int C) {
    const int CG = C >> 3;
    const unsigned idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= static_cast<unsigned>(IW) * CG) return;
    const int gx = idx / CG, cg = idx - gx * CG;
    const int gy = blockIdx.y, n = blockIdx.z;
    const int xs[3] = {max(gx - 1, 0), gx, min(gx + 1, IW - 1)};
    const int ys[3] = {max(gy - 1, 0), gy, min(gy + 1, IH - 1)};
    const bf16* b = x + static_cast<long long>(n) * IH * IW * ldx + cg * 8;
    float f[3][3][8];
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            Vec16<bf16> v;
            v.load(b + (static_cast<long long>(ys[r]) * IW + xs[c]) * ldx);
            v.unpack(f[r][c]);
        }
    const int OW = 4 * IW;
    bf16* o = y + ((static_cast<long long>(n) * 4 * IH + 4 * gy) * OW + 4 * gx) * ldy + cg * 8;
#pragma unroll
    for (int jy = 0; jy < 4; ++jy) {
        const int ra = jy < 2 ? 0 : 1;                       // rows (ra, ra + 1)
        const float wy = jy < 2 ? 0.625f + 0.25f * jy : 0.125f + 0.25f * (jy - 2);
        float v[3][8];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int k = 0; k < 8; ++k) v[c][k] = f[ra][c][k] + wy * (f[ra + 1][c][k] - f[ra][c][k]);
#pragma unroll
        for (int jx = 0; jx < 4; ++jx) {
            const int ca = jx < 2 ? 0 : 1;
            const float wx = jx < 2 ? 0.625f + 0.25f * jx : 0.125f + 0.25f * (jx - 2);
            float r[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) r[k] = v[ca][k] + wx * (v[ca + 1][k] - v[ca][k]);
            Vec16<bf16> ov;
            ov.pack(r);
            ov.store(o + (static_cast<long long>(jy) * OW + jx) * ldy);
        }
    }
}

// ---------------------------------------------------------------------------------- logits tail
// Each thread produces 8 consecutive output pixels [8g, 8g+8) of one output row for ALL classes and hands them,
// class by class, to a consumer (NCHW store / running argmax).
//  * exact x8 path (OH = 8*IH, OW = 8*IW, the CABiNet case whenever H, W are multiples of 64): the 8 pixels
//    touch only source columns g-1, g, g+1 with compile-time weights, the row touches source rows (k-1,k) or
//    (k,k+1): 6 fp32 vectors per class chunk -> 8 outputs, ~2.5 ALU ops per output.
//  * generic path (any sizes): per-pixel taps, 4 loads per output.
// Both evaluate the same expression tree per output, so the NCHW kernel and the argmax kernel agree bit for bit:
//   v = top + wy * (bot - top),  top/bot = a + wx * (b - a).
constexpr int PXG = 8;

// exact x8: 8 output pixels [8g, 8g+8) of one row for classes [c4, c4+4) from the 6 source vectors around them
__device__ __forceinline__ void exact8_chunk4(const float* __restrict__ r0, const float* __restrict__ r1, int xa, int xb,
                                              int xc, int C, int c4, float wy, float (&v)[4][PXG]) {
    const float4 ta = __ldg(reinterpret_cast<const float4*>(r0 + xa * C + c4));
    const float4 tb = __ldg(reinterpret_cast<const float4*>(r0 + xb * C + c4));
    const float4 tcc = __ldg(reinterpret_cast<const float4*>(r0 + xc * C + c4));
    const float4 ba = __ldg(reinterpret_cast<const float4*>(r1 + xa * C + c4));
    const float4 bb = __ldg(reinterpret_cast<const float4*>(r1 + xb * C + c4));
    const float4 bc = __ldg(reinterpret_cast<const float4*>(r1 + xc * C + c4));
    const float tav[4] = {ta.x, ta.y, ta.z, ta.w}, tbv[4] = {tb.x, tb.y, tb.z, tb.w};
    const float tcv[4] = {tcc.x, tcc.y, tcc.z, tcc.w}, bav[4] = {ba.x, ba.y, ba.z, ba.w};
    const float bbv[4] = {bb.x, bb.y, bb.z, bb.w}, bcv[4] = {bc.x, bc.y, bc.z, bc.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float va = tav[k] + wy * (bav[k] - tav[k]), vb = tbv[k] + wy * (bbv[k] - tbv[k]);
        const float vc = tcv[k] + wy * (bcv[k] - tcv[k]);
        const float d0 = vb - va, d1 = vc - vb;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            v[k][j] = va + ((j + 4.5f) * 0.125f) * d0;
            v[k][j + 4] = vb + ((j + 0.5f) * 0.125f) * d1;
        }
    }
}

template <bool EXACT8, typename Consumer>
__device__ __forceinline__ void upsample_group8(const float* __restrict__ x, int n, int oh, int g, int IH, int IW,
                                                int C, int OW, float sh, float sw, Consumer&& consume) {
    int y0, y1;
    float wy;
    cab_bilinear_tap(oh, sh, IH, y0, y1, wy);
    const float* r0 = x + (static_cast<long long>(n) * IH + y0) * IW * C;
    const float* r1 = x + (static_cast<long long>(n) * IH + y1) * IW * C;
    if constexpr (EXACT8) {
        const int xa = max(g - 1, 0), xb = g, xc = min(g + 1, IW - 1);
        int cstart = 0;
        if ((C & 3) == 0) {  // 4 classes per 16-byte load: 6 loads feed 32 outputs
            cstart = C;
            for (int c4 = 0; c4 < C; c4 += 4) {
                float v[4][PXG];
                exact8_chunk4(r0, r1, xa, xb, xc, C, c4, wy, v);
#pragma unroll
                for (int k = 0; k < 4; ++k) consume(c4 + k, v[k]);
            }
        }
        for (int c = cstart; c < C; ++c) {
            const float ta = __ldg(r0 + xa * C + c), tb = __ldg(r0 + xb * C + c), tcc = __ldg(r0 + xc * C + c);
            const float ba = __ldg(r1 + xa * C + c), bb = __ldg(r1 + xb * C + c), bc = __ldg(r1 + xc * C + c);
            const float va = ta + wy * (ba - ta), vb = tb + wy * (bb - tb), vc = tcc + wy * (bc - tcc);
            const float d0 = vb - va, d1 = vc - vb;
            float v[PXG];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                // at the left edge (g == 0) ATen clamps src to 0 -> weight 0 on column 0; va == vb there, so the
                // unclamped static weight gives the same value
                v[j] = va + ((j + 4.5f) * 0.125f) * d0;
                v[j + 4] = vb + ((j + 0.5f) * 0.125f) * d1;
            }
            consume(c, v);
        }
    } else {
        int x0[PXG], x1[PXG];
        float wx[PXG];
#pragma unroll
        for (int p = 0; p < PXG; ++p) cab_bilinear_tap(min(g * PXG + p, OW - 1), sw, IW, x0[p], x1[p], wx[p]);
        for (int c = 0; c < C; ++c) {
            float v[PXG];
#pragma unroll
            for (int p = 0; p < PXG; ++p) {
                const float t0 = __ldg(r0 + x0[p] * C + c), t1 = __ldg(r0 + x1[p] * C + c);
                const float b0 = __ldg(r1 + x0[p] * C + c), b1 = __ldg(r1 + x1[p] * C + c);
                const float top = t0 + wx[p] * (t1 - t0), bot = b0 + wx[p] * (b1 - b0);
                v[p] = top + wy * (bot - top);
            }
            consume(c, v);
        }
    }
}

template <typename TO, bool EXACT8>
__global__ void __launch_bounds__(128)
upsample_logits_nchw_kernel(const float* __restrict__ x, int IH, int IW, int C, TO* __restrict__ y, int OH, int OW,
                            float sh, float sw) {
    const int groups_w = (OW + PXG - 1) / PXG;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= groups_w) return;
    const int oh = blockIdx.y, n = blockIdx.z;
    const int ow0 = g * PXG;
    const bool full = (OW % PXG) == 0;  // rows are 16-byte aligned and the group is complete
    upsample_group8<EXACT8>(x, n, oh, g, IH, IW, C, OW, sh, sw, [&](int c, const float* v) {
        TO* o = y + ((static_cast<long long>(n) * C + c) * OH + oh) * OW + ow0;
        if (full) {
            if constexpr (sizeof(TO) == 4) {
                __stcs(reinterpret_cast<float4*>(o), make_float4(v[0], v[1], v[2], v[3]));
                __stcs(reinterpret_cast<float4*>(o) + 1, make_float4(v[4], v[5], v[6], v[7]));
            } else {
                Vec16<bf16> ov;
                ov.pack(v);
                __stcs(reinterpret_cast<uint4*>(o), ov.raw);
            }
        } else {
#pragma unroll
            for (int p = 0; p < PXG; ++p)
                if (ow0 + p < OW) o[p] = from_f32<TO>(v[p]);
        }
    });
}

template <bool EXACT8>
__global__ void __launch_bounds__(128)
upsample_argmax_kernel(const float* __restrict__ x, int IH, int IW, int C, uint8_t* __restrict__ mask, int OH, int OW,
                       float sh, float sw, const void* __restrict__ labels, int label_dtype, int ignore_label,
                       unsigned long long* __restrict__ hist) {
    extern __shared__ unsigned int s_hist[];  // [C*C] when hist != nullptr
    if (hist) {
        for (int i = threadIdx.x; i < C * C; i += blockDim.x) s_hist[i] = 0u;
        __syncthreads();
    }
    const int groups_w = (OW + PXG - 1) / PXG;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int oh = blockIdx.y, n = blockIdx.z;
    if (g < groups_w) {
        const int ow0 = g * PXG;
        float best[PXG];
        int arg[PXG];
#pragma unroll
        for (int p = 0; p < PXG; ++p) {
            best[p] = -INFINITY;
            arg[p] = 0;
        }
        upsample_group8<EXACT8>(x, n, oh, g, IH, IW, C, OW, sh, sw, [&](int c, const float* v) {
#pragma unroll
            for (int p = 0; p < PXG; ++p)
                if (v[p] > best[p]) {  // strict: first maximum wins (torch.argmax)
                    best[p] = v[p];
                    arg[p] = c;
                }
        });
        const long long obase = (static_cast<long long>(n) * OH + oh) * OW + ow0;
        if (mask) {
            if ((OW % PXG) == 0) {
                uint32_t lo = arg[0] | (arg[1] << 8) | (arg[2] << 16) | (arg[3] << 24);
                uint32_t hi = arg[4] | (arg[5] << 8) | (arg[6] << 16) | (arg[7] << 24);
                *reinterpret_cast<uint2*>(mask + obase) = make_uint2(lo, hi);
            } else {
#pragma unroll
                for (int p = 0; p < PXG; ++p)
                    if (ow0 + p < OW) mask[obase + p] = static_cast<uint8_t>(arg[p]);
            }
        }
        if (hist) {
#pragma unroll
            for (int p = 0; p < PXG; ++p) {
                if (ow0 + p >= OW) continue;
                long long lb = label_dtype == 0 ? reinterpret_cast<const long long*>(labels)[obase + p]
                                                : static_cast<long long>(reinterpret_cast<const uint8_t*>(labels)[obase + p]);
                if (lb == ignore_label) continue;
                const int l = static_cast<int>(min(max(lb, 0LL), static_cast<long long>(C - 1)));
                atomicAdd(&s_hist[arg[p] * C + l], 1u);
            }
        }
    }
    if (hist) {
        __syncthreads();
        for (int i = threadIdx.x; i < C * C; i += blockDim.x)
            if (s_hist[i]) atomicAdd(&hist[i], static_cast<unsigned long long>(s_hist[i]));
    }
}

template <typename TP, typename TL>
__global__ void __launch_bounds__(256)
confusion_hist_kernel(const TP* __restrict__ pred, const TL* __restrict__ labels, long long n, int C, int ignore_label,
                      unsigned long long* __restrict__ hist) {
    extern __shared__ unsigned int s_hist[];
    for (int i = threadIdx.x; i < C * C; i += blockDim.x) s_hist[i] = 0u;
    __syncthreads();
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long lb = static_cast<long long>(labels[i]);
        if (lb == ignore_label) continue;
        const long long pr = static_cast<long long>(pred[i]);
        const int l = static_cast<int>(min(max(lb, 0LL), static_cast<long long>(C - 1)));
        const int p = static_cast<int>(min(max(pr, 0LL), static_cast<long long>(C - 1)));
        atomicAdd(&s_hist[p * C + l], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < C * C; i += blockDim.x)
        if (s_hist[i]) atomicAdd(&hist[i], static_cast<unsigned long long>(s_hist[i]));
}

// uint8 HWC image -> normalised fp32 NCHW: y[n][c][h][w] = (x[n][h][w][c] / 255 - mean[c]) / std[c]
// (torchvision ToTensor + Normalize of the reference datasets, src/datasets/uavid.py:175-183, cityscapes.py:102-109).
// One thread = 4 pixels: three 32-bit loads (12 bytes), three float4 stores (one per plane).
__global__ void __launch_bounds__(256)
normalize_u8_kernel(const uint8_t* __restrict__ x, float* __restrict__ y, long long HW4, long long HW, float m0, float m1,
                    float m2, float i0, float i1, float i2) {
    const int n = blockIdx.y;
    const long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (q >= HW4) return;
    const uint32_t* src = reinterpret_cast<const uint32_t*>(x + (static_cast<long long>(n) * HW + q * 4) * 3);
    const uint32_t w0 = __ldg(src), w1 = __ldg(src + 1), w2 = __ldg(src + 2);
    uint8_t b[12];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        b[i] = (w0 >> (8 * i)) & 0xff;
        b[4 + i] = (w1 >> (8 * i)) & 0xff;
        b[8 + i] = (w2 >> (8 * i)) & 0xff;
    }
    const float k = 1.f / 255.f;
    float* o = y + static_cast<long long>(n) * 3 * HW + q * 4;
    __stcs(reinterpret_cast<float4*>(o), make_float4((b[0] * k - m0) * i0, (b[3] * k - m0) * i0, (b[6] * k - m0) * i0,
                                                      (b[9] * k - m0) * i0));
    __stcs(reinterpret_cast<float4*>(o + HW), make_float4((b[1] * k - m1) * i1, (b[4] * k - m1) * i1,
                                                           (b[7] * k - m1) * i1, (b[10] * k - m1) * i1));
    __stcs(reinterpret_cast<float4*>(o + 2 * HW), make_float4((b[2] * k - m2) * i2, (b[5] * k - m2) * i2,
                                                               (b[8] * k - m2) * i2, (b[11] * k - m2) * i2));
}

// ---------------------------------------------------------------------------------- evaluator tail (MscEvalV0)
// eval_chip + the window accumulation of crop_eval (src/scripts/evaluate.py:74-87,139-146) in one pass over the
// probability planes: x8 bilinear of the chip's class map -> softmax over classes -> (average with the softmax of the
// horizontally flipped chip's map, read mirrored) -> weighted add into the window of the fp32 NCHW accumulator.
// The full-resolution logits, the two softmax outputs, the flipped copy and the chip-sized sum never reach HBM.
// Thread = 8 consecutive chip pixels of one row, all classes; the class map is evaluated twice (max + sum, then
// write): it is <= 1/64 of the output and L1/L2 resident.
template <bool EXACT8>
__device__ __forceinline__ void softmax_stats8(const float* __restrict__ x, int n, int oh, int g, int IH, int IW, int C,
                                               int OW, float sh, float sw, float* m, float* l) {
#pragma unroll
    for (int p = 0; p < PXG; ++p) {
        m[p] = -INFINITY;
        l[p] = 0.f;
    }
    upsample_group8<EXACT8>(x, n, oh, g, IH, IW, C, OW, sh, sw, [&](int, const float* v) {
#pragma unroll
        for (int p = 0; p < PXG; ++p) {  // online softmax: rescale the running sum when the maximum moves
            const float mn = fmaxf(m[p], v[p]);
            l[p] = l[p] * __expf(m[p] - mn) + __expf(v[p] - mn);
            m[p] = mn;
        }
    });
}

// FLIP is a template parameter: the plain variant keeps half the per-pixel state (64 instead of 126 registers,
// twice the resident warps: the kernel is latency bound at 25 % occupancy)
template <bool EXACT8, bool FLIP>
__global__ void __launch_bounds__(128, EXACT8 ? (FLIP ? 4 : 6) : 3)
upsample_softmax_accum_kernel(const float* __restrict__ x, const float* __restrict__ xf_arg, int IH, int IW, int C, int OH,
                              int OW, float sh, float sw, float* __restrict__ prob, long long sn, long long sc,
                              long long sr, int dy0, int dx0, int dh, int dw, const float* __restrict__ wy,
                              const float* __restrict__ wx, float weight) {
    const float* __restrict__ xf = FLIP ? xf_arg : nullptr;
    const int groups_w = (OW + PXG - 1) / PXG;
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    const int oh = blockIdx.y, n = blockIdx.z;
    const int y = dy0 + oh;
    if (g >= groups_w || y < 0 || y >= dh) return;
    const int ow0 = g * PXG;
    if (dx0 + ow0 >= dw || dx0 + ow0 + PXG <= 0) return;
    float m[PXG], l[PXG], mf[PXG], lf[PXG], k[PXG], kf[PXG];
    softmax_stats8<EXACT8>(x, n, oh, g, IH, IW, C, OW, sh, sw, m, l);
    const float rowk = weight * (wy ? __ldg(wy + oh) : 1.f) * (FLIP ? 0.5f : 1.f);
#pragma unroll
    for (int p = 0; p < PXG; ++p) k[p] = rowk * (wx ? __ldg(wx + min(ow0 + p, OW - 1)) : 1.f) / l[p];
    // mirrored group of the flipped chip's map: chip column ow <-> flipped column OW-1-ow.  With OW % 8 == 0 that
    // is group (groups_w-1-g) read back to front; otherwise the mirrored pixels straddle two groups -> per-pixel path.
    const bool mirror_fast = EXACT8 || (OW % PXG) == 0;
    const int gf = groups_w - 1 - g;
    if (FLIP && mirror_fast) {
        softmax_stats8<EXACT8>(xf, n, oh, gf, IH, IW, C, OW, sh, sw, mf, lf);
#pragma unroll
        for (int p = 0; p < PXG; ++p) kf[p] = k[PXG - 1 - p] * l[PXG - 1 - p] / lf[p];  // weight of mirrored pixel p
    }
    float* orow = prob + static_cast<long long>(n) * sn + static_cast<long long>(y) * sr + dx0 + ow0;
    const bool inside = dx0 + ow0 >= 0 && dx0 + ow0 + PXG <= dw && ow0 + PXG <= OW;
    auto emit = [&](int c, const float* pv) {
        float* o = orow + c * sc;
        if (inside && (reinterpret_cast<uintptr_t>(o) & 15) == 0) {
            float4 a = *reinterpret_cast<const float4*>(o), b = *(reinterpret_cast<const float4*>(o) + 1);
            a.x += pv[0]; a.y += pv[1]; a.z += pv[2]; a.w += pv[3];
            b.x += pv[4]; b.y += pv[5]; b.z += pv[6]; b.w += pv[7];
            *reinterpret_cast<float4*>(o) = a;
            *(reinterpret_cast<float4*>(o) + 1) = b;
        } else {
#pragma unroll
            for (int p = 0; p < PXG; ++p)
                if (ow0 + p < OW && dx0 + ow0 + p >= 0 && dx0 + ow0 + p < dw) o[p] += pv[p];
        }
    };
    if constexpr (EXACT8) {
        if (FLIP && (C & 3) == 0) {
            // both class maps per 4-class chunk, ONE read-modify-write of the window
            int y0, y1;
            float wyy;
            cab_bilinear_tap(oh, sh, IH, y0, y1, wyy);
            const float* r0 = x + (static_cast<long long>(n) * IH + y0) * IW * C;
            const float* r1 = x + (static_cast<long long>(n) * IH + y1) * IW * C;
            const float* q0 = xf + (static_cast<long long>(n) * IH + y0) * IW * C;
            const float* q1 = xf + (static_cast<long long>(n) * IH + y1) * IW * C;
            const int xa = max(g - 1, 0), xc = min(g + 1, IW - 1), fa = max(gf - 1, 0), fc = min(gf + 1, IW - 1);
            for (int c4 = 0; c4 < C; c4 += 4) {
                float v[4][PXG], vf[4][PXG];
                exact8_chunk4(r0, r1, xa, g, xc, C, c4, wyy, v);
                exact8_chunk4(q0, q1, fa, gf, fc, C, c4, wyy, vf);
#pragma unroll
                for (int k4 = 0; k4 < 4; ++k4) {
                    float pv[PXG];
#pragma unroll
                    for (int p = 0; p < PXG; ++p)
                        pv[p] = __expf(v[k4][p] - m[p]) * k[p] +
                                __expf(vf[k4][PXG - 1 - p] - mf[PXG - 1 - p]) * kf[PXG - 1 - p];
                    emit(c4 + k4, pv);
                }
            }
            return;
        }
    }
    if constexpr (!FLIP) {
        upsample_group8<EXACT8>(x, n, oh, g, IH, IW, C, OW, sh, sw, [&](int c, const float* v) {
            float pv[PXG];
#pragma unroll
            for (int p = 0; p < PXG; ++p) pv[p] = __expf(v[p] - m[p]) * k[p];
            emit(c, pv);
        });
    } else if (mirror_fast) {
        // two sweeps over the classes (plain, mirrored): the consumer interface hands out one class at a time, and the
        // window is L1/L2-hot for the second read-modify-write
        upsample_group8<EXACT8>(x, n, oh, g, IH, IW, C, OW, sh, sw, [&](int c, const float* v) {
            float pv[PXG];
#pragma unroll
            for (int p = 0; p < PXG; ++p) pv[p] = __expf(v[p] - m[p]) * k[p];
            emit(c, pv);
        });
        upsample_group8<EXACT8>(xf, n, oh, gf, IH, IW, C, OW, sh, sw, [&](int c, const float* v) {
            float pv[PXG];
#pragma unroll
            for (int p = 0; p < PXG; ++p) pv[PXG - 1 - p] = __expf(v[p] - mf[p]) * kf[p];
            emit(c, pv);
        });
    } else if constexpr (!EXACT8) {
        upsample_group8<EXACT8>(x, n, oh, g, IH, IW, C, OW, sh, sw, [&](int c, const float* v) {
            float pv[PXG];
#pragma unroll
            for (int p = 0; p < PXG; ++p) pv[p] = __expf(v[p] - m[p]) * k[p];
            emit(c, pv);
        });
        // generic mirrored read: one flipped-map pixel at a time (chip widths that are not a multiple of 8)
        int y0, y1;
        float wyy;
        cab_bilinear_tap(oh, sh, IH, y0, y1, wyy);
        const float* r0 = xf + (static_cast<long long>(n) * IH + y0) * IW * C;
        const float* r1 = xf + (static_cast<long long>(n) * IH + y1) * IW * C;
#pragma unroll
        for (int p = 0; p < PXG; ++p) {
            const int ow = ow0 + p;
            if (ow >= OW || dx0 + ow < 0 || dx0 + ow >= dw) continue;
            int x0, x1;
            float wxx;
            cab_bilinear_tap(OW - 1 - ow, sw, IW, x0, x1, wxx);
            float mm = -INFINITY, ll = 0.f;
            for (int c = 0; c < C; ++c) {
                const float t0 = __ldg(r0 + x0 * C + c), t1 = __ldg(r0 + x1 * C + c);
                const float b0 = __ldg(r1 + x0 * C + c), b1 = __ldg(r1 + x1 * C + c);
                const float top = t0 + wxx * (t1 - t0), bot = b0 + wxx * (b1 - b0);
                const float v = top + wyy * (bot - top);
                const float mn = fmaxf(mm, v);
                ll = ll * __expf(mm - mn) + __expf(v - mn);
                mm = mn;
            }
            const float kk = k[p] * l[p] / ll;
            for (int c = 0; c < C; ++c) {
                const float t0 = __ldg(r0 + x0 * C + c), t1 = __ldg(r0 + x1 * C + c);
                const float b0 = __ldg(r1 + x0 * C + c), b1 = __ldg(r1 + x1 * C + c);
                const float top = t0 + wxx * (t1 - t0), bot = b0 + wxx * (b1 - b0);
                const float v = top + wyy * (bot - top);
                orow[c * sc + p] += __expf(v - mm) * kk;
            }
        }
    }
}

// dst[n][c][y][x] += bilinear(src[n][c][cy0 : cy0+ch][cx0 : cx0+cw] -> (H, W))   (align_corners=False): the un-pad crop
// and the resize back to the image size of scale_crop_eval plus `probs += prob` of evaluate()
// (src/scripts/evaluate.py:152-158,216-220) in one pass.  Thread = one output pixel, all classes (taps computed once).
__global__ void __launch_bounds__(256)
prob_resize_accum_kernel(const float* __restrict__ src, int C, int SH, int SW, int cy0, int cx0, int ch, int cw,
                         float* __restrict__ dst, int H, int W, float sh, float sw) {
    // thread = 4 consecutive output pixels of one row, all classes: taps once, one 16-byte read-modify-write per class
    const int xq = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (xq >= W) return;
    const int yo = blockIdx.y, n = blockIdx.z;
    int y0, y1, x0[4], x1[4];
    float wy, wx[4];
    cab_bilinear_tap(yo, sh, ch, y0, y1, wy);
#pragma unroll
    for (int p = 0; p < 4; ++p) cab_bilinear_tap(min(xq + p, W - 1), sw, cw, x0[p], x1[p], wx[p]);
    const long long plane_s = static_cast<long long>(SH) * SW, plane_d = static_cast<long long>(H) * W;
    const float* s0 = src + static_cast<long long>(n) * C * plane_s + static_cast<long long>(cy0 + y0) * SW + cx0;
    const float* s1 = src + static_cast<long long>(n) * C * plane_s + static_cast<long long>(cy0 + y1) * SW + cx0;
    float* d = dst + static_cast<long long>(n) * C * plane_d + static_cast<long long>(yo) * W + xq;
    const bool vec = xq + 4 <= W && (reinterpret_cast<uintptr_t>(d) & 15) == 0 && (plane_d & 3) == 0;
    for (int c = 0; c < C; ++c) {
        const float* a = s0 + c * plane_s;
        const float* b = s1 + c * plane_s;
        float r[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            // ATen's expression: h0 * (w0 * a + w1 * b) + h1 * (w0 * c + w1 * d)
            const float top = (1.f - wx[p]) * __ldg(a + x0[p]) + wx[p] * __ldg(a + x1[p]);
            const float bot = (1.f - wx[p]) * __ldg(b + x0[p]) + wx[p] * __ldg(b + x1[p]);
            r[p] = (1.f - wy) * top + wy * bot;
        }
        float* o = d + c * plane_d;
        if (vec) {
            float4 t = *reinterpret_cast<const float4*>(o);
            t.x += r[0]; t.y += r[1]; t.z += r[2]; t.w += r[3];
            *reinterpret_cast<float4*>(o) = t;
        } else {
#pragma unroll
            for (int p = 0; p < 4; ++p)
                if (xq + p < W) o[p] += r[p];
        }
    }
}

// argmax over the class planes of an fp32 NCHW probability map (first maximum wins, torch.argmax) fused with the
// confusion matrix (src/scripts/evaluate.py:222-228,162-191): the int64 prediction map is never written.
template <typename TL>
__global__ void __launch_bounds__(256)
argmax_hist_nchw_kernel(const float* __restrict__ probs, int C, long long HW, uint8_t* __restrict__ mask,
                        const TL* __restrict__ labels, int ignore_label, unsigned long long* __restrict__ hist) {
    extern __shared__ unsigned int s_hist[];
    if (hist) {
        for (int i = threadIdx.x; i < C * C; i += blockDim.x) s_hist[i] = 0u;
        __syncthreads();
    }
    const int n = blockIdx.y;
    const float* base = probs + static_cast<long long>(n) * C * HW;
    const bool vec = (HW & 3) == 0 && (reinterpret_cast<uintptr_t>(probs) & 15) == 0 && (reinterpret_cast<uintptr_t>(mask) & 3) == 0;
    const long long HWv = vec ? HW / 4 : 0;
    for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < HWv;
         q += static_cast<long long>(gridDim.x) * blockDim.x) {
        const float4 f = __ldcs(reinterpret_cast<const float4*>(base) + q);
        float best[4] = {f.x, f.y, f.z, f.w};
        int arg[4] = {0, 0, 0, 0};
        for (int c = 1; c < C; ++c) {
            const float4 t = __ldcs(reinterpret_cast<const float4*>(base + c * HW) + q);
            const float v[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
            for (int p = 0; p < 4; ++p)
                if (v[p] > best[p]) {
                    best[p] = v[p];
                    arg[p] = c;
                }
        }
        const long long o = static_cast<long long>(n) * HW + q * 4;
        if (mask) *reinterpret_cast<uint32_t*>(mask + o) = arg[0] | (arg[1] << 8) | (arg[2] << 16) | (arg[3] << 24);
        if (hist) {
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const long long lb = static_cast<long long>(labels[o + p]);
                if (lb != ignore_label) {
                    const int lc = static_cast<int>(min(max(lb, 0LL), static_cast<long long>(C - 1)));
                    atomicAdd(&s_hist[arg[p] * C + lc], 1u);
                }
            }
        }
    }
    for (long long i = (vec ? HW : 0) + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < HW;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        float best = __ldg(base + i);
        int arg = 0;
        for (int c = 1; c < C; ++c) {
            const float v = __ldg(base + c * HW + i);
            if (v > best) {
                best = v;
                arg = c;
            }
        }
        const long long o = static_cast<long long>(n) * HW + i;
        if (mask) mask[o] = static_cast<uint8_t>(arg);
        if (hist) {
            const long long lb = static_cast<long long>(labels[o]);
            if (lb != ignore_label) {
                const int lc = static_cast<int>(min(max(lb, 0LL), static_cast<long long>(C - 1)));
                atomicAdd(&s_hist[arg * C + lc], 1u);
            }
        }
    }
    if (hist) {
        __syncthreads();
        for (int i = threadIdx.x; i < C * C; i += blockDim.x)
            if (s_hist[i]) atomicAdd(&hist[i], static_cast<unsigned long long>(s_hist[i]));
    }
}

}  // namespace

extern "C" int cabinet_upsample_softmax_accum(const float* x, const float* x_flip, int N, int IH, int IW, int C, int OH,
                                              int OW, float* prob, long long stride_n, long long stride_c,
                                              long long stride_row, int dst_y0, int dst_x0, int dst_h, int dst_w,
                                              const float* weight_y, const float* weight_x, float weight,
                                              cabinet_stream_t stream) {
    CAB_REQUIRE(x && prob && IH > 0 && IW > 0 && OH > 0 && OW > 0 && C > 0 && dst_h > 0 && dst_w > 0,
                "upsample_softmax_accum: bad arguments");
    CAB_REQUIRE(OH <= 65535 && N <= 65535, "upsample_softmax_accum: OH/N exceed grid limits");
    if (N == 0) return CABINET_OK;
    const float sh = static_cast<float>(IH) / static_cast<float>(OH), sw = static_cast<float>(IW) / static_cast<float>(OW);
    const bool exact8 = OH == 8 * IH && OW == 8 * IW;
    const int groups = (OW + PXG - 1) / PXG;
    dim3 grid((groups + 127) / 128, OH, N);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define CAB_USA(E8, FL)                                                                                              \
    upsample_softmax_accum_kernel<E8, FL><<<grid, 128, 0, s>>>(x, x_flip, IH, IW, C, OH, OW, sh, sw, prob, stride_n,    \
                                                               stride_c, stride_row, dst_y0, dst_x0, dst_h, dst_w,      \
                                                               weight_y, weight_x, weight)
    if (exact8) {
        if (x_flip) CAB_USA(true, true); else CAB_USA(true, false);
    } else {
        if (x_flip) CAB_USA(false, true); else CAB_USA(false, false);
    }
#undef CAB_USA
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_prob_resize_accum(const float* src, int N, int C, int src_h, int src_w, int crop_y0, int crop_x0,
                                         int crop_h, int crop_w, float* dst, int H, int W, cabinet_stream_t stream) {
    CAB_REQUIRE(src && dst && C > 0 && crop_h > 0 && crop_w > 0 && H > 0 && W > 0 && crop_y0 >= 0 && crop_x0 >= 0 &&
                    crop_y0 + crop_h <= src_h && crop_x0 + crop_w <= src_w,
                "prob_resize_accum: bad arguments");
    CAB_REQUIRE(H <= 65535 && N <= 65535, "prob_resize_accum: H/N exceed grid limits");
    if (N == 0) return CABINET_OK;
    const float sh = static_cast<float>(crop_h) / static_cast<float>(H), sw = static_cast<float>(crop_w) / static_cast<float>(W);
    dim3 grid((W + 1023) / 1024, H, N);
    prob_resize_accum_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(src, C, src_h, src_w, crop_y0, crop_x0,
                                                                                 crop_h, crop_w, dst, H, W, sh, sw);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_argmax_hist_nchw(const float* probs, int N, int C, long long HW, uint8_t* mask,
                                        const void* labels, int label_dtype, int ignore_label, long long* hist,
                                        cabinet_stream_t stream) {
    CAB_REQUIRE(probs && (mask || hist) && C > 0 && C <= 255 && HW > 0, "argmax_hist_nchw: bad arguments (1 <= C <= 255)");
    CAB_REQUIRE(!hist || labels, "argmax_hist_nchw: hist requested without labels");
    CAB_REQUIRE(C * C * sizeof(unsigned) <= 48 * 1024, "argmax_hist_nchw: C*C histogram does not fit shared memory");
    CAB_REQUIRE(N <= 65535, "argmax_hist_nchw: N exceeds grid limits");
    if (N == 0) return CABINET_OK;
    dim3 grid(static_cast<unsigned>(std::min<long long>(cab_ceil_div(HW, 256 * 4), 148 * 16)), N);
    const size_t smem = hist ? sizeof(unsigned) * C * C : 0;
    auto* h = reinterpret_cast<unsigned long long*>(hist);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (label_dtype == 0)
        argmax_hist_nchw_kernel<long long><<<grid, 256, smem, s>>>(probs, C, HW, mask, reinterpret_cast<const long long*>(labels),
                                                                   ignore_label, h);
    else
        argmax_hist_nchw_kernel<uint8_t><<<grid, 256, smem, s>>>(probs, C, HW, mask, reinterpret_cast<const uint8_t*>(labels),
                                                                 ignore_label, h);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_normalize_u8(const uint8_t* x, float* y, int N, int H, int W, float mean0, float mean1,
                                    float mean2, float std0, float std1, float std2, cabinet_stream_t stream) {
    CAB_REQUIRE(x && y && H > 0 && W > 0 && N >= 0 && N <= 65535, "normalize_u8: bad arguments");
    const long long HW = static_cast<long long>(H) * W;
    CAB_REQUIRE(HW % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 3) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0,
                "normalize_u8: H*W must be a multiple of 4 and the buffers aligned");
    CAB_REQUIRE(std0 > 0 && std1 > 0 && std2 > 0, "normalize_u8: std must be positive");
    if (N == 0) return CABINET_OK;
    dim3 grid(static_cast<unsigned>(cab_ceil_div(HW / 4, 256)), N);
    normalize_u8_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, HW / 4, HW, mean0, mean1, mean2,
                                                                             1.f / std0, 1.f / std1, 1.f / std2);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_bilinear_nhwc(const void* x, long long ldx, int x_dtype, void* y, long long ldy, int y_dtype,
                                     int N, int IH, int IW, int C, int OH, int OW, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("bilinear_nhwc", x_dtype, CAB_DT_F32 | CAB_DT_BF16);
    CAB_REQUIRE_DTYPE("bilinear_nhwc", y_dtype, CAB_DT_F32 | CAB_DT_BF16);
    CAB_REQUIRE(x && y && IH > 0 && IW > 0 && OH > 0 && OW > 0 && C > 0 && ldx >= C && ldy >= C,
                "bilinear_nhwc: bad arguments");
    if (N == 0) return CABINET_OK;
    const float sh = static_cast<float>(IH) / static_cast<float>(OH), sw = static_cast<float>(IW) / static_cast<float>(OW);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (x_dtype == CABINET_BF16 && y_dtype == CABINET_BF16 && C % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 &&
        (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0) {
        CAB_REQUIRE(OH <= 65535 && N <= 65535, "bilinear_nhwc: OH/N exceed grid limits");
        if (OH == 4 * IH && OW == 4 * IW) {
            dim3 g4(static_cast<unsigned>(cab_ceil_div(static_cast<long long>(IW) * (C / 8), 256)), IH, N);
            bilinear_x4_bf16_kernel<<<g4, 256, 0, s>>>(reinterpret_cast<const bf16*>(x), ldx, reinterpret_cast<bf16*>(y),
                                                       ldy, IH, IW, C);
            CAB_LAUNCH_CHECK();
            return CABINET_OK;
        }
        dim3 g8(static_cast<unsigned>(cab_ceil_div(static_cast<long long>(OW) * (C / 8), 256)), OH, N);
        bilinear_nhwc_bf16x8_kernel<<<g8, 256, 0, s>>>(reinterpret_cast<const bf16*>(x), ldx, reinterpret_cast<bf16*>(y),
                                                       ldy, IH, IW, C, OH, OW, sh, sw);
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    const long long total = static_cast<long long>(N) * OH * OW * ((C + 3) / 4);
    dim3 grid(static_cast<unsigned>(cab_ceil_div(total, 256)));
#define CAB_BL(TI, TO)                                                                                       \
    bilinear_nhwc_kernel<TI, TO><<<grid, 256, 0, s>>>(reinterpret_cast<const TI*>(x), ldx,                   \
                                                      reinterpret_cast<TO*>(y), ldy, IH, IW, C, OH, OW, total, sh, sw)
    if (x_dtype == CABINET_F32 && y_dtype == CABINET_F32) CAB_BL(float, float);
    else if (x_dtype == CABINET_F32) CAB_BL(float, bf16);
    else if (y_dtype == CABINET_F32) CAB_BL(bf16, float);
    else CAB_BL(bf16, bf16);
#undef CAB_BL
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_upsample_logits_nchw(const float* x, int N, int IH, int IW, int C, void* y, int y_dtype, int OH,
                                            int OW, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("upsample_logits_nchw", y_dtype, CAB_DT_F32 | CAB_DT_BF16);
    CAB_REQUIRE(x && y && IH > 0 && IW > 0 && OH > 0 && OW > 0 && C > 0, "upsample_logits_nchw: bad arguments");
    CAB_REQUIRE(OH <= 65535 && N <= 65535, "upsample_logits_nchw: OH/N exceed grid limits");
    if (N == 0) return CABINET_OK;
    const float sh = static_cast<float>(IH) / static_cast<float>(OH), sw = static_cast<float>(IW) / static_cast<float>(OW);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool exact8 = OH == 8 * IH && OW == 8 * IW;
    const int groups = (OW + PXG - 1) / PXG;
    dim3 grid((groups + 127) / 128, OH, N);
#define CAB_UP(TO, E8) \
    upsample_logits_nchw_kernel<TO, E8><<<grid, 128, 0, s>>>(x, IH, IW, C, reinterpret_cast<TO*>(y), OH, OW, sh, sw)
    if (y_dtype == CABINET_F32) {
        if (exact8) CAB_UP(float, true); else CAB_UP(float, false);
    } else {
        if (exact8) CAB_UP(bf16, true); else CAB_UP(bf16, false);
    }
#undef CAB_UP
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_upsample_argmax(const float* x, int N, int IH, int IW, int C, uint8_t* mask, int OH, int OW,
                                       const void* labels, int label_dtype, int ignore_label, long long* hist,
                                       cabinet_stream_t stream) {
    CAB_REQUIRE(x && (mask || hist) && IH > 0 && IW > 0 && OH > 0 && OW > 0 && C > 0 && C <= 255,
                "upsample_argmax: bad arguments (1 <= C <= 255)");
    CAB_REQUIRE(!hist || labels, "upsample_argmax: hist requested without labels");
    CAB_REQUIRE(C * C * sizeof(unsigned) <= 48 * 1024, "upsample_argmax: C*C histogram does not fit shared memory");
    CAB_REQUIRE(OH <= 65535 && N <= 65535, "upsample_argmax: OH/N exceed grid limits");
    if (N == 0) return CABINET_OK;
    const float sh = static_cast<float>(IH) / static_cast<float>(OH), sw = static_cast<float>(IW) / static_cast<float>(OW);
    const bool exact8 = OH == 8 * IH && OW == 8 * IW;
    const int groups = (OW + PXG - 1) / PXG;
    dim3 grid((groups + 127) / 128, OH, N);
    const size_t smem = hist ? sizeof(unsigned) * C * C : 0;
    auto* h = reinterpret_cast<unsigned long long*>(hist);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (exact8)
        upsample_argmax_kernel<true><<<grid, 128, smem, s>>>(x, IH, IW, C, mask, OH, OW, sh, sw, labels, label_dtype,
                                                            ignore_label, h);
    else
        upsample_argmax_kernel<false><<<grid, 128, smem, s>>>(x, IH, IW, C, mask, OH, OW, sh, sw, labels, label_dtype,
                                                             ignore_label, h);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_confusion_hist(const void* pred, int pred_dtype, const void* labels, int label_dtype,
                                      long long n_pixels, int C, int ignore_label, long long* hist,
                                      cabinet_stream_t stream) {
    CAB_REQUIRE(pred && labels && hist && C > 0 && C * C * sizeof(unsigned) <= 48 * 1024,
                "confusion_hist: bad arguments");
    if (n_pixels == 0) return CABINET_OK;
    dim3 grid(static_cast<unsigned>(std::min<long long>(cab_ceil_div(n_pixels, 256 * 16), 148 * 8)));
    grid.x = grid.x ? grid.x : 1;
    const size_t smem = sizeof(unsigned) * C * C;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    auto* h = reinterpret_cast<unsigned long long*>(hist);
#define CAB_CH(TP, TL)                                                                                             \
    confusion_hist_kernel<TP, TL><<<grid, 256, smem, s>>>(reinterpret_cast<const TP*>(pred),                       \
                                                          reinterpret_cast<const TL*>(labels), n_pixels, C, ignore_label, h)
    if (pred_dtype == 0 && label_dtype == 0) CAB_CH(long long, long long);
    else if (pred_dtype == 0) CAB_CH(long long, uint8_t);
    else if (label_dtype == 0) CAB_CH(uint8_t, long long);
    else CAB_CH(uint8_t, uint8_t);
#undef CAB_CH
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}
