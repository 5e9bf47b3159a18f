// OHEM cross-entropy (src/utils/loss.py:38-80, the training loss of src/scripts/train.py:344-349,435) without a sort.
//
// The reference computes a per-pixel CE map, sorts all valid losses (8.4 M elements at 8 x 1024^2) and takes either
// everything above `thresh` or the `n_min` largest.  Here:
//   ohem_ce_px_kernel     one pass over the NCHW logits: l = w[y] * (logsumexp(x) - x[y]) per valid pixel -> loss_px
//                         (fp32, -1 marks ignored pixels) + #valid, #(l > thresh), sum(l > thresh) + the first level of
//                         a radix histogram over the float bit patterns (l >= 0, so the unsigned order is the float order)
//   ohem_pick_kernel      one block: "k-th largest > thresh" <=> "#(l > thresh) >= k", k = min(n_min, #valid).  If so the
//                         loss is sum/count of the thresholded set.  Otherwise walk the histogram from the top to the
//                         bin holding the k-th largest value and refine it (levels 2 and 3: ohem_hist_kernel over
//                         loss_px restricted to the chosen prefix) down to its exact 31-bit pattern v_k; then
//                         top-k sum = sum(l > v_k) [ohem_sum_above_kernel] + (k - #(l > v_k)) * v_k, exactly what the
//                         sorted prefix sums to.
//   ohem_ce_bwd_kernel    d loss / d logits = g * coef_i * w[y] * (softmax(x) - onehot(y)), coef_i = 1/M on the selected
//                         set (ties at v_k share the remaining (k - #(l > v_k)) / #(l == v_k) -- a sort would pick an
//                         arbitrary subset of equal losses; the loss value is identical).
// Everything stays on the device (no host round trip decides between the two cases); counts are integers and the
// sums are accumulated in double, so the result does not depend on the block schedule beyond fp64 round-off.
#include "common.cuh"

namespace {

constexpr int L1_BINS = 2048, L2_BINS = 2048, L3_BINS = 512;  // bits [30:20] | [19:9] | [8:0]

struct OhemWs {
    unsigned int hist[3][2048];
    unsigned long long n_valid, n_gt;
    double sum_gt;
    // selection state (written by the pick kernels, read by the later levels and by the backward pass)
    int mode;                  // 0: not decided yet, 1: no valid pixel, 2: thresholded set, 3: top-k (radix select running)
    unsigned int prefix;       // bit pattern of v_k decided so far
    unsigned long long k, k_rem;
    double sum_above;
    float sel_thresh;          // select l > sel_thresh ...
    float tie_value, tie_frac; // ... plus tie_frac of the pixels with l == tie_value
    float inv_m, loss;
    unsigned int n_nonfinite;  // valid pixels whose loss is NaN / Inf (overflowed logits): the loss and the gradients become NaN
};

template <typename T> __device__ __forceinline__ float ld_logit(const T* p);
template <> __device__ __forceinline__ float ld_logit<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ld_logit<bf16>(const bf16* p) {
    return __uint_as_float(static_cast<uint32_t>(__ldg(reinterpret_cast<const unsigned short*>(p))) << 16);
}

// 4 consecutive pixels of one class plane (16-byte / 8-byte aligned)
template <typename T> __device__ __forceinline__ void ld_logit4(const T* p, float* v);
template <> __device__ __forceinline__ void ld_logit4<float>(const float* p, float* v) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
template <> __device__ __forceinline__ void ld_logit4<bf16>(const bf16* p, float* v) {
    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p));
    v[0] = __uint_as_float(t.x << 16); v[1] = __uint_as_float(t.x & 0xffff0000u);
    v[2] = __uint_as_float(t.y << 16); v[3] = __uint_as_float(t.y & 0xffff0000u);
}
template <typename T> __device__ __forceinline__ void st_grad4(T* p, const float* v);
template <> __device__ __forceinline__ void st_grad4<float>(float* p, const float* v) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(v[0], v[1], v[2], v[3]));
}
template <> __device__ __forceinline__ void st_grad4<bf16>(bf16* p, const float* v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
    __stcs(reinterpret_cast<uint2*>(p), make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b)));
}

// max and sum(exp(x - max)) over the classes for 4 consecutive pixels (second sweep hits L1)
template <typename T>
__device__ __forceinline__ void softmax_stats4(const T* __restrict__ x, int C, long long HW, float* m, float* s) {
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        m[p] = -INFINITY;
        s[p] = 0.f;
    }
    for (int c = 0; c < C; ++c) {
        float v[4];
        ld_logit4<T>(x + c * HW, v);
#pragma unroll
        for (int p = 0; p < 4; ++p) m[p] = fmaxf(m[p], v[p]);
    }
    for (int c = 0; c < C; ++c) {
        float v[4];
        ld_logit4<T>(x + c * HW, v);
#pragma unroll
        for (int p = 0; p < 4; ++p) s[p] += expf(v[p] - m[p]);
    }
}

__device__ __forceinline__ long long ld_label(const void* labels, int label_dtype, long long i) {
    return label_dtype == 0 ? __ldg(reinterpret_cast<const long long*>(labels) + i)
                            : static_cast<long long>(__ldg(reinterpret_cast<const uint8_t*>(labels) + i));
}

// per-pixel weighted cross-entropy of pixel (n, i); returns -1 for ignored / out-of-range labels
template <typename T>
__device__ __forceinline__ float pixel_ce(const T* __restrict__ x, int C, long long HW, long long lb,
                                          const float* __restrict__ weight, float* m_out, float* l_out) {
    float m = -INFINITY;
    for (int c = 0; c < C; ++c) m = fmaxf(m, ld_logit<T>(x + c * HW));
    float s = 0.f;
    for (int c = 0; c < C; ++c) s += expf(ld_logit<T>(x + c * HW) - m);
    if (m_out) {
        *m_out = m;
        *l_out = s;
    }
    if (lb < 0 || lb >= C) return -1.f;
    const float w = weight ? __ldg(weight + lb) : 1.f;
    // clamp fp32 round-off below zero and clear a -0.0 sign: the radix select orders losses by their bit patterns
    return __uint_as_float(__float_as_uint(fmaxf(w * (m + logf(s) - ld_logit<T>(x + lb * HW)), 0.f)) & 0x7fffffffu);
}

template <typename T>
__global__ void __launch_bounds__(256)
ohem_ce_px_kernel(const T* __restrict__ logits, const void* __restrict__ labels, int label_dtype, int C, long long HW,
                  const float* __restrict__ weight, int ignore_label, float thresh, float* __restrict__ loss_px,
                  OhemWs* __restrict__ ws) {
    __shared__ unsigned int s_hist[L1_BINS];
    __shared__ unsigned long long s_cnt[2];
    __shared__ double s_gt;
    for (int i = threadIdx.x; i < L1_BINS; i += blockDim.x) s_hist[i] = 0u;
    if (threadIdx.x < 2) s_cnt[threadIdx.x] = 0ull;
    if (threadIdx.x == 0) s_gt = 0.0;
    __syncthreads();
    const int n = blockIdx.y;
    const T* base = logits + static_cast<long long>(n) * C * HW;
    unsigned long long nv = 0, ng = 0;
    unsigned int bad = 0;
    double sg = 0.0;
    // 4 pixels per thread when every class plane is 16-byte aligned (HW % 8 == 0 covers bf16 too)
    const bool vec = (HW & 7) == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(loss_px) & 15) == 0;
    const long long HWv = vec ? HW / 4 : 0;
    for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < HWv;
         q += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long i = q * 4, o = static_cast<long long>(n) * HW + i;
        float m[4], s[4], l[4];
        softmax_stats4<T>(base + i, C, HW, m, s);
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            const long long lb = ld_label(labels, label_dtype, o + p);
            l[p] = -1.f;
            if (lb != ignore_label && lb >= 0 && lb < C) {
                const float w = weight ? __ldg(weight + lb) : 1.f;
                const float raw = w * (m[p] + logf(s[p]) - ld_logit<T>(base + lb * HW + i + p));
                if (!isfinite(raw)) ++bad;  // fmaxf would turn a NaN into 0: the reference propagates it (GradScaler then skips the step)
                const float v = fmaxf(raw, 0.f);
                l[p] = __uint_as_float(__float_as_uint(v) & 0x7fffffffu);
                ++nv;
                if (l[p] > thresh) {
                    ++ng;
                    sg += l[p];
                }
                atomicAdd(&s_hist[__float_as_uint(l[p]) >> 20], 1u);
            }
        }
        *reinterpret_cast<float4*>(loss_px + o) = make_float4(l[0], l[1], l[2], l[3]);
    }
    for (long long i = (vec ? HW : 0) + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < HW;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long o = static_cast<long long>(n) * HW + i;
        const long long lb = ld_label(labels, label_dtype, o);
        float l = -1.f;
        if (lb != ignore_label) {
            float mm, ss;
            l = pixel_ce<T>(base + i, C, HW, lb, weight, &mm, &ss);
            if (l >= 0.f && !(isfinite(l) && isfinite(mm) && isfinite(ss) && ss > 0.f)) ++bad;
        }
        loss_px[o] = l;
        if (l >= 0.f) {
            ++nv;
            if (l > thresh) {
                ++ng;
                sg += l;
            }
            atomicAdd(&s_hist[__float_as_uint(l) >> 20], 1u);
        }
    }
    if (bad) atomicAdd(&ws->n_nonfinite, bad);
    // block reduction of the three scalars (warp shuffles, then one shared atomic per warp)
    for (int d = 16; d > 0; d >>= 1) {
        nv += __shfl_down_sync(0xffffffffu, nv, d);
        ng += __shfl_down_sync(0xffffffffu, ng, d);
        sg += __shfl_down_sync(0xffffffffu, sg, d);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&s_cnt[0], nv);
        atomicAdd(&s_cnt[1], ng);
        atomicAdd(&s_gt, sg);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < L1_BINS; i += blockDim.x)
        if (s_hist[i]) atomicAdd(&ws->hist[0][i], s_hist[i]);
    if (threadIdx.x == 0) {
        atomicAdd(&ws->n_valid, s_cnt[0]);
        atomicAdd(&ws->n_gt, s_cnt[1]);
        atomicAdd(&ws->sum_gt, s_gt);
    }
}

// histogram of level `level` (1 or 2) over the losses whose higher bits equal the prefix chosen so far
__global__ void __launch_bounds__(256)
ohem_hist_kernel(const float* __restrict__ loss_px, long long total, int level, OhemWs* __restrict__ ws) {
    if (ws->mode != 3) return;  // thresholded set or no valid pixel: nothing to refine
    __shared__ unsigned int s_hist[2048];
    for (int i = threadIdx.x; i < 2048; i += blockDim.x) s_hist[i] = 0u;
    __syncthreads();
    const unsigned int prefix = ws->prefix;
    const int hi_shift = level == 1 ? 20 : 9, lo_shift = level == 1 ? 9 : 0;
    const unsigned int lo_mask = level == 1 ? 0x7ffu : 0x1ffu;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const float l = __ldg(loss_px + i);
        if (l < 0.f) continue;
        const unsigned int u = __float_as_uint(l);
        if ((u >> hi_shift) != (prefix >> hi_shift)) continue;
        atomicAdd(&s_hist[(u >> lo_shift) & lo_mask], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2048; i += blockDim.x)
        if (s_hist[i]) atomicAdd(&ws->hist[level][i], s_hist[i]);
}

// sum of the losses strictly above v_k (top-k case only), fp64 block partials
__global__ void __launch_bounds__(256)
ohem_sum_above_kernel(const float* __restrict__ loss_px, long long total, OhemWs* __restrict__ ws) {
    if (ws->mode != 3) return;
    __shared__ double s_part[8];
    const float vk = ws->sel_thresh;
    double acc = 0.0;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const float l = __ldg(loss_px + i);
        if (l > vk) acc += l;
    }
    for (int d = 16; d > 0; d >>= 1) acc += __shfl_down_sync(0xffffffffu, acc, d);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += s_part[w];
        if (t != 0.0) atomicAdd(&ws->sum_above, t);
    }
}

__global__ void ohem_finish_kernel(OhemWs* __restrict__ ws, float* __restrict__ loss_out) {
    if (ws->mode != 3) return;
    const double k = static_cast<double>(ws->k);
    ws->loss = static_cast<float>((ws->sum_above + static_cast<double>(ws->k_rem) * static_cast<double>(ws->tie_value)) / k);
    *loss_out = ws->loss;
}

// Non-finite per-pixel losses (NaN / Inf logits): the loss becomes NaN, as with the reference's F.cross_entropy.
__global__ void ohem_nonfinite_kernel(OhemWs* __restrict__ ws, float* __restrict__ loss_out) {
    if (ws->n_nonfinite) {
        ws->loss = __int_as_float(0x7fc00000);
        *loss_out = ws->loss;
    }
}

// One block of 1024 threads.  level 0 also decides the mode; level 2 finishes the selection and writes the loss.
__global__ void __launch_bounds__(1024)
ohem_pick_kernel(int level, float thresh, long long n_min, OhemWs* __restrict__ ws, float* __restrict__ loss_out) {
    __shared__ unsigned long long s_cnt[2048];
    const int t = threadIdx.x;
    if (level == 0) {
        if (t == 0) {
            const unsigned long long nv = ws->n_valid, ng = ws->n_gt;
            const unsigned long long k = nv < static_cast<unsigned long long>(n_min) ? nv : static_cast<unsigned long long>(n_min);
            ws->k = k;
            ws->k_rem = k;
            ws->sum_above = 0.0;
            ws->prefix = 0u;
            ws->tie_frac = 0.f;
            ws->tie_value = -2.f;
            if (nv == 0) {  // loss.py:61-62
                ws->mode = 1;
                ws->sel_thresh = INFINITY;
                ws->inv_m = 0.f;
                ws->loss = 0.f;
                *loss_out = 0.f;
            } else if (ng >= k) {  // sorted[k-1] > thresh  (loss.py:71-72): every loss above the threshold
                ws->mode = 2;
                ws->sel_thresh = thresh;
                ws->inv_m = static_cast<float>(1.0 / static_cast<double>(ng));
                ws->loss = static_cast<float>(ws->sum_gt / static_cast<double>(ng));
                *loss_out = ws->loss;
            } else {
                ws->mode = 3;  // the k largest (loss.py:73-74)
            }
        }
        __syncthreads();
    }
    if (ws->mode != 3) return;
    const int bins = level == 2 ? L3_BINS : 2048;
    // suffix sums (from the largest bin down) of counts and sums: Hillis-Steele over 2048 entries, 2 per thread
    for (int i = t; i < 2048; i += 1024) s_cnt[i] = i < bins ? ws->hist[level][i] : 0ull;
    __syncthreads();
    for (int d = 1; d < 2048; d <<= 1) {
        unsigned long long c[2];
        for (int j = 0; j < 2; ++j) {
            const int i = t + j * 1024;
            c[j] = s_cnt[i] + (i + d < 2048 ? s_cnt[i + d] : 0ull);
        }
        __syncthreads();
        for (int j = 0; j < 2; ++j) s_cnt[t + j * 1024] = c[j];
        __syncthreads();
    }
    // the bin b with suffix(b) >= k_rem > suffix(b + 1) holds the k_rem-th largest of this level
    const unsigned long long k_rem = ws->k_rem;
    __syncthreads();
    for (int j = 0; j < 2; ++j) {
        const int b = t + j * 1024;
        const unsigned long long above = b + 1 < 2048 ? s_cnt[b + 1] : 0ull;
        if (s_cnt[b] >= k_rem && above < k_rem) {
            const unsigned long long rem = k_rem - above;
            const unsigned int prefix = ws->prefix | (static_cast<unsigned int>(b) << (level == 0 ? 20 : level == 1 ? 9 : 0));
            ws->prefix = prefix;
            ws->k_rem = rem;
            if (level == 2) {  // v_k is exact now; the loss follows after ohem_sum_above_kernel (ohem_finish_kernel)
                const float vk = __uint_as_float(prefix);
                const unsigned long long n_eq = s_cnt[b] - above;
                ws->sel_thresh = vk;
                ws->tie_value = vk;
                ws->tie_frac = static_cast<float>(static_cast<double>(rem) / static_cast<double>(n_eq));
                ws->inv_m = static_cast<float>(1.0 / static_cast<double>(ws->k));
            }
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(256)
ohem_ce_bwd_kernel(const T* __restrict__ logits, const void* __restrict__ labels, int label_dtype, int C, long long HW,
                   const float* __restrict__ weight, const float* __restrict__ loss_px, const OhemWs* __restrict__ ws,
                   const float* __restrict__ grad_out, T* __restrict__ grad_logits) {
    const int n = blockIdx.y;
    const float sel = ws->sel_thresh, tie_v = ws->tie_value, tie_f = ws->tie_frac;
    const float g = ws->n_nonfinite ? __int_as_float(0x7fc00000) : __ldg(grad_out) * ws->inv_m;  // NaN loss -> NaN gradients
    const T* base = logits + static_cast<long long>(n) * C * HW;
    T* gbase = grad_logits + static_cast<long long>(n) * C * HW;
    const bool vec = (HW & 7) == 0 && (reinterpret_cast<uintptr_t>(logits) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(grad_logits) & 15) == 0 && (reinterpret_cast<uintptr_t>(loss_px) & 15) == 0;
    const long long HWv = vec ? HW / 4 : 0;
    for (long long q = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; q < HWv;
         q += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long i = q * 4, o = static_cast<long long>(n) * HW + i;
        const float4 l4 = __ldg(reinterpret_cast<const float4*>(loss_px + o));
        const float l[4] = {l4.x, l4.y, l4.z, l4.w};
        float k[4];
        long long lb[4];
        bool any = false;
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            float coef = 0.f;
            if (l[p] >= 0.f) coef = l[p] > sel ? 1.f : (l[p] == tie_v ? tie_f : 0.f);
            lb[p] = -1;
            k[p] = 0.f;
            if (coef != 0.f) {
                lb[p] = ld_label(labels, label_dtype, o + p);
                k[p] = g * coef * (weight ? __ldg(weight + lb[p]) : 1.f);
                any = true;
            }
        }
        if (!any) {  // nothing selected among the 4 pixels: zero the gradient without reading the logits
            const float z[4] = {0.f, 0.f, 0.f, 0.f};
            for (int c = 0; c < C; ++c) st_grad4<T>(gbase + c * HW + i, z);
            continue;
        }
        float m[4], s[4];
        softmax_stats4<T>(base + i, C, HW, m, s);
#pragma unroll
        for (int p = 0; p < 4; ++p) s[p] = 1.f / s[p];
        for (int c = 0; c < C; ++c) {
            float v[4], r[4];
            ld_logit4<T>(base + c * HW + i, v);
#pragma unroll
            for (int p = 0; p < 4; ++p) r[p] = k[p] * (expf(v[p] - m[p]) * s[p] - (c == lb[p] ? 1.f : 0.f));
            st_grad4<T>(gbase + c * HW + i, r);
        }
    }
    for (long long i = (vec ? HW : 0) + static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < HW;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long o = static_cast<long long>(n) * HW + i;
        const float l = __ldg(loss_px + o);
        float coef = 0.f;
        if (l >= 0.f) coef = l > sel ? 1.f : (l == tie_v ? tie_f : 0.f);
        if (coef == 0.f) {  // not selected (or ignored): the gradient plane entries are zero
            for (int c = 0; c < C; ++c) gbase[c * HW + i] = from_f32<T>(0.f);
            continue;
        }
        const long long lb = ld_label(labels, label_dtype, o);
        float m, s;
        pixel_ce<T>(base + i, C, HW, lb, weight, &m, &s);
        const float w = weight ? __ldg(weight + lb) : 1.f;
        const float k = g * coef * w, inv_s = 1.f / s;
        for (int c = 0; c < C; ++c) {
            const float p = expf(ld_logit<T>(base + c * HW + i) - m) * inv_s;
            gbase[c * HW + i] = from_f32<T>(k * (p - (c == lb ? 1.f : 0.f)));
        }
    }
}

}  // namespace

extern "C" long long cabinet_ohem_workspace_bytes(void) { return static_cast<long long>(sizeof(OhemWs)); }

extern "C" int cabinet_ohem_ce_forward(const void* logits, int dtype, const void* labels, int label_dtype, int N, int C,
                                       long long HW, const float* weight, int ignore_label, float thresh,
                                       long long n_min, float* loss_px, void* workspace, float* loss_out,
                                       cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("ohem_ce_forward", dtype, CAB_DT_F32 | CAB_DT_BF16);
    CAB_REQUIRE(logits && labels && loss_px && workspace && loss_out && C > 0 && HW > 0 && N >= 0 && N <= 65535 &&
                    n_min >= 1,
                "ohem_ce_forward: bad arguments");
    CAB_REQUIRE((reinterpret_cast<uintptr_t>(workspace) & 7) == 0, "ohem_ce_forward: workspace must be 8-byte aligned");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    OhemWs* ws = reinterpret_cast<OhemWs*>(workspace);
    CAB_CUDA(cudaMemsetAsync(ws, 0, sizeof(OhemWs), s));
    if (N > 0) {
        dim3 grid(static_cast<unsigned>(std::min<long long>(cab_ceil_div(HW, 256 * 4), 148 * 8 / std::min(N, 8) + 1)), N);
        if (dtype == CABINET_F32)
            ohem_ce_px_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(logits), labels, label_dtype, C,
                                                          HW, weight, ignore_label, thresh, loss_px, ws);
        else
            ohem_ce_px_kernel<bf16><<<grid, 256, 0, s>>>(reinterpret_cast<const bf16*>(logits), labels, label_dtype, C, HW,
                                                         weight, ignore_label, thresh, loss_px, ws);
        CAB_LAUNCH_CHECK();
    }
    const long long total = static_cast<long long>(N) * HW;
    const unsigned hgrid = static_cast<unsigned>(std::max<long long>(1, std::min<long long>(cab_ceil_div(total, 256 * 8), 148 * 4)));
    ohem_pick_kernel<<<1, 1024, 0, s>>>(0, thresh, n_min, ws, loss_out);
    ohem_hist_kernel<<<hgrid, 256, 0, s>>>(loss_px, total, 1, ws);
    ohem_pick_kernel<<<1, 1024, 0, s>>>(1, thresh, n_min, ws, loss_out);
    ohem_hist_kernel<<<hgrid, 256, 0, s>>>(loss_px, total, 2, ws);
    ohem_pick_kernel<<<1, 1024, 0, s>>>(2, thresh, n_min, ws, loss_out);
    ohem_sum_above_kernel<<<hgrid, 256, 0, s>>>(loss_px, total, ws);
    ohem_finish_kernel<<<1, 1, 0, s>>>(ws, loss_out);
    ohem_nonfinite_kernel<<<1, 1, 0, s>>>(ws, loss_out);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_ohem_ce_backward(const void* logits, int dtype, const void* labels, int label_dtype, int N, int C,
                                        long long HW, const float* weight, const float* loss_px, const void* workspace,
                                        const float* grad_out, void* grad_logits, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("ohem_ce_backward", dtype, CAB_DT_F32 | CAB_DT_BF16);
    CAB_REQUIRE(logits && labels && loss_px && workspace && grad_out && grad_logits && C > 0 && HW > 0 && N >= 0 &&
                    N <= 65535,
                "ohem_ce_backward: bad arguments");
    if (N == 0) return CABINET_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const OhemWs* ws = reinterpret_cast<const OhemWs*>(workspace);
    dim3 grid(static_cast<unsigned>(std::min<long long>(cab_ceil_div(HW, 256 * 4), 148 * 16)), N);
    if (dtype == CABINET_F32)
        ohem_ce_bwd_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(logits), labels, label_dtype, C, HW,
                                                       weight, loss_px, ws, grad_out, reinterpret_cast<float*>(grad_logits));
    else
        ohem_ce_bwd_kernel<bf16><<<grid, 256, 0, s>>>(reinterpret_cast<const bf16*>(logits), labels, label_dtype, C, HW,
                                                      weight, loss_px, ws, grad_out, reinterpret_cast<bf16*>(grad_logits));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}
