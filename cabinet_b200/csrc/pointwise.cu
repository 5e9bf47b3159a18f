// Small fused elementwise / reduction kernels: SE & FFM gate MLP, scale(+act) apply, row softmax, CAB combine.
#include "common.cuh"

namespace {

// grid (N, splits): every block recomputes the (cheap) hidden layer of its image, then produces a 1/splits slice
// of the C gates.  Warp-per-output dot products so the weight rows are read coalesced.  fp32 throughout.
__global__ void __launch_bounds__(256)
gate_mlp_kernel(const float* __restrict__ gap_sum, float inv_hw, const float* __restrict__ w1,
                const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2,
                float* __restrict__ scale, int C, int Cmid, int gate) {
    extern __shared__ float sm[];  // mean[C] | hidden[Cmid]
    float* mean = sm;
    float* hidden = sm + C;
    const int n = blockIdx.x;
    for (int c = threadIdx.x; c < C; c += blockDim.x) mean[c] = gap_sum[static_cast<long long>(n) * C + c] * inv_hw;
    __syncthreads();
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32, nwarps = blockDim.x / 32;
    for (int j = warp; j < Cmid; j += nwarps) {
        float acc = 0.f;
        for (int c = lane; c < C; c += 32) acc = fmaf(__ldg(w1 + static_cast<long long>(j) * C + c), mean[c], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) hidden[j] = fmaxf(acc + (b1 ? b1[j] : 0.f), 0.f);
    }
    __syncthreads();
    const int per = (C + gridDim.y - 1) / gridDim.y;
    const int c_begin = blockIdx.y * per, c_end = min(C, c_begin + per);
    for (int c = c_begin + warp; c < c_end; c += nwarps) {
        float acc = 0.f;
        for (int j = lane; j < Cmid; j += 32) acc = fmaf(__ldg(w2 + static_cast<long long>(c) * Cmid + j), hidden[j], acc);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) scale[static_cast<long long>(n) * C + c] = cab_act(acc + (b2 ? b2[c] : 0.f), gate);
    }
}

// Batched tiny fully-connected layer for ALL images: grid = (ceil(J / 8), ceil(N / FC_NB)), block = 256.
constexpr int FC_NB = 8;      // images per block (blockIdx.y walks the batch)
constexpr int FC_WMAX = 32;   // weights per lane kept in registers: rows of up to 32 * 32 = 1024 inputs

// out[n][j] = act(b[j] + sum_c W[j][c] * in[n][c] * in_scale): warp = one output j for FC_NB images.  The whole
// weight row of the warp is fetched into registers up front (all loads in flight at once, issued before the input
// staging barrier), so a launch pays ONE global round trip instead of one per 32 inputs.
__global__ void __launch_bounds__(256)
gate_fc_kernel(const float* __restrict__ in, float in_scale, const float* __restrict__ W, const float* __restrict__ b,
               float* __restrict__ out, int N, int C, int J, int act, int in_fixed) {
    extern __shared__ float s_in[];  // [FC_NB][C]
    const int warp = threadIdx.x / 32, lane = threadIdx.x % 32;
    const int j = blockIdx.x * 8 + warp;
    const int n0 = blockIdx.y * FC_NB;
    const int nb = min(FC_NB, N - n0);
    float w[FC_WMAX];
    if (j < J) {
        const float* wr = W + static_cast<long long>(j) * C + lane;
#pragma unroll
        for (int i = 0; i < FC_WMAX; ++i) w[i] = (lane + 32 * i < C) ? __ldg(wr + 32 * i) : 0.f;
    }
    // stage the inputs of this block's images: rows are contiguous, so it is one flat copy; all loads of a thread are
    // issued before the first store (C <= 1024, FC_NB = 8: at most 8 float4 per thread)
    const float* src = in + static_cast<long long>(n0) * C;
    const int total = nb * C;
    if (in_fixed) {
        // in = [N][C] 64-bit fixed-point sums (2^-24): the deterministic SE pooling sums of the depthwise kernels
        // (int64 -> fp32 with ONE rounding, then an exact power-of-two scale: no double-precision arithmetic)
        const longlong2* fx = reinterpret_cast<const longlong2*>(reinterpret_cast<const long long*>(in) + static_cast<long long>(n0) * C);
        const float sc = in_scale * (1.0f / CABINET_GAP_FIXED_ONE);
        if ((C & 1) == 0) {  // 16-byte loads, all of a thread's loads in flight before the first use
            longlong2 v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int i = threadIdx.x + u * 256;
                if (2 * i < total) v[u] = __ldg(fx + i);
            }
#pragma unroll
            for (int u = 0; u < 16; ++u) {
                const int i = threadIdx.x + u * 256;
                if (2 * i < total) *reinterpret_cast<float2*>(s_in + 2 * i) = make_float2(__ll2float_rn(v[u].x) * sc, __ll2float_rn(v[u].y) * sc);
            }
        } else {
            const long long* f1 = reinterpret_cast<const long long*>(fx);
            for (int i = threadIdx.x; i < total; i += blockDim.x) s_in[i] = __ll2float_rn(__ldg(f1 + i)) * sc;
        }
    } else if ((C & 3) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = (threadIdx.x + u * 256) * 4;
            if (i < total) v[u] = __ldg(reinterpret_cast<const float4*>(src + i));
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int i = (threadIdx.x + u * 256) * 4;
            if (i < total)
                *reinterpret_cast<float4*>(s_in + i) =
                    make_float4(v[u].x * in_scale, v[u].y * in_scale, v[u].z * in_scale, v[u].w * in_scale);
        }
    } else {
        for (int i = threadIdx.x; i < total; i += blockDim.x) s_in[i] = src[i] * in_scale;
    }
    __syncthreads();
    if (j >= J) return;
    float acc[FC_NB];
#pragma unroll
    for (int k = 0; k < FC_NB; ++k) acc[k] = 0.f;
#pragma unroll
    for (int i = 0; i < FC_WMAX; ++i) {
        const int c = lane + 32 * i;
        if (c < C) {
#pragma unroll
            for (int k = 0; k < FC_NB; ++k)
                if (k < nb) acc[k] = fmaf(w[i], s_in[k * C + c], acc[k]);
        }
    }
#pragma unroll
    for (int k = 0; k < FC_NB; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
    if (lane == 0) {
        const float bj = b ? b[j] : 0.f;
        float v[FC_NB];
#pragma unroll
        for (int k = 0; k < FC_NB; ++k) v[k] = acc[k] + bj;
        cab_act_vec<FC_NB>(v, act);
#pragma unroll
        for (int k = 0; k < FC_NB; ++k)
            if (k < nb) out[static_cast<long long>(n0 + k) * J + j] = v[k];
    }
}

// grid (pixel chunks, N); blockDim = (CG channel-vector lanes) x (pixel lanes): a thread keeps its 16-byte channel
// vector's scales in registers and walks pixels with pure 32-bit strided addressing (no div/mod in the loop).
template <typename T>
__global__ void __launch_bounds__(256)
scale_act_kernel(T* __restrict__ x, long long ldx, const float* __restrict__ scale, int HW, int C, int act,
                 int plus_one, int pix_per_block) {
    constexpr int V = Vec16<T>::N;
    // (walking the tensor back to front, as channel_sum does, measured 10-15 % SLOWER here: these tensors fit L2 whole)
    const int n = blockIdx.y;
    const int bx = blockIdx.x;
    const int CG = C / V;
    const int lanes = blockDim.x / CG;  // pixel lanes (CG <= 256 / 2 checked by the host)
    const int cg = threadIdx.x % CG, pl = threadIdx.x / CG;
    if (pl >= lanes) return;
    float sc[V];
#pragma unroll
    for (int i = 0; i < V; ++i) sc[i] = __ldg(scale + static_cast<long long>(n) * C + cg * V + i);
    const int p0 = bx * pix_per_block;
    const int p1 = min(p0 + pix_per_block, HW);
    T* base = x + (static_cast<long long>(n) * HW) * ldx + cg * V;
    for (int p = p0 + pl; p < p1; p += lanes) {
        T* ptr = base + static_cast<long long>(p) * ldx;
        Vec16<T> v;
        v.load(ptr);
        float f[V];
        v.unpack(f);
        if (plus_one) {
#pragma unroll
            for (int i = 0; i < V; ++i) f[i] = fmaf(f[i], sc[i], f[i]);
        } else {
#pragma unroll
            for (int i = 0; i < V; ++i) f[i] *= sc[i];
            cab_act_vec<V>(f, act);
        }
        v.pack(f);
        v.store(ptr);
    }
}

// One warp per row; cols arbitrary.  exp in fp32 with max subtraction (F.softmax semantics).
template <typename T>
__global__ void __launch_bounds__(256)
softmax_rows_kernel(const float* __restrict__ s, T* __restrict__ p, long long rows, int cols) {
    const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x % 32;
    if (row >= rows) return;
    const float* in = s + row * cols;
    float m = -INFINITY;
    for (int c = lane; c < cols; c += 32) m = fmaxf(m, in[c]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float sum = 0.f;
    for (int c = lane; c < cols; c += 32) sum += expf(in[c] - m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.f / sum;
    T* out = p + row * cols;
    for (int c = lane; c < cols; c += 32) out[c] = from_f32<T>(expf(in[c] - m) * inv);
}

template <typename T>
__global__ void __launch_bounds__(256)
cab_combine_kernel(const T* __restrict__ g, const T* __restrict__ x, const T* __restrict__ r, T* __restrict__ out,
                   long long ldo, int CG, const float* __restrict__ gamma, long long nvec) {
    constexpr int V = Vec16<T>::N;
    const float gm = __ldg(gamma);
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        Vec16<T> gv, xv, rv, ov;
        gv.load(g + i * V);
        xv.load(x + i * V);
        rv.load(r + i * V);
        float gf[V], xf[V], rf[V], of[V];
        gv.unpack(gf);
        xv.unpack(xf);
        rv.unpack(rf);
#pragma unroll
        for (int k = 0; k < V; ++k) of[k] = gm * gf[k] + (xf[k] + xf[k] * (1.f / (1.f + __expf(-rf[k]))));
        ov.pack(of);
        ov.store(out + (i / CG) * ldo + (i % CG) * V);
    }
}

// Per-(image, channel) sum over pixels: grid (chunks, N); smem accumulation then one atomic per channel per block.
// Deterministic two-level sum: every block reduces its pixel range in a fixed order and writes partial[n][b][c]; the
// block that arrives last (per-image ticket) adds the partials in block order -> out[n][c].  No floating-point atomics:
// the FFM gate (and the per-image head weights derived from it) is bit-reproducible from run to run.
template <typename T>
__global__ void __launch_bounds__(256)
channel_sum_kernel(const T* __restrict__ x, long long ldx, long long HW, int C, float* __restrict__ out,
                   long long pix_per_block, float* __restrict__ partial, unsigned int* __restrict__ tickets) {
    constexpr int V = Vec16<T>::N;
    extern __shared__ float s_red[];  // [rows][C]
    __shared__ bool s_last;
    // blocks are dispatched in (x, y) order: map them back to front, so the kernel starts on the part of the 134 MB
    // tensor its producer wrote last (still L2 resident) instead of evicting it while streaming the evicted head
    const int n = static_cast<int>(gridDim.y - 1 - blockIdx.y), nb = gridDim.x;
    const int bxr = static_cast<int>(gridDim.x - 1 - blockIdx.x);
    const int CG = C / V;
    const long long p0 = bxr * pix_per_block;
    const long long p1 = min(p0 + pix_per_block, HW);
    const int rows = blockDim.x / CG;  // pixels processed per sweep (CG <= blockDim.x is checked by the host)
    const int cg = threadIdx.x % CG, pr = threadIdx.x / CG;
    if (pr < rows) {
        float acc[V];
#pragma unroll
        for (int i = 0; i < V; ++i) acc[i] = 0.f;
        const T* base = x + static_cast<long long>(n) * HW * ldx + cg * V;
        // 32-bit pixel / element offsets inside one image (the host checks HW * ldx < 2^31)
        const unsigned q1 = static_cast<unsigned>(p1), step = static_cast<unsigned>(rows), ld = static_cast<unsigned>(ldx);
        for (unsigned pb = static_cast<unsigned>(p0) + pr; pb < q1; pb += 4u * step) {  // four 16-byte loads in flight
            Vec16<T> v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (pb + u * step < q1) v[u].load(base + (pb + u * step) * ld);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                if (pb + u * step < q1) {
                    float f[V];
                    v[u].unpack(f);
#pragma unroll
                    for (int i = 0; i < V; ++i) acc[i] += f[i];
                }
            }
        }
#pragma unroll
        for (int i = 0; i < V; ++i) s_red[pr * C + cg * V + i] = acc[i];
    }
    __syncthreads();
    float* mine = partial + (static_cast<long long>(n) * nb + bxr) * C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float sum = 0.f;
        for (int r = 0; r < rows; ++r) sum += s_red[r * C + c];
        mine[c] = sum;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&tickets[n], 1u) == static_cast<unsigned>(nb - 1);
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    const float* all = partial + static_cast<long long>(n) * nb * C;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float sum = 0.f;
        for (int b = 0; b < nb; ++b) sum += __ldcg(all + static_cast<long long>(b) * C + c);
        out[static_cast<long long>(n) * C + c] = sum;
    }
    if (threadIdx.x == 0) tickets[n] = 0;  // ready for the next launch
}

}  // namespace

extern "C" int cabinet_channel_sum(const void* x, long long ldx, int dtype, int N, long long HW, int C, float* out,
                                   float* scratch, long long scratch_bytes, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("channel_sum", dtype, CAB_DT_ALL);
    CAB_REQUIRE(x && out && scratch, "channel_sum: null pointer");
    const int V = dtype == CABINET_F32 ? 4 : 8;
    CAB_REQUIRE(C > 0 && C % V == 0 && ldx % V == 0 && ldx >= C && C / V <= 256 && N <= 65535 && HW * ldx < (1LL << 31),
                "channel_sum: unsupported C=%d ldx=%lld", C, ldx);
    if (N == 0 || HW == 0) return CABINET_OK;
    // >= 256 pixels per block and at most 64 blocks per image (the last block of an image adds their partial sums)
    const long long pix_per_block = std::max<long long>(256, cab_ceil_div(HW, 64));
    const int nb = static_cast<int>(cab_ceil_div(HW, pix_per_block));
    const int rows = 256 / (C / V);
    const size_t smem = static_cast<size_t>(rows) * C * sizeof(float);
    CAB_REQUIRE(smem <= 48 * 1024, "channel_sum: C too large");
    // scratch layout: [N] tickets (uint32, must be zero before the first launch; the kernel leaves them zero), then the
    // partial sums [N][nb][C] fp32 at the next 256-byte boundary
    const size_t off = (static_cast<size_t>(N) * sizeof(unsigned int) + 255) & ~size_t(255);
    const size_t need = off + static_cast<size_t>(N) * nb * C * sizeof(float);
    CAB_REQUIRE(static_cast<size_t>(scratch_bytes) >= need, "channel_sum: scratch needs %zu bytes", need);
    unsigned int* tickets = reinterpret_cast<unsigned int*>(scratch);
    float* partial = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(scratch) + off);
    dim3 grid(nb, N);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CAB_DISPATCH_DT(dtype, T,
                    channel_sum_kernel<T><<<grid, 256, smem, s>>>(reinterpret_cast<const T*>(x), ldx, HW, C, out, pix_per_block,
                                                                  partial, tickets));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_gate_mlp(const float* gap_sum, float inv_hw, const float* w1, const float* b1,
                                const float* w2, const float* b2, float* scale, int N, int C, int Cmid, int gate,
                                cabinet_stream_t stream) {
    CAB_REQUIRE(gap_sum && w1 && w2 && scale, "gate_mlp: null pointer");
    CAB_REQUIRE(C > 0 && Cmid > 0 && (C + Cmid) * sizeof(float) <= 48 * 1024, "gate_mlp: C=%d Cmid=%d unsupported", C,
                Cmid);
    if (N == 0) return CABINET_OK;
    const int splits = std::max(1, std::min(16, C / 32));
    gate_mlp_kernel<<<dim3(N, splits), 256, (C + Cmid) * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
        gap_sum, inv_hw, w1, b1, w2, b2, scale, C, Cmid, gate);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_gate_fc(const float* in, float in_scale, const float* W, const float* b, float* out, int N,
                               int C, int J, int act, int in_fixed, cabinet_stream_t stream) {
    CAB_REQUIRE(in && W && out && C > 0 && J > 0 && C <= 32 * FC_WMAX, "gate_fc: bad arguments (C=%d J=%d, C <= 1024)", C, J);
    if (N == 0) return CABINET_OK;
    CAB_REQUIRE((N + FC_NB - 1) / FC_NB <= 65535, "gate_fc: N exceeds grid limits");
    gate_fc_kernel<<<dim3((J + 7) / 8, (N + FC_NB - 1) / FC_NB), 256, FC_NB * C * sizeof(float),
                     static_cast<cudaStream_t>(stream)>>>(
        in, in_scale, W, b, out, N, C, J, act, in_fixed);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_scale_act(void* x, long long ldx, int dtype, const float* scale, int N, long long HW, int C,
                                 int act, int plus_one, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("scale_act", dtype, CAB_DT_F32 | CAB_DT_BF16);
    CAB_REQUIRE(x && scale, "scale_act: null pointer");
    const int V = dtype == CABINET_F32 ? 4 : 8;
    CAB_REQUIRE(C > 0 && C % V == 0 && ldx % V == 0 && ldx >= C && C / V <= 256 && HW < (1LL << 31) && N <= 65535,
                "scale_act: C/ldx must be multiples of %d, C/%d <= 256", V, V);
    if (N == 0 || HW == 0) return CABINET_OK;
    const int CG = C / V;
    const int threads = std::max(CG, 256 / CG * CG);   // a multiple of CG close to 256
    const int lanes = threads / CG;
    // ~8 pixels per thread, but at least ~4 blocks per SM across the batch
    int pix_per_block = lanes * 8;
    const long long want_blocks = 148LL * 8;
    while (pix_per_block > lanes && cab_ceil_div(HW, pix_per_block) * N < want_blocks) pix_per_block -= lanes;
    dim3 grid(static_cast<unsigned>(cab_ceil_div(HW, pix_per_block)), N);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (dtype == CABINET_BF16)
        scale_act_kernel<bf16><<<grid, threads, 0, s>>>(reinterpret_cast<bf16*>(x), ldx, scale, static_cast<int>(HW), C, act,
                                                        plus_one, pix_per_block);
    else
        scale_act_kernel<float><<<grid, threads, 0, s>>>(reinterpret_cast<float*>(x), ldx, scale, static_cast<int>(HW), C, act,
                                                         plus_one, pix_per_block);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

namespace {
// out[n][r][k] = bf16(w[r][k] * (scale[n][k % cin_pad] + plus)) for k % cin_pad < Cin, 0 otherwise (the K padding)
__global__ void __launch_bounds__(256)
scale_weights_kernel(const bf16* __restrict__ w, const float* __restrict__ scale, bf16* __restrict__ out, unsigned per_image,
                     unsigned cin_pad, int Cin, float plus) {
    const unsigned i = (blockIdx.x * 256u + threadIdx.x) * 8u;  // 32-bit index math (a 64-bit modulo costs ~100 instructions)
    if (i >= per_image) return;
    const int n = blockIdx.y;
    const int ci = static_cast<int>(i % cin_pad);  // 8 consecutive k share the tap (cin_pad % 8 == 0)
    Vec16<bf16> v;
    v.load(w + i);
    float f[8];
    v.unpack(f);
    const float* sc = scale + static_cast<long long>(n) * Cin + ci;
    if (ci + 8 <= Cin) {
        const float4 s0 = __ldg(reinterpret_cast<const float4*>(sc)), s1 = __ldg(reinterpret_cast<const float4*>(sc) + 1);
        f[0] *= s0.x + plus; f[1] *= s0.y + plus; f[2] *= s0.z + plus; f[3] *= s0.w + plus;
        f[4] *= s1.x + plus; f[5] *= s1.y + plus; f[6] *= s1.z + plus; f[7] *= s1.w + plus;
    } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = (ci + j < Cin) ? f[j] * (sc[j] + plus) : 0.f;
    }
    v.pack(f);
    v.store(out + static_cast<size_t>(n) * per_image + i);
}
}  // namespace

namespace {
// Gate MLP + per-image weight scaling in ONE launch (the squeeze-excite gate of a ReLU block folded into its project conv,
// the FFM attention folded into the head conv): every block recomputes the (tiny) two-layer gate of its image in shared
// memory -- C x J multiply-adds, a few microseconds hidden behind the other blocks -- then scales its slice of the weights:
//   out[n][r][k] = bf16(w[r][k] * (gate[n][k % cin_pad] + plus)),  gate = act(W2 relu(W1 mean + b1) + b2)
// Replaces gate_fc -> gate_fc -> scale_weights (three dependent launches on the critical path).
constexpr int GSW_ELEMS = 65536;  // weight elements per block (each block re-reads the gate weights: keep the grid small)

// out[o] = act(b[o] + sum_i W[o][i] * in[i]) + plus for one block of 256 threads, inputs / outputs in shared memory.
// 256 / O threads share an output (interleaved i, so a group reads consecutive weights), every thread's loads are
// independent of each other (all in flight at once: the layer costs about one L2 round trip); the group's partial sums are
// added in a fixed order.  Ends with a barrier.
__device__ __forceinline__ void fc_block(const float* __restrict__ W, const float* __restrict__ b, const float* in, float* out,
                                         float* red, int O, int I, int act, float plus) {
    int parts = 1;
    while (parts * 2 * O <= 256 && parts * 2 <= 32) parts *= 2;
    for (int o0 = 0; o0 < O; o0 += 256 / parts) {
        const int o = o0 + threadIdx.x / parts, part = threadIdx.x % parts;
        float acc = 0.f;
        if (o < O) {
            const float* wr = W + static_cast<long long>(o) * I;
#pragma unroll 8
            for (int i = part; i < I; i += parts) acc = fmaf(__ldg(wr + i), in[i], acc);
        }
        red[threadIdx.x] = acc;
        __syncthreads();
        if (o < O && part == 0) {
            float sum = 0.f;
            for (int k = 0; k < parts; ++k) sum += red[threadIdx.x + k];
            out[o] = cab_act(sum + (b ? b[o] : 0.f), act) + plus;
        }
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256)
gate_scale_weights_kernel(const void* __restrict__ gap, int in_fixed, float inv_hw, const float* __restrict__ w1,
                          const float* __restrict__ b1, const float* __restrict__ w2, const float* __restrict__ b2, int gate,
                          int C, int J, const bf16* __restrict__ w, bf16* __restrict__ out, unsigned per_image, unsigned cin_pad,
                          float plus) {
    extern __shared__ float sm[];  // mean[C] | hidden[J] | gate[C] | red[256]
    float* mean = sm;
    float* hidden = sm + C;
    float* g = hidden + J;
    float* red = g + C;
    const int n = blockIdx.y;
    if (in_fixed) {
        const long long* fx = reinterpret_cast<const long long*>(gap) + static_cast<long long>(n) * C;
        for (int c = threadIdx.x; c < C; c += 256) mean[c] = __ll2float_rn(__ldg(fx + c)) * (inv_hw * (1.0f / CABINET_GAP_FIXED_ONE));
    } else {
        const float* fp = reinterpret_cast<const float*>(gap) + static_cast<long long>(n) * C;
        for (int c = threadIdx.x; c < C; c += 256) mean[c] = __ldg(fp + c) * inv_hw;
    }
    __syncthreads();
    fc_block(w1, b1, mean, hidden, red, J, C, CABINET_ACT_RELU, 0.f);
    fc_block(w2, b2, hidden, g, red, C, J, gate, plus);
    const unsigned base = blockIdx.x * GSW_ELEMS;
    for (unsigned i = base + threadIdx.x * 8u; i < min(base + GSW_ELEMS, per_image); i += 256u * 8u) {
        const int ci = static_cast<int>(i % cin_pad);
        Vec16<bf16> v;
        v.load(w + i);
        float f[8];
        v.unpack(f);
#pragma unroll
        for (int k = 0; k < 8; ++k) f[k] = (ci + k < C) ? f[k] * g[ci + k] : 0.f;
        v.pack(f);
        v.store(out + static_cast<size_t>(n) * per_image + i);
    }
}
}  // namespace

extern "C" int cabinet_gate_scale_weights(const void* gap_sum, int in_fixed, float inv_hw, const float* w1, const float* b1,
                                          const float* w2, const float* b2, int gate, int C, int Cmid, const void* w_packed,
                                          void* out, int N, int rows, int taps, int cin_pad, int plus_one,
                                          cabinet_stream_t stream) {
    CAB_REQUIRE(gap_sum && w1 && w2 && w_packed && out && C > 0 && Cmid > 0 && rows > 0 && taps > 0 && cin_pad % 8 == 0 &&
                    C <= cin_pad && C <= 1024 && Cmid <= 1024 && N <= 65535,
                "gate_scale_weights: bad arguments");
    CAB_REQUIRE((reinterpret_cast<uintptr_t>(w_packed) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                "gate_scale_weights: alignment");
    if (N == 0) return CABINET_OK;
    const long long per_image = static_cast<long long>(rows) * taps * cin_pad;
    CAB_REQUIRE(per_image < (1LL << 31), "gate_scale_weights: weight matrix too large");
    dim3 grid(static_cast<unsigned>(cab_ceil_div(per_image, GSW_ELEMS)), N);
    gate_scale_weights_kernel<<<grid, 256, (2 * C + Cmid + 256) * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
        gap_sum, in_fixed, inv_hw, w1, b1, w2, b2, gate, C, Cmid, reinterpret_cast<const bf16*>(w_packed),
        reinterpret_cast<bf16*>(out), static_cast<unsigned>(per_image), static_cast<unsigned>(cin_pad), plus_one ? 1.f : 0.f);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_scale_weights(const void* w_packed, const float* scale, void* out, int N, int rows, int taps,
                                     int cin_pad, int Cin, int plus_one, cabinet_stream_t stream) {
    CAB_REQUIRE(w_packed && scale && out && rows > 0 && taps > 0 && cin_pad > 0 && cin_pad % 8 == 0 && Cin > 0 && Cin <= cin_pad,
                "scale_weights: bad arguments");
    CAB_REQUIRE((reinterpret_cast<uintptr_t>(w_packed) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && N <= 65535,
                "scale_weights: alignment / batch");
    if (N == 0) return CABINET_OK;
    const long long per_image = static_cast<long long>(rows) * taps * cin_pad;
    CAB_REQUIRE(per_image < (1LL << 31), "scale_weights: weight matrix too large");
    CAB_REQUIRE(Cin % 4 == 0 && (reinterpret_cast<uintptr_t>(scale) & 15) == 0, "scale_weights: Cin %% 4 and a 16-byte aligned scale");
    dim3 grid(static_cast<unsigned>(cab_ceil_div(per_image / 8, 256)), N);
    scale_weights_kernel<<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        reinterpret_cast<const bf16*>(w_packed), scale, reinterpret_cast<bf16*>(out), static_cast<unsigned>(per_image),
        static_cast<unsigned>(cin_pad), Cin, plus_one ? 1.f : 0.f);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_softmax_rows(const float* s, void* p, int p_dtype, long long rows, int cols,
                                    cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("softmax_rows", p_dtype, CAB_DT_F32 | CAB_DT_BF16);
    CAB_REQUIRE(s && p && cols > 0, "softmax_rows: bad arguments");
    if (rows == 0) return CABINET_OK;
    dim3 grid(static_cast<unsigned>(cab_ceil_div(rows, 8)));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (p_dtype == CABINET_BF16)
        softmax_rows_kernel<bf16><<<grid, 256, 0, st>>>(s, reinterpret_cast<bf16*>(p), rows, cols);
    else
        softmax_rows_kernel<float><<<grid, 256, 0, st>>>(s, reinterpret_cast<float*>(p), rows, cols);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_cab_combine(const void* g, const void* x, const void* r, void* out, long long ldo,
                                   const float* gamma, int dtype, long long n_pixels, int C,
                                   cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("cab_combine", dtype, CAB_DT_ALL);
    CAB_REQUIRE(g && x && r && out && gamma, "cab_combine: null pointer");
    const int V = dtype == CABINET_F32 ? 4 : 8;
    CAB_REQUIRE(C > 0 && C % V == 0 && ldo % V == 0 && ldo >= C, "cab_combine: C/ldo must be multiples of %d", V);
    if (n_pixels == 0) return CABINET_OK;
    const int CG = C / V;
    const long long nvec = n_pixels * CG;
    dim3 grid(static_cast<unsigned>(std::min<long long>(cab_ceil_div(nvec, 256), 148 * 16)));
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CAB_DISPATCH_DT(dtype, T,
                    cab_combine_kernel<T><<<grid, 256, 0, s>>>(reinterpret_cast<const T*>(g), reinterpret_cast<const T*>(x),
                                                               reinterpret_cast<const T*>(r), reinterpret_cast<T*>(out), ldo, CG,
                                                               gamma, nvec));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}
