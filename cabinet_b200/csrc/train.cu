// Training-step kernels (BASELINE config 5; reference: src/scripts/train.py:429-441 = autocast forward in .train() mode,
// two OHEM losses, backward).  Everything the inference path does not have:
//   * train-mode BatchNorm: batch statistics (shifted single pass, deterministic two-level sums), running-statistics
//     update (momentum 0.1, unbiased variance), normalise + activation, and its backward (two reductions + apply);
//   * eval-mode BatchNorm inside a training step (frozen BN): statistics from the running statistics, one-pass backward;
//   * data gradients and weight gradients of the dense and depthwise convolutions (CUDA-core implicit GEMM with
//     fp32 accumulation; split over the pixel dimension with a fixed-order second-level sum for the weight gradients);
//   * squeeze-excite / FFM gate backward, CAB combine backward, softmax backward, the adjoints of every bilinear
//     resize / adaptive average pool as ONE separable sparse resampling kernel, small helpers.
// All reductions have a fixed summation order (no floating-point atomics): a training step is bit-reproducible.
// Activations are NHWC (fp32, bf16 or fp16), statistics / gradients of parameters fp32.
#include <type_traits>

#include "tc_common.cuh"

namespace {

template <typename T> __device__ __forceinline__ float ldf(const T* p) { return to_f32<T>(*p); }

// derivative of the activation with respect to its input u
__device__ __forceinline__ float act_grad(float u, int act) {
    switch (act) {
        case CABINET_ACT_RELU: return u > 0.f ? 1.f : 0.f;
        case CABINET_ACT_HSWISH:  // d/du [u * relu6(u + 3) / 6]
            return u <= -3.f ? 0.f : (u >= 3.f ? 1.f : (2.f * u + 3.f) * (1.f / 6.f));
        case CABINET_ACT_HSIGMOID: return (u > -3.f && u < 3.f) ? (1.f / 6.f) : 0.f;
        case CABINET_ACT_SIGMOID: {
            const float s = 1.f / (1.f + __expf(-u));
            return s * (1.f - s);
        }
        default: return 1.f;
    }
}

// ... over a small register array: ONE uniform branch per call, straight-line code per case (a switch per element is an
// indirect branch per element: it made the BN backward passes instruction bound)
template <int N> __device__ __forceinline__ void act_grad_vec(const float* u, int act, float* d) {
    if (act == CABINET_ACT_RELU) {
#pragma unroll
        for (int i = 0; i < N; ++i) d[i] = u[i] > 0.f ? 1.f : 0.f;
    } else if (act == CABINET_ACT_HSWISH) {
#pragma unroll
        for (int i = 0; i < N; ++i) d[i] = u[i] <= -3.f ? 0.f : (u[i] >= 3.f ? 1.f : fmaf(u[i], 1.f / 3.f, 0.5f));
    } else if (act == CABINET_ACT_NONE) {
#pragma unroll
        for (int i = 0; i < N; ++i) d[i] = 1.f;
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) d[i] = act_grad(u[i], act);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Column reductions over the pixel dimension: out[q][c] = sum over rows m of f_q(m, c), q < NQ.
// Level 1: block b reduces rows [b * rows_per_block, ...) -> partial[b][q][c] (fixed order inside the block);
// level 2 (the *_finalize kernels) adds the blocks in index order.
constexpr int RED_THREADS = 256;

template <int NQ, typename F>
__device__ __forceinline__ void col_reduce_block(long long M, int C, long long rows_per_block, float* __restrict__ partial,
                                                 F f) {
    extern __shared__ float s_red[];  // [lanes][NQ][cw]
    const long long m0 = static_cast<long long>(blockIdx.x) * rows_per_block;
    const long long m1 = min(m0 + rows_per_block, M);
    for (int c0 = 0; c0 < C; c0 += RED_THREADS) {
        const int cw = min(RED_THREADS, C - c0);
        const int lanes = RED_THREADS / cw;          // pixel lanes working on this channel chunk
        const int cl = threadIdx.x % cw, lane = threadIdx.x / cw;
        float acc[NQ];
#pragma unroll
        for (int q = 0; q < NQ; ++q) acc[q] = 0.f;
        if (lane < lanes)
            for (long long m = m0 + lane; m < m1; m += lanes) f(m, c0 + cl, acc);
        __syncthreads();
        if (lane < lanes)
#pragma unroll
            for (int q = 0; q < NQ; ++q) s_red[(lane * NQ + q) * cw + cl] = acc[q];
        __syncthreads();
        if (threadIdx.x < cw) {
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                float sum = 0.f;
                for (int l = 0; l < lanes; ++l) sum += s_red[(l * NQ + q) * cw + threadIdx.x];
                partial[(static_cast<long long>(blockIdx.x) * NQ + q) * C + c0 + threadIdx.x] = sum;
            }
        }
    }
}

// 16-byte vector accessors (8 bf16 / 4 fp32 per access)
template <typename T> __device__ __forceinline__ void ldv(const T* p, float* f) {
    Vec16<T> v;
    v.load(p);
    v.unpack(f);
}
template <typename T> __device__ __forceinline__ void stv(T* p, const float* f) {
    Vec16<T> v;
    v.pack(f);
    v.store(p);
}
template <typename T> __host__ __device__ constexpr int vec_n() { return sizeof(T) == 4 ? 4 : 8; }

// Vectorised form of col_reduce_block: a thread owns one 16-byte channel vector (V channels) of a pixel lane.
// f(m, c0, acc[NQ * V]) accumulates quantity q of channel c0 + v into acc[q * V + v].  C % V == 0.
template <int NQ, int V, bool UNROLL2 = true, typename F>
__device__ __forceinline__ void col_reduce_block_v(long long M, int C, long long rows_per_block, float* __restrict__ partial,
                                                   F f) {
    extern __shared__ float s_red[];  // [lanes][NQ][cw]
    const long long m0 = static_cast<long long>(blockIdx.x) * rows_per_block;
    const long long m1 = min(m0 + rows_per_block, M);
    const int CV = C / V;
    for (int v0 = 0; v0 < CV; v0 += RED_THREADS) {
        const int cwv = min(RED_THREADS, CV - v0), cw = cwv * V;
        const int lanes = RED_THREADS / cwv;
        const int cv = threadIdx.x % cwv, lane = threadIdx.x / cwv;
        float acc[NQ * V];
#pragma unroll
        for (int q = 0; q < NQ * V; ++q) acc[q] = 0.f;
        if (!UNROLL2) {
            if (lane < lanes)
                for (long long m = m0 + lane; m < m1; m += lanes) f(m, (v0 + cv) * V, acc);
        } else if (lane < lanes) {
            // two independent accumulator sets / rows in flight per thread (fixed pairing: still deterministic)
            float acc2[NQ * V];
#pragma unroll
            for (int q = 0; q < NQ * V; ++q) acc2[q] = 0.f;
            long long m = m0 + lane;
            for (; m + lanes < m1; m += 2 * lanes) {
                f(m, (v0 + cv) * V, acc);
                f(m + lanes, (v0 + cv) * V, acc2);
            }
            if (m < m1) f(m, (v0 + cv) * V, acc);
#pragma unroll
            for (int q = 0; q < NQ * V; ++q) acc[q] += acc2[q];
        }
        __syncthreads();
        if (lane < lanes)
#pragma unroll
            for (int q = 0; q < NQ; ++q)
#pragma unroll
                for (int v = 0; v < V; ++v) s_red[(lane * NQ + q) * cw + cv * V + v] = acc[q * V + v];
        __syncthreads();
        for (int c = threadIdx.x; c < cw; c += RED_THREADS) {
#pragma unroll
            for (int q = 0; q < NQ; ++q) {
                float sum = 0.f;
                for (int l = 0; l < lanes; ++l) sum += s_red[(l * NQ + q) * cw + c];
                partial[(static_cast<long long>(blockIdx.x) * NQ + q) * C + v0 * V + c] = sum;
            }
        }
    }
}
template <typename T> constexpr size_t red_smem_v(int nq) { return static_cast<size_t>(RED_THREADS) * vec_n<T>() * nq * sizeof(float); }

inline int red_blocks(long long M, long long* rows_per_block) {
    // at most 8 blocks per SM: the reduction kernels hold 2 or 4 blocks of 256 threads per SM (121 / 64 registers), so
    // 1184 equal blocks are exactly 4 or 2 full waves (1024 left the last wave half empty)
    long long nb = std::min<long long>(148 * 8, std::max<long long>(1, M / 64));
    *rows_per_block = cab_ceil_div(M, nb);
    return static_cast<int>(cab_ceil_div(M, *rows_per_block));
}
constexpr size_t RED_SMEM = RED_THREADS * 3 * sizeof(float);

// ---- BN statistics: shifted sums (k = the value at row 0) keep E[(x-k)^2] - E[x-k]^2 well conditioned in fp32
template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
bn_stats_kernel(const T* __restrict__ x, long long ldx, long long M, int C, long long rpb, float* __restrict__ partial) {
    col_reduce_block<2>(M, C, rpb, partial, [&](long long m, int c, float* acc) {
        const float d = ldf(x + m * ldx + c) - ldf(x + c);
        acc[0] += d;
        acc[1] = fmaf(d, d, acc[1]);
    });
}

template <typename T>
__global__ void bn_finalize_kernel(const float* __restrict__ partial, int nb, long long M, int C, const T* __restrict__ x,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, float eps,
                                   float momentum, float* __restrict__ run_mean, float* __restrict__ run_var,
                                   float* __restrict__ stats /* [4][C]: mean, invstd, scale, shift */) {
    // one WARP per channel: lane l adds blocks l, l + 32, ... in order, then a fixed butterfly (deterministic)
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (c >= C) return;
    double s1 = 0.0, s2 = 0.0;
    for (int b = lane; b < nb; b += 32) {
        s1 += partial[(static_cast<long long>(b) * 2 + 0) * C + c];
        s2 += partial[(static_cast<long long>(b) * 2 + 1) * C + c];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane != 0) return;
    const double k = ldf(x + c), inv_m = 1.0 / static_cast<double>(M);
    const double d = s1 * inv_m;
    const double mean = k + d;
    const double var = fmax(s2 * inv_m - d * d, 0.0);  // biased (normalisation)
    const float invstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    const float g = gamma ? gamma[c] : 1.f, bt = beta ? beta[c] : 0.f;
    stats[c] = static_cast<float>(mean);
    stats[C + c] = invstd;
    stats[2 * C + c] = g * invstd;
    stats[3 * C + c] = bt - static_cast<float>(mean) * g * invstd;
    if (run_mean) {  // nn.BatchNorm2d: running = (1 - momentum) * running + momentum * batch (unbiased variance)
        const double unb = M > 1 ? var * static_cast<double>(M) / static_cast<double>(M - 1) : var;
        run_mean[c] = (1.f - momentum) * run_mean[c] + momentum * static_cast<float>(mean);
        run_var[c] = (1.f - momentum) * run_var[c] + momentum * static_cast<float>(unb);
    }
}

// y = act((z * scale[c] + shift[c]) * gate[n][c]) + res     (scale/shift/gate/res optional)
template <typename TZ, typename TY>
__global__ void __launch_bounds__(256)
affine_act_kernel(const TZ* __restrict__ z, long long ldz, const float* __restrict__ scale, const float* __restrict__ shift,
                  const float* __restrict__ gate, float gate_plus, const TY* __restrict__ res, long long ldres,
                  TY* __restrict__ y, long long ldy, long long M, long long HW, int C, int act) {
    const long long total = M * C;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long m = i / C;
        const int c = static_cast<int>(i - m * C);
        float u = ldf(z + m * ldz + c);
        if (scale) u = fmaf(u, scale[c], shift[c]);
        if (gate) u *= gate[(m / HW) * C + c] + gate_plus;
        u = cab_act(u, act);
        if (res) u += ldf(res + m * ldres + c);
        y[m * ldy + c] = from_f32<TY>(u);
    }
}

// ---- The same column reductions with the rows staged through shared memory by bulk copies (dense bf16 tensors only):
// a producer warp keeps RT_STAGES chunks of up to 16 KB per block in flight (cp.async.bulk + mbarrier ring), the 256
// consumer threads read their 16-byte channel vectors from shared memory.  The register-fed kernels above hold the
// bytes in flight in registers (two 16-byte loads per thread and source) and top out at 3.1-3.5 TB/s with 2-4 blocks
// per SM; here the in-flight bytes cost no registers.  Same per-block summation tree shape (pixel lanes -> shared
// memory -> fixed-order sum), so the result is deterministic; `nb` blocks write partial[b][q][c] as before.
constexpr int RT_STAGES = 4, RT_STAGE_BYTES = 16384, RT_THREADS = RED_THREADS + 32;

__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     tc::smem_u32(dst)),
                 "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(tc::smem_u32(bar))
                 : "memory");
}

// f(row0, row1, acc): row0 / row1 = this thread's 8 channels of one row of source 0 / 1 as fp32 (T = bf16 or f16)
template <int NQ, int NSRC, typename T, typename F>
__device__ __forceinline__ void col_reduce_tma(const T* __restrict__ src0, const T* __restrict__ src1, long long M, int C,
                                               long long rows_per_block, int chunk_rows, float* __restrict__ partial, F f) {
    constexpr int V = 8;
    extern __shared__ __align__(128) uint8_t s_ring[];  // [RT_STAGES][NSRC][chunk_rows * C] T; reused for the block sum
    __shared__ __align__(8) uint64_t full_bar[RT_STAGES], empty_bar[RT_STAGES];
    const int warp = threadIdx.x >> 5;
    const long long m0 = static_cast<long long>(blockIdx.x) * rows_per_block;
    const long long m1 = min(m0 + rows_per_block, M);
    const int n_chunks = static_cast<int>((m1 - m0 + chunk_rows - 1) / chunk_rows);
    const uint32_t src_bytes = static_cast<uint32_t>(chunk_rows) * C * 2;
    if (threadIdx.x == 0) {
        for (int i = 0; i < RT_STAGES; ++i) {
            tc::mbar_init(&full_bar[i], 1);
            tc::mbar_init(&empty_bar[i], RED_THREADS / 32);
        }
        tc::mbar_fence_init();
    }
    __syncthreads();
    float acc[NQ * V];
#pragma unroll
    for (int q = 0; q < NQ * V; ++q) acc[q] = 0.f;
    const int cwv = C / V, lanes = RED_THREADS / cwv;
    const int cv = threadIdx.x % cwv, lane = threadIdx.x / cwv;
    if (warp == RED_THREADS / 32) {
        // ---------------- producer
        if ((threadIdx.x & 31) == 0) {
            for (int i = 0; i < n_chunks; ++i) {
                const int st = i % RT_STAGES;
                if (i >= RT_STAGES) tc::mbar_wait(&empty_bar[st], ((i / RT_STAGES) - 1) & 1);
                const long long r0 = m0 + static_cast<long long>(i) * chunk_rows;
                const uint32_t bytes = static_cast<uint32_t>(min(static_cast<long long>(chunk_rows), m1 - r0)) * C * 2;
                uint8_t* dst = s_ring + static_cast<size_t>(st) * NSRC * src_bytes;
                tc::mbar_expect_tx(&full_bar[st], bytes * NSRC);
                bulk_load_1d(dst, src0 + r0 * C, bytes, &full_bar[st]);
                if (NSRC == 2) bulk_load_1d(dst + src_bytes, src1 + r0 * C, bytes, &full_bar[st]);
            }
        }
    } else {
        // ---------------- consumers
        for (int i = 0; i < n_chunks; ++i) {
            const int st = i % RT_STAGES;
            tc::mbar_wait(&full_bar[st], (i / RT_STAGES) & 1);
            const int rows = static_cast<int>(min(static_cast<long long>(chunk_rows), m1 - (m0 + static_cast<long long>(i) * chunk_rows)));
            const T* c0 = reinterpret_cast<const T*>(s_ring + static_cast<size_t>(st) * NSRC * src_bytes) + cv * V;
            const T* c1 = reinterpret_cast<const T*>(s_ring + static_cast<size_t>(st) * NSRC * src_bytes + src_bytes) + cv * V;
            if (lane < lanes) {
                for (int r = lane; r < rows; r += lanes) {
                    float a[V], b[V];
                    ldv(c0 + r * C, a);
                    if (NSRC == 2) ldv(c1 + r * C, b);
                    f(a, b, acc);
                }
            }
            __syncwarp();
            if ((threadIdx.x & 31) == 0) tc::mbar_arrive(&empty_bar[st]);
        }
    }
    __syncthreads();  // every chunk consumed: the ring is free for the block sum
    float* s_red = reinterpret_cast<float*>(s_ring);  // [lanes][NQ][C]
    if (warp < RED_THREADS / 32 && lane < lanes)
#pragma unroll
        for (int q = 0; q < NQ; ++q)
#pragma unroll
            for (int v = 0; v < V; ++v) s_red[(lane * NQ + q) * C + cv * V + v] = acc[q * V + v];
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += RT_THREADS) {
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
            float sum = 0.f;
            for (int l = 0; l < lanes; ++l) sum += s_red[(l * NQ + q) * C + c];
            partial[(static_cast<long long>(blockIdx.x) * NQ + q) * C + c] = sum;
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(RT_THREADS)
bn_stats_tma_kernel(const T* __restrict__ x, long long M, int C, long long rpb, int chunk_rows, float* __restrict__ partial) {
    float kv[8];  // the shift (row 0) of this thread's channel vector
    ldv(x + (threadIdx.x % (C / 8)) * 8, kv);
    col_reduce_tma<2, 1, T>(x, nullptr, M, C, rpb, chunk_rows, partial, [&](const float* xv, const float*, float* acc) {
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            const float d = xv[v] - kv[v];
            acc[v] += d;
            acc[8 + v] = fmaf(d, d, acc[8 + v]);
        }
    });
}

template <typename T>
__global__ void __launch_bounds__(RT_THREADS)
bn_bwd_reduce_tma_kernel(const T* __restrict__ dy, const T* __restrict__ z, const float* __restrict__ stats, int act,
                         long long M, int C, long long rpb, int chunk_rows, float* __restrict__ partial) {
    float mean[8], invstd[8], scale[8], shift[8];
    const int c0 = (threadIdx.x % (C / 8)) * 8;
#pragma unroll
    for (int v = 0; v < 8; ++v) {
        mean[v] = stats[c0 + v]; invstd[v] = stats[C + c0 + v]; scale[v] = stats[2 * C + c0 + v]; shift[v] = stats[3 * C + c0 + v];
    }
    col_reduce_tma<2, 2, T>(dy, z, M, C, rpb, chunk_rows, partial, [&](const float* dv, const float* zv, float* acc) {
        float u[8], ag[8];
#pragma unroll
        for (int v = 0; v < 8; ++v) u[v] = fmaf(zv[v], scale[v], shift[v]);
        act_grad_vec<8>(u, act, ag);
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            const float g = dv[v] * ag[v];
            acc[v] += g;
            acc[8 + v] = fmaf(g, (zv[v] - mean[v]) * invstd[v], acc[8 + v]);
        }
    });
}

// ---- BN (+activation) backward.  g = dy * act'(u), u = z * scale + shift, xhat = (z - mean) * invstd.
template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
bn_bwd_reduce_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ z, long long ldz,
                     const float* __restrict__ stats, int act, long long M, int C, long long rpb,
                     float* __restrict__ partial) {
    col_reduce_block<2>(M, C, rpb, partial, [&](long long m, int c, float* acc) {
        const float zv = ldf(z + m * ldz + c);
        const float u = fmaf(zv, stats[2 * C + c], stats[3 * C + c]);
        const float g = ldf(dy + m * lddy + c) * act_grad(u, act);
        acc[0] += g;
        acc[1] = fmaf(g, (zv - stats[c]) * stats[C + c], acc[1]);
    });
}

// ---- 16-byte vectorised variants (C and every pixel stride a multiple of the vector width, 16-byte aligned bases)
template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
bn_stats_v_kernel(const T* __restrict__ x, long long ldx, long long M, int C, long long rpb, float* __restrict__ partial) {
    constexpr int V = vec_n<T>();
    float kv[V];      // the shift (row 0) of this thread's channel vector: loaded once per channel chunk
    int kc = -1;
    col_reduce_block_v<2, V>(M, C, rpb, partial, [&](long long m, int c0, float* acc) {
        if (c0 != kc) {
            ldv(x + c0, kv);
            kc = c0;
        }
        float xv[V];
        ldv(x + m * ldx + c0, xv);
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float d = xv[v] - kv[v];
            acc[v] += d;
            acc[V + v] = fmaf(d, d, acc[V + v]);
        }
    });
}

template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
bn_bwd_reduce_v_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ z, long long ldz,
                       const float* __restrict__ stats, int act, long long M, int C, long long rpb,
                       float* __restrict__ partial) {
    constexpr int V = vec_n<T>();
    float mean[V], invstd[V], scale[V], shift[V];   // per-channel constants of this thread's vector, loaded once
    int kc = -1;
    col_reduce_block_v<2, V>(M, C, rpb, partial, [&](long long m, int c0, float* acc) {
        if (c0 != kc) {
#pragma unroll
            for (int v = 0; v < V; ++v) {
                mean[v] = stats[c0 + v]; invstd[v] = stats[C + c0 + v]; scale[v] = stats[2 * C + c0 + v]; shift[v] = stats[3 * C + c0 + v];
            }
            kc = c0;
        }
        float zv[V], dv[V], u[V], ag[V];
        ldv(z + m * ldz + c0, zv);
        ldv(dy + m * lddy + c0, dv);
#pragma unroll
        for (int v = 0; v < V; ++v) u[v] = fmaf(zv[v], scale[v], shift[v]);
        act_grad_vec<V>(u, act, ag);
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float g = dv[v] * ag[v];
            acc[v] += g;
            acc[V + v] = fmaf(g, (zv[v] - mean[v]) * invstd[v], acc[V + v]);
        }
    });
}

// one thread = one channel vector, walking pixels with a fixed stride: the per-channel constants stay in registers
template <typename T>
__global__ void __launch_bounds__(256)
bn_bwd_apply_v_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ z, long long ldz,
                      const float* __restrict__ stats, const float* __restrict__ coef, int act, T* __restrict__ dz,
                      long long lddz, long long M, int C, int accumulate) {
    constexpr int V = vec_n<T>();
    const int CV = C / V;
    const int cv = threadIdx.x % CV, lane = threadIdx.x / CV, lanes = blockDim.x / CV;
    if (lane >= lanes) return;
    const int c0 = cv * V;
    float mean[V], invstd[V], scale[V], shift[V], k1[V], k2[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
        mean[v] = stats[c0 + v]; invstd[v] = stats[C + c0 + v]; scale[v] = stats[2 * C + c0 + v]; shift[v] = stats[3 * C + c0 + v];
        k1[v] = coef[c0 + v]; k2[v] = coef[C + c0 + v];
    }
    const long long step = static_cast<long long>(gridDim.x) * lanes;
    for (long long m = static_cast<long long>(blockIdx.x) * lanes + lane; m < M; m += 2 * step) {
        // two rows in flight per thread
        const long long m2 = m + step;
        const bool two = m2 < M;
        float zv[V], dv[V], o[V], zv2[V], dv2[V], o2[V];
        ldv(z + m * ldz + c0, zv);
        ldv(dy + m * lddy + c0, dv);
        if (two) {
            ldv(z + m2 * ldz + c0, zv2);
            ldv(dy + m2 * lddy + c0, dv2);
        }
        if (accumulate) {
            ldv(dz + m * lddz + c0, o);
            if (two) ldv(dz + m2 * lddz + c0, o2);
        }
        float u[V], ag[V];
#pragma unroll
        for (int v = 0; v < V; ++v) u[v] = fmaf(zv[v], scale[v], shift[v]);
        act_grad_vec<V>(u, act, ag);
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float g = dv[v] * ag[v];
            const float r = scale[v] * (g - k1[v] - (zv[v] - mean[v]) * invstd[v] * k2[v]);
            o[v] = accumulate ? o[v] + r : r;
        }
        stv(dz + m * lddz + c0, o);
        if (two) {
#pragma unroll
            for (int v = 0; v < V; ++v) u[v] = fmaf(zv2[v], scale[v], shift[v]);
            act_grad_vec<V>(u, act, ag);
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const float g = dv2[v] * ag[v];
                const float r = scale[v] * (g - k1[v] - (zv2[v] - mean[v]) * invstd[v] * k2[v]);
                o2[v] = accumulate ? o2[v] + r : r;
            }
            stv(dz + m2 * lddz + c0, o2);
        }
    }
}

template <typename TZ, typename TY>
__global__ void __launch_bounds__(256)
affine_act_v_kernel(const TZ* __restrict__ z, long long ldz, const float* __restrict__ scale, const float* __restrict__ shift,
                    const float* __restrict__ gate, float gate_plus, const TY* __restrict__ res, long long ldres,
                    TY* __restrict__ y, long long ldy, long long M, long long HW, int C, int act) {
    constexpr int V = 8;  // 8 channels per thread: one or two 16-byte accesses per tensor
    const int CV = C / V;
    const int cv = threadIdx.x % CV, lane = threadIdx.x / CV, lanes = blockDim.x / CV;
    if (lane >= lanes) return;
    const int c0 = cv * V;
    float sc[V], sh[V];
#pragma unroll
    for (int v = 0; v < V; ++v) {
        sc[v] = scale ? scale[c0 + v] : 1.f;
        sh[v] = scale ? shift[c0 + v] : 0.f;
    }
    auto ld8 = [](auto* p, float* f) {
        using TT = std::remove_cv_t<std::remove_pointer_t<decltype(p)>>;
        if constexpr (sizeof(TT) == 2) ldv(p, f);
        else { ldv(p, f); ldv(p + 4, f + 4); }
    };
    for (long long m = static_cast<long long>(blockIdx.x) * lanes + lane; m < M; m += static_cast<long long>(gridDim.x) * lanes) {
        float u[V], r[V];
        ld8(z + m * ldz + c0, u);
        if (res) ld8(res + m * ldres + c0, r);
        const float* gp = gate ? gate + (m / HW) * C + c0 : nullptr;
#pragma unroll
        for (int v = 0; v < V; ++v) {
            float t = fmaf(u[v], sc[v], sh[v]);
            if (gp) t *= __ldg(gp + v) + gate_plus;
            u[v] = t;
        }
        cab_act_vec<V>(u, act);
        if (res) {
#pragma unroll
            for (int v = 0; v < V; ++v) u[v] += r[v];
        }
        TY* o = y + m * ldy + c0;
        if constexpr (sizeof(TY) == 2) stv(o, u);
        else { stv(o, u); stv(o + 4, u + 4); }
    }
}

// sums the block partials in order; dgamma / dbeta accumulate into the parameter gradients; coef[2][C] (may be NULL) =
// the two per-channel means the apply kernel subtracts
__global__ void bn_bwd_finalize_kernel(const float* __restrict__ partial, int nb, long long M, int C,
                                       float* __restrict__ dgamma, float* __restrict__ dbeta, float* __restrict__ coef) {
    const int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;  // one warp per channel
    if (c >= C) return;
    float s1 = 0.f, s2 = 0.f, t1[3] = {0.f, 0.f, 0.f}, t2[3] = {0.f, 0.f, 0.f};
    int b = lane;
    for (; b + 96 < nb; b += 128) {  // four independent chains per lane (the loads of a lane's blocks go out together)
        s1 += partial[(static_cast<long long>(b) * 2 + 0) * C + c];
        s2 += partial[(static_cast<long long>(b) * 2 + 1) * C + c];
#pragma unroll
        for (int u = 0; u < 3; ++u) {
            t1[u] += partial[(static_cast<long long>(b + 32 * (u + 1)) * 2 + 0) * C + c];
            t2[u] += partial[(static_cast<long long>(b + 32 * (u + 1)) * 2 + 1) * C + c];
        }
    }
    for (; b < nb; b += 32) {
        s1 += partial[(static_cast<long long>(b) * 2 + 0) * C + c];
        s2 += partial[(static_cast<long long>(b) * 2 + 1) * C + c];
    }
    s1 += t1[0] + t1[1] + t1[2];
    s2 += t2[0] + t2[1] + t2[2];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s1 += __shfl_xor_sync(0xffffffffu, s1, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if (lane != 0) return;
    if (dbeta) dbeta[c] += s1;
    if (dgamma) dgamma[c] += s2;
    if (!coef) return;  // eval-mode BN: its dz needs no means
    coef[c] = s1 / static_cast<float>(M);
    coef[C + c] = s2 / static_cast<float>(M);
}

template <typename T>
__global__ void __launch_bounds__(256)
bn_bwd_apply_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ z, long long ldz,
                    const float* __restrict__ stats, const float* __restrict__ coef, int act, T* __restrict__ dz,
                    long long lddz, long long M, int C, int accumulate) {
    const long long total = M * C;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long m = i / C;
        const int c = static_cast<int>(i - m * C);
        const float zv = ldf(z + m * ldz + c);
        const float u = fmaf(zv, stats[2 * C + c], stats[3 * C + c]);
        const float g = ldf(dy + m * lddy + c) * act_grad(u, act);
        const float xhat = (zv - stats[c]) * stats[C + c];
        float v = stats[2 * C + c] * (g - coef[c] - xhat * coef[C + c]);
        T* o = dz + m * lddz + c;
        if (accumulate) v += ldf(o);
        *o = from_f32<T>(v);
    }
}

// ---- eval-mode BatchNorm: stats[4][C] from the running statistics (the layout bn_finalize_kernel writes), on the device
// so that a replayed graph reads the running statistics of replay time
__global__ void bn_frozen_stats_kernel(const float* __restrict__ gamma, const float* __restrict__ beta,
                                       const float* __restrict__ run_mean, const float* __restrict__ run_var, float eps, int C,
                                       float* __restrict__ stats) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    const float mean = run_mean[c];
    const float invstd = static_cast<float>(1.0 / sqrt(static_cast<double>(run_var[c]) + static_cast<double>(eps)));
    const float g = gamma ? gamma[c] : 1.f, bt = beta ? beta[c] : 0.f;
    stats[c] = mean;
    stats[C + c] = invstd;
    stats[2 * C + c] = g * invstd;
    stats[3 * C + c] = bt - mean * g * invstd;
}

// ---- eval-mode BatchNorm (+activation) backward.  The statistics do not depend on z, so dz (+)= scale * g needs no
// column sum: ONE pass writes dz and (RED) the block partials of sum g and sum g * xhat (dbeta, dgamma; level 2 is
// bn_bwd_finalize_kernel).  dz may be NULL (parameter gradients only).  RED = false: an elementwise grid-stride pass.
template <typename T, bool RED>
__global__ void __launch_bounds__(RED_THREADS)
bn_frozen_bwd_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ z, long long ldz,
                     const float* __restrict__ stats, int act, T* __restrict__ dz, long long lddz, long long M, int C,
                     int accumulate, long long rpb, float* __restrict__ partial) {
    auto one = [&](long long m, int c, float* acc) {
        const float zv = ldf(z + m * ldz + c);
        const float sc = stats[2 * C + c];
        const float g = ldf(dy + m * lddy + c) * act_grad(fmaf(zv, sc, stats[3 * C + c]), act);
        if (dz) {
            T* o = dz + m * lddz + c;
            float r = __fmul_rn(sc, g);  // never fused into the add: every path rounds dz the same way
            if (accumulate) r += ldf(o);
            *o = from_f32<T>(r);
        }
        if (RED) {
            acc[0] += g;
            acc[1] = fmaf(g, (zv - stats[c]) * stats[C + c], acc[1]);
        }
    };
    if constexpr (RED) {
        col_reduce_block<2>(M, C, rpb, partial, one);
    } else {
        float acc[2];
        const long long total = M * C;
        for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
             i += static_cast<long long>(gridDim.x) * blockDim.x) {
            const long long m = i / C;
            one(m, static_cast<int>(i - m * C), acc);
        }
    }
}

// 16-byte vectorised form (C / V <= RED_THREADS, C and every pixel stride a multiple of V, 16-byte aligned bases)
template <typename T, bool RED>
__global__ void __launch_bounds__(RED_THREADS)
bn_frozen_bwd_v_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ z, long long ldz,
                       const float* __restrict__ stats, int act, T* __restrict__ dz, long long lddz, long long M, int C,
                       int accumulate, long long rpb, float* __restrict__ partial) {
    constexpr int V = vec_n<T>();
    float mean[V], invstd[V], scale[V], shift[V];   // per-channel constants of this thread's vector, loaded once
    int kc = -1;
    auto one = [&](long long m, int c0, float* acc) {
        if (c0 != kc) {
#pragma unroll
            for (int v = 0; v < V; ++v) {
                mean[v] = stats[c0 + v]; invstd[v] = stats[C + c0 + v]; scale[v] = stats[2 * C + c0 + v]; shift[v] = stats[3 * C + c0 + v];
            }
            kc = c0;
        }
        float zv[V], dv[V], u[V], ag[V], o[V];
        ldv(z + m * ldz + c0, zv);
        ldv(dy + m * lddy + c0, dv);
        if (dz && accumulate) ldv(dz + m * lddz + c0, o);
#pragma unroll
        for (int v = 0; v < V; ++v) u[v] = fmaf(zv[v], scale[v], shift[v]);
        act_grad_vec<V>(u, act, ag);
#pragma unroll
        for (int v = 0; v < V; ++v) {
            const float g = dv[v] * ag[v];
            if (RED) {
                acc[v] += g;
                acc[V + v] = fmaf(g, (zv[v] - mean[v]) * invstd[v], acc[V + v]);
            }
            const float r = __fmul_rn(scale[v], g);
            o[v] = accumulate ? o[v] + r : r;
        }
        if (dz) stv(dz + m * lddz + c0, o);
    };
    if constexpr (RED) {
        col_reduce_block_v<2, V>(M, C, rpb, partial, one);
    } else {
        const int CV = C / V;
        const int cv = threadIdx.x % CV, lane = threadIdx.x / CV, lanes = blockDim.x / CV;
        if (lane >= lanes) return;
        float acc[2 * V];
        for (long long m = static_cast<long long>(blockIdx.x) * lanes + lane; m < M; m += static_cast<long long>(gridDim.x) * lanes)
            one(m, cv * V, acc);
    }
}

// ---- plain activation / bias-free elementwise backward: dx = dy * act'(x)   (layers without BN)
// and the gated form y = act(v * (s[n][c] + plus)): dv = dy * act'(v * s') * s' + dm[n][c] * inv_hw
template <typename T>
__global__ void __launch_bounds__(256)
gate_bwd_apply_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ v, long long ldv,
                      const float* __restrict__ s, float plus, const float* __restrict__ dm, float inv_hw, int act,
                      T* __restrict__ dv, long long lddv, long long M, long long HW, int C, int accumulate) {
    const long long total = M * C;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long m = i / C;
        const int c = static_cast<int>(i - m * C);
        const long long nc = (m / HW) * C + c;
        const float sv = s ? s[nc] + plus : 1.f;
        const float x = ldf(v + m * ldv + c);
        float r = ldf(dy + m * lddy + c) * act_grad(x * sv, act) * sv;
        if (dm) r = fmaf(dm[nc], inv_hw, r);
        T* o = dv + m * lddv + c;
        if (accumulate) r += ldf(o);
        *o = from_f32<T>(r);
    }
}

// 16-byte vectorised forms (one thread = one channel vector of a pixel lane of image blockIdx.y: the per-(image, channel)
// constants stay in registers, no per-element index division, no per-element activation switch)
template <typename T>
__global__ void __launch_bounds__(256)
gate_bwd_apply_v_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ v, long long ldvs,
                        const float* __restrict__ s, float plus, const float* __restrict__ dm, float inv_hw, int act,
                        T* __restrict__ dv, long long lddv, long long HW, int C, int accumulate) {
    constexpr int V = vec_n<T>();
    const int CV = C / V;
    const int cv = threadIdx.x % CV, lane = threadIdx.x / CV, lanes = blockDim.x / CV;
    if (lane >= lanes) return;
    const int n = blockIdx.y, c0 = cv * V;
    float sv[V], dmv[V];
#pragma unroll
    for (int k = 0; k < V; ++k) {
        sv[k] = s ? s[static_cast<long long>(n) * C + c0 + k] + plus : 1.f;
        dmv[k] = dm ? dm[static_cast<long long>(n) * C + c0 + k] * inv_hw : 0.f;
    }
    const long long base = static_cast<long long>(n) * HW;
    for (long long m = static_cast<long long>(blockIdx.x) * lanes + lane; m < HW; m += static_cast<long long>(gridDim.x) * lanes) {
        float x[V], g[V], u[V], ag[V], o[V];
        ldv(v + (base + m) * ldvs + c0, x);
        ldv(dy + (base + m) * lddy + c0, g);
        if (accumulate) ldv(dv + (base + m) * lddv + c0, o);
#pragma unroll
        for (int k = 0; k < V; ++k) u[k] = x[k] * sv[k];
        act_grad_vec<V>(u, act, ag);
#pragma unroll
        for (int k = 0; k < V; ++k) {
            const float r = fmaf(g[k] * ag[k], sv[k], dmv[k]);
            o[k] = accumulate ? o[k] + r : r;
        }
        stv(dv + (base + m) * lddv + c0, o);
    }
}

template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
gate_bwd_reduce_v_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ v, long long ldvs,
                         const float* __restrict__ s, float plus, int act, long long HW, int C, long long rpb,
                         float* __restrict__ partial /* [N][nb][C] */) {
    constexpr int V = vec_n<T>();
    const int n = blockIdx.y, nb = gridDim.x;
    const T* dyn = dy + static_cast<long long>(n) * HW * lddy;
    const T* vn = v + static_cast<long long>(n) * HW * ldvs;
    const float* sn = s + static_cast<long long>(n) * C;
    float sv[V];
    int kc = -1;
    col_reduce_block_v<1, V>(HW, C, rpb, partial + static_cast<long long>(n) * nb * C, [&](long long m, int c0, float* acc) {
        if (c0 != kc) {
#pragma unroll
            for (int k = 0; k < V; ++k) sv[k] = sn[c0 + k] + plus;
            kc = c0;
        }
        float x[V], g[V], u[V], ag[V];
        ldv(vn + m * ldvs + c0, x);
        ldv(dyn + m * lddy + c0, g);
#pragma unroll
        for (int k = 0; k < V; ++k) u[k] = x[k] * sv[k];
        act_grad_vec<V>(u, act, ag);
#pragma unroll
        for (int k = 0; k < V; ++k) acc[k] = fmaf(g[k] * ag[k], x[k], acc[k]);
    });
}

// ds[n][c] = sum over the pixels of image n of dy * act'(v * s') * v : one block per (pixel chunk, image); two-level
template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
gate_bwd_reduce_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ v, long long ldv,
                       const float* __restrict__ s, float plus, int act, long long HW, int C, long long rpb,
                       float* __restrict__ partial /* [N][nb][C] */) {
    const int n = blockIdx.y, nb = gridDim.x;
    const T* dyn = dy + static_cast<long long>(n) * HW * lddy;
    const T* vn = v + static_cast<long long>(n) * HW * ldv;
    const float* sn = s + static_cast<long long>(n) * C;
    col_reduce_block<1>(HW, C, rpb, partial + static_cast<long long>(n) * nb * C, [&](long long m, int c, float* acc) {
        const float x = ldf(vn + m * ldv + c);
        acc[0] = fmaf(ldf(dyn + m * lddy + c) * act_grad(x * (sn[c] + plus), act), x, acc[0]);
    });
}

// out[n][c] (+)= alpha * sum_b partial[n][b][c]  (fixed order)
__global__ void sum_partials_kernel(const float* __restrict__ partial, int nb, long long count, long long group_stride,
                                    float* __restrict__ out, float alpha, int accumulate) {
    // partial is [groups][nb][count]; blockIdx.y = group
    const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const float* p = partial + static_cast<long long>(blockIdx.y) * group_stride + i;
    float sum = 0.f;
    for (int b = 0; b < nb; ++b) sum += p[static_cast<long long>(b) * count];
    float* o = out + static_cast<long long>(blockIdx.y) * count + i;
    *o = (accumulate ? *o : 0.f) + alpha * sum;
}

// column sums of a [M][C] tensor (bias gradients, per-image channel sums use cabinet_channel_sum)
template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
col_sum_kernel(const T* __restrict__ x, long long ldx, long long M, int C, long long rpb, float* __restrict__ partial) {
    col_reduce_block<1>(M, C, rpb, partial, [&](long long m, int c, float* acc) { acc[0] += ldf(x + m * ldx + c); });
}

// ---------------------------------------------------------------------------------------------------------------
// Weight packing: PyTorch OIHW fp32 -> [cout_pad][KH*KW][cin_pad] (ci fastest, zero padded) in fp32 or bf16: the layout
// cabinet_conv2d_simt / cabinet_conv_tc consume and the data-gradient kernel reads.  transposed_1 = depthwise
// ([C][1][k][k] -> [k*k][C]).
// transpose_flip: the weights of the data-gradient convolution (rows = input channels, taps mirrored, K = output channels)
template <typename TO>
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, int Cout, int Cin, int taps, int rows_pad,
                                        int k_pad, int transpose_flip, TO* __restrict__ out) {
    const long long total = static_cast<long long>(rows_pad) * taps * k_pad;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int kk = static_cast<int>(i % k_pad);
        const long long t = i / k_pad;
        const int tap = static_cast<int>(t % taps), r = static_cast<int>(t / taps);
        const int co = transpose_flip ? kk : r, ci = transpose_flip ? r : kk;
        const int src_tap = transpose_flip ? taps - 1 - tap : tap;
        float v = 0.f;
        if (co < Cout && ci < Cin) v = w[(static_cast<long long>(co) * Cin + ci) * taps + src_tap];
        out[i] = from_f32<TO>(v);
    }
}

// Sub-filter of one input-parity class (py, px) of a stride-2 convolution's data gradient, transposed for cabinet_conv_tc:
//   dx[2a+py][2b+px][ci] = sum_{jy, jx, co} dy[a - pad2 + jy][b - pad2 + jx][co] * w[co][ci][ky(jy)][kx(jx)],
//   ky(j) = py + pad - 2 (j - pad2)   (taps outside [0, K) are zero)
// out [rows_pad >= Cin][KH2 * KW2][k_pad >= Cout] bf16 / fp16, zero padded.
template <typename T>
__global__ void pack_conv_weight_parity_kernel(const float* __restrict__ w, int Cout, int Cin, int K, int pad, int py, int px,
                                               int KH2, int KW2, int pad2, int rows_pad, int k_pad, T* __restrict__ out) {
    const long long total = static_cast<long long>(rows_pad) * KH2 * KW2 * k_pad;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int co = static_cast<int>(i % k_pad);
        const long long t = i / k_pad;
        const int tap = static_cast<int>(t % (KH2 * KW2)), ci = static_cast<int>(t / (KH2 * KW2));
        const int jy = tap / KW2, jx = tap - jy * KW2;
        const int ky = py + pad - 2 * (jy - pad2), kx = px + pad - 2 * (jx - pad2);
        float v = 0.f;
        if (co < Cout && ci < Cin && ky >= 0 && ky < K && kx >= 0 && kx < K) v = w[((static_cast<long long>(co) * Cin + ci) * K + ky) * K + kx];
        out[i] = from_f32<T>(v);
    }
}

__global__ void pack_dw_weight_kernel(const float* __restrict__ w, int C, int taps, int flip, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= C * taps) return;
    const int c = i % C, t = i / C;
    out[i] = w[c * taps + (flip ? taps - 1 - t : t)];
}

// ---------------------------------------------------------------------------------------------------------------
// im2col of the fp32 NCHW network input for the two stem convolutions (7x7 s2 p3 and, embedded in its centre, 3x3 s2 p1):
// out[n*OH*OW + oy*OW + ox][ci*K*K + ky*K + kx] = T(x[n][ci][oy*S - P + ky][ox*S - P + kx]) (0 outside the image and in
// the padding columns >= Cin*K*K).  The column order is the OIHW flattening of the filter, so the stem convolutions and
// their weight gradients become plain 1x1 GEMMs on the tensor cores with the parameter / gradient tensors used in place.
template <typename T>
__global__ void __launch_bounds__(256)
im2col_nchw_kernel(const float* __restrict__ x, int N, int Cin, int H, int W, int K, int S, int P, int OH, int OW,
                   T* __restrict__ out, int ld) {
    // one thread = one output pixel x one 16-byte chunk (8 columns): consecutive threads write consecutive chunks of a row
    const unsigned chunks = ld / 8, cols = Cin * K * K, KK = K * K;
    const long long total = static_cast<long long>(N) * OH * OW * chunks;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const unsigned iu = static_cast<unsigned>(i);
        const unsigned ch = iu % chunks, pix = iu / chunks;
        const int ox = pix % OW;
        const unsigned t = pix / OW;
        const int oy = t % OH, n = t / OH;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const unsigned col = ch * 8 + j;
            v[j] = 0.f;
            if (col < cols) {
                const unsigned ci = col / KK, rem = col - ci * KK;
                const int ky = rem / K, kx = rem - ky * K;
                const int iy = oy * S - P + ky, ix = ox * S - P + kx;
                if (iy >= 0 && iy < H && ix >= 0 && ix < W) v[j] = __ldg(x + ((static_cast<long long>(n) * Cin + ci) * H + iy) * W + ix);
            }
        }
        Vec16<T> o;
        o.pack(v);
        o.store(out + static_cast<long long>(pix) * ld + ch * 8);
    }
}

// Row-segment variant: a block stages the input window of IM2COL_PX consecutive output pixels of one output row
// ([Cin][K][PX * S + K - S] fp32, coalesced along x, zero outside the image) and a column -> window-offset table in shared
// memory, then writes the PX dense rows 16 bytes per thread -- no per-element index division, every input element read from
// global memory once per block instead of once per (pixel, tap) (the per-element kernel above ran at 0.7 TB/s of its
// output bytes: 0.94 ms for the 1024 x 1024 stem of batch 8).
constexpr int IM2COL_PX = 64;
template <typename T>
__global__ void __launch_bounds__(256)
im2col_nchw_row_kernel(const float* __restrict__ x, int Cin, int H, int W, int K, int S, int P, int OH, int OW,
                       T* __restrict__ out, int ld, int segs) {
    extern __shared__ float s_win[];  // [Cin * K][winw] | int table[ld]
    const int winw = IM2COL_PX * S + K - S, rows = Cin * K, cols = Cin * K * K;
    int* s_tab = reinterpret_cast<int*>(s_win + rows * winw);
    const int seg = blockIdx.x % segs;
    const int t = blockIdx.x / segs;
    const int oy = t % OH, n = t / OH;
    const int ox0 = seg * IM2COL_PX, npx = min(IM2COL_PX, OW - ox0);
    const int ix0 = ox0 * S - P, iy0 = oy * S - P;
    for (int i = threadIdx.x; i < rows * winw; i += 256) {
        const int r = i / winw, j = i - r * winw;
        const int ci = r / K, ky = r - ci * K;
        const int iy = iy0 + ky, ix = ix0 + j;
        s_win[i] = (iy >= 0 && iy < H && ix >= 0 && ix < W) ? __ldg(x + ((static_cast<long long>(n) * Cin + ci) * H + iy) * W + ix) : 0.f;
    }
    for (int c = threadIdx.x; c < ld; c += 256) {
        const int r = c / K;  // = ci * K + ky for c = ci*K*K + ky*K + kx
        s_tab[c] = c < cols ? r * winw + (c - r * K) : -1;
    }
    __syncthreads();
    const int chunks = ld / 8;
    T* orow = out + ((static_cast<long long>(n) * OH + oy) * OW + ox0) * ld;
    for (int i = threadIdx.x; i < npx * chunks; i += 256) {
        const int px = i / chunks, ch = i - px * chunks;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int o = s_tab[ch * 8 + j];
            v[j] = o >= 0 ? s_win[o + px * S] : 0.f;
        }
        Vec16<T> o;
        o.pack(v);
        o.store(orow + static_cast<long long>(px) * ld + ch * 8);
    }
}

// dst[r][c0 + c] (+)= src[r][c] for a [rows][cols] block (embedding a 3x3 filter / its gradient in the 7x7 footprint)
__global__ void embed_filter_kernel(const float* __restrict__ w_small, int Cout, int Cin, int k, int K, float* __restrict__ w_big,
                                    int ld_big, int extract_add) {
    // w_small [Cout][Cin][k][k]  <->  w_big [Cout][ld_big], column ci*K*K + (ky + off)*K + kx + off, off = (K - k) / 2
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int total = Cout * Cin * k * k;
    if (i >= total) return;
    const int kx = i % k, ky = (i / k) % k, ci = (i / (k * k)) % Cin, co = i / (k * k * Cin);
    const int off = (K - k) / 2;
    float* big = w_big + static_cast<long long>(co) * ld_big + ci * K * K + (ky + off) * K + kx + off;
    if (extract_add) const_cast<float*>(w_small)[i] += *big;   // gradient of the embedded filter back into the small one
    else *big = w_small[i];
}

// ---------------------------------------------------------------------------------------------------------------
// Dense convolution, data gradient (implicit GEMM over (ky, kx, co)):
//   dx[n][iy][ix][ci] (+)= sum_{ky,kx,co} dy[n][oy][ox][co] * w[co][ky*KW+kx][ci],  oy = (iy + pad - ky) / stride (exact)
constexpr int GBM = 64, GBN = 64, GBK = 16;

struct DgradArgs {
    const void* dy; long long lddy;
    const void* w; long long w_sco, w_stap;  // element strides of the packed weights ([co][tap][ci], ci contiguous)
    void* dx; long long lddx;
    int N, H, W, Cin, Cout, KH, KW, stride, pad, OH, OW, accumulate;
    long long M;  // N*H*W (stride 1) or the pixels of the largest parity class (stride 2)
    int K;        // KH*KW*Cout
};

// Stride 2: the input pixels split into four parity classes (iy & 1, ix & 1) = blockIdx.z; a pixel of class (py, px) only
// meets the taps with ky = (py + pad) mod 2 (+2, +4, ...), kx likewise -- a quarter of the (pixel, tap) pairs.  Each class
// is its own dense GEMM over its valid taps (no multiplications by structural zeros).
struct ParityTaps {
    int ky0, nky, kx0, nkx, hc, wc;  // first valid ky / kx, their counts, pixel grid of the class
};
__device__ __forceinline__ ParityTaps parity_taps(const DgradArgs& a, int cls) {
    ParityTaps t;
    const int py = cls >> 1, px = cls & 1;
    t.ky0 = (py + a.pad) & 1;
    t.kx0 = (px + a.pad) & 1;
    t.nky = (a.KH - t.ky0 + 1) / 2;
    t.nkx = (a.KW - t.kx0 + 1) / 2;
    t.hc = (a.H - py + 1) / 2;
    t.wc = (a.W - px + 1) / 2;
    return t;
}

template <typename T, typename TW, bool S2>
__global__ void __launch_bounds__(256) conv_dgrad_kernel(DgradArgs a) {
    __shared__ __align__(16) float As[GBK][GBM];
    __shared__ __align__(16) float Bs[GBK][GBN + 4];
    __shared__ int pix_n[GBM], pix_y[GBM], pix_x[GBM];
    const int tid = threadIdx.x;
    const long long m0 = static_cast<long long>(blockIdx.x) * GBM;
    const int n0 = blockIdx.y * GBN;
    const T* __restrict__ dy = reinterpret_cast<const T*>(a.dy);
    const TW* __restrict__ w = reinterpret_cast<const TW*>(a.w);
    ParityTaps pt;
    int py = 0, px = 0, nkx = a.KW, Kc = a.K;
    long long Mc = a.M;
    if (S2) {
        pt = parity_taps(a, blockIdx.z);
        py = blockIdx.z >> 1; px = blockIdx.z & 1;
        nkx = pt.nkx;
        Kc = pt.nky * pt.nkx * a.Cout;
        Mc = static_cast<long long>(a.N) * pt.hc * pt.wc;
        if (m0 >= Mc || Kc == 0) {
            if (Kc != 0 || m0 >= Mc || a.accumulate) return;  // (no valid tap: the class gets zeros unless it accumulates)
        }
    }
    if (tid < GBM) {
        const long long m = m0 + tid;
        if (m < Mc) {
            const int wc = S2 ? pt.wc : a.W, hc = S2 ? pt.hc : a.H;
            const int xx = static_cast<int>(m % wc);
            const long long t = m / wc;
            pix_x[tid] = S2 ? 2 * xx + px : xx;
            pix_y[tid] = S2 ? 2 * static_cast<int>(t % hc) + py : static_cast<int>(t % hc);
            pix_n[tid] = static_cast<int>(t / hc);
        } else {
            pix_n[tid] = -1;
            pix_y[tid] = pix_x[tid] = 0;
        }
    }
    __syncthreads();
    const int ty = tid / 16, tx = tid % 16;
    float acc[4][4] = {};
    const int a_pix = tid % GBM, a_kq = tid / GBM;
    const int b_ci = tid % GBN, b_kq = tid / GBN;
    const int pn = pix_n[a_pix], iy = pix_y[a_pix], ix = pix_x[a_pix];
    for (int k0 = 0; k0 < Kc; k0 += GBK) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + a_kq * 4 + j;
            float v = 0.f;
            if (k < Kc && pn >= 0) {
                const int tap = k / a.Cout, co = k - tap * a.Cout;
                int ky = tap / nkx, kx = tap - ky * nkx;
                if (S2) { ky = pt.ky0 + 2 * ky; kx = pt.kx0 + 2 * kx; }
                const int ty2 = iy + a.pad - ky, tx2 = ix + a.pad - kx;
                if (ty2 >= 0 && tx2 >= 0 && (S2 || (ty2 % a.stride == 0 && tx2 % a.stride == 0))) {
                    const int oy = ty2 / a.stride, ox = tx2 / a.stride;
                    if (oy < a.OH && ox < a.OW)
                        v = ldf(dy + ((static_cast<long long>(pn) * a.OH + oy) * a.OW + ox) * a.lddy + co);
                }
            }
            As[a_kq * 4 + j][a_pix] = v;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int k = k0 + b_kq * 4 + j;
            const int ci = n0 + b_ci;
            float v = 0.f;
            if (k < Kc && ci < a.Cin) {
                const int tap = k / a.Cout, co = k - tap * a.Cout;
                int wtap = tap;
                if (S2) {
                    const int ky = tap / nkx, kx = tap - ky * nkx;
                    wtap = (pt.ky0 + 2 * ky) * a.KW + pt.kx0 + 2 * kx;
                }
                v = to_f32<TW>(w[co * a.w_sco + wtap * a.w_stap + ci]);
            }
            Bs[b_kq * 4 + j][b_ci] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GBK; ++kk) {
            const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float af[4] = {av.x, av.y, av.z, av.w};
            const float bf[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(af[i], bf[j], acc[i][j]);
        }
        __syncthreads();
    }
    T* __restrict__ dx = reinterpret_cast<T*>(a.dx);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int r = ty * 4 + i;
        if (m0 + r >= Mc) continue;
        const long long pix = (static_cast<long long>(pix_n[r]) * a.H + pix_y[r]) * a.W + pix_x[r];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int ci = n0 + tx * 4 + j;
            if (ci >= a.Cin) continue;
            T* o = dx + pix * a.lddx + ci;
            float v = acc[i][j];
            if (a.accumulate) v += ldf(o);
            *o = from_f32<T>(v);
        }
    }
}

// Dense convolution, weight gradient, split over the pixel dimension (blockIdx.z):
//   partial[z][co][tap*Cin + ci] = sum over the split's output pixels of dy[pix][co] * x[n][oy*s-p+ky][ox*s-p+kx][ci]
struct WgradArgs {
    const void* dy; long long lddy;
    const void* x; long long sxn, sxh, sxw, sxc;
    float* partial;
    int N, H, W, Cin, Cout, KH, KW, stride, pad, OH, OW;
    long long M, rows_per_split;  // M = N*OH*OW
    int Kn;                       // KH*KW*Cin
};

template <typename T, typename TX>
__global__ void __launch_bounds__(256) conv_wgrad_kernel(WgradArgs a) {
    __shared__ __align__(16) float As[GBK][GBM];       // dy^T : [pixel][co]
    __shared__ __align__(16) float Bs[GBK][GBN + 4];   // x    : [pixel][(tap, ci)]
    const int tid = threadIdx.x;
    const int co0 = blockIdx.x * GBM, kn0 = blockIdx.y * GBN;
    const long long r0 = static_cast<long long>(blockIdx.z) * a.rows_per_split;
    const long long r1 = min(r0 + a.rows_per_split, a.M);
    const T* __restrict__ dy = reinterpret_cast<const T*>(a.dy);
    const TX* __restrict__ x = reinterpret_cast<const TX*>(a.x);
    const int ty = tid / 16, tx = tid % 16;
    float acc[4][4] = {};
    // loaders: A: thread -> (pixel row kk = tid / 16, 4 consecutive co); B: thread -> (kk = tid / 16, 4 consecutive kn)
    const int l_kk = tid / 16, l_q = (tid % 16) * 4;
    // the (tap, ci) decomposition of this thread's four B columns is loop invariant
    int b_ky[4], b_kx[4], b_ci[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int kn = kn0 + l_q + j;
        if (kn < a.Kn) {
            const int tap = kn / a.Cin;
            b_ci[j] = kn - tap * a.Cin;
            b_ky[j] = tap / a.KW;
            b_kx[j] = tap - b_ky[j] * a.KW;
        } else {
            b_ci[j] = -1;
            b_ky[j] = b_kx[j] = 0;
        }
    }
    for (long long p0 = r0; p0 < r1; p0 += GBK) {
        const long long m = p0 + l_kk;
        int n = 0, oy = 0, ox = 0;
        const bool valid = m < r1;
        if (valid) {
            ox = static_cast<int>(m % a.OW);
            const long long t = m / a.OW;
            oy = static_cast<int>(t % a.OH);
            n = static_cast<int>(t / a.OH);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int co = co0 + l_q + j;
            As[l_kk][l_q + j] = (valid && co < a.Cout) ? ldf(dy + m * a.lddy + co) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float v = 0.f;
            if (valid && b_ci[j] >= 0) {
                const int iy = oy * a.stride - a.pad + b_ky[j], ix = ox * a.stride - a.pad + b_kx[j];
                if (iy >= 0 && iy < a.H && ix >= 0 && ix < a.W)
                    v = to_f32<TX>(x[n * a.sxn + iy * a.sxh + ix * a.sxw + b_ci[j] * a.sxc]);
            }
            Bs[l_kk][l_q + j] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < GBK; ++kk) {
            const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float af[4] = {av.x, av.y, av.z, av.w};
            const float bf[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(af[i], bf[j], acc[i][j]);
        }
        __syncthreads();
    }
    float* out = a.partial + static_cast<long long>(blockIdx.z) * a.Cout * a.Kn;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int co = co0 + ty * 4 + i;
        if (co >= a.Cout) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int kn = kn0 + tx * 4 + j;
            if (kn < a.Kn) out[static_cast<long long>(co) * a.Kn + kn] = acc[i][j];
        }
    }
}

// dW (OIHW) += sum over splits of partial[z][co][tap*Cin + ci]
__global__ void wgrad_finalize_kernel(const float* __restrict__ partial, int splits, int Cout, int Cin, int taps,
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

// ---------------------------------------------------------------------------------------------------------------
// Depthwise convolution gradients.
template <typename T>
__global__ void __launch_bounds__(256)
dw_dgrad_kernel(const T* __restrict__ dy, long long lddy, const float* __restrict__ w /* [k*k][C] */, T* __restrict__ dx,
                long long lddx, int N, int H, int W, int C, int K, int stride, int OH, int OW, int accumulate) {
    const int pad = (K - 1) / 2;
    const long long total = static_cast<long long>(N) * H * W * C;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int c = static_cast<int>(i % C);
        long long t = i / C;
        const int ix = static_cast<int>(t % W);
        t /= W;
        const int iy = static_cast<int>(t % H), n = static_cast<int>(t / H);
        float acc = 0.f;
        for (int ky = 0; ky < K; ++ky) {
            const int ty = iy + pad - ky;
            if (ty < 0 || ty % stride) continue;
            const int oy = ty / stride;
            if (oy >= OH) continue;
            for (int kx = 0; kx < K; ++kx) {
                const int tx = ix + pad - kx;
                if (tx < 0 || tx % stride) continue;
                const int ox = tx / stride;
                if (ox >= OW) continue;
                acc = fmaf(ldf(dy + ((static_cast<long long>(n) * OH + oy) * OW + ox) * lddy + c), w[(ky * K + kx) * C + c], acc);
            }
        }
        T* o = dx + ((static_cast<long long>(n) * H + iy) * W + ix) * lddx + c;
        if (accumulate) acc += ldf(o);
        *o = from_f32<T>(acc);
    }
}

// vectorised: one thread = one input pixel x one 16-byte channel vector; only the taps whose parity meets the pixel
template <typename T>
__global__ void __launch_bounds__(256)
dw_dgrad_v_kernel(const T* __restrict__ dy, long long lddy, const float* __restrict__ w, T* __restrict__ dx, long long lddx,
                  int N, int H, int W, int C, int K, int stride, int OH, int OW, int accumulate) {
    constexpr int V = vec_n<T>();
    const int pad = (K - 1) / 2, CV = C / V;
    const long long total = static_cast<long long>(N) * H * W * CV;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const unsigned iu = static_cast<unsigned>(i);  // (the host checks the vector count < 2^31)
        const int c0 = static_cast<int>(iu % static_cast<unsigned>(CV)) * V;
        unsigned t = iu / static_cast<unsigned>(CV);
        const int ix = static_cast<int>(t % static_cast<unsigned>(W));
        t /= static_cast<unsigned>(W);
        const int iy = static_cast<int>(t % static_cast<unsigned>(H)), n = static_cast<int>(t / static_cast<unsigned>(H));
        float acc[V];
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] = 0.f;
        for (int ky = (iy + pad) % stride; ky < K; ky += stride) {
            const int ty = iy + pad - ky;
            if (ty < 0) break;
            const int oy = ty / stride;
            if (oy >= OH) continue;
            for (int kx = (ix + pad) % stride; kx < K; kx += stride) {
                const int tx = ix + pad - kx;
                if (tx < 0) break;
                const int ox = tx / stride;
                if (ox >= OW) continue;
                float g[V];
                ldv(dy + ((static_cast<long long>(n) * OH + oy) * OW + ox) * lddy + c0, g);
                const float* wp = w + (ky * K + kx) * C + c0;
#pragma unroll
                for (int v = 0; v < V; ++v) acc[v] = fmaf(g[v], __ldg(wp + v), acc[v]);
            }
        }
        T* o = dx + ((static_cast<long long>(n) * H + iy) * W + ix) * lddx + c0;
        if (accumulate) {
            float old[V];
            ldv(o, old);
#pragma unroll
            for (int v = 0; v < V; ++v) acc[v] += old[v];
        }
        stv(o, acc);
    }
}

// stride 2, compile-time filter size: parity tests and shifts instead of runtime divisions, the tap loops unrolled, the
// tap weights as two 16-byte loads
template <typename T, int K>
__global__ void __launch_bounds__(256)
dw_dgrad_s2_kernel(const T* __restrict__ dy, long long lddy, const float* __restrict__ w, T* __restrict__ dx, long long lddx,
                   int N, int H, int W, int C, int OH, int OW, int accumulate) {
    constexpr int V = vec_n<T>(), pad = (K - 1) / 2, NT = (K + 1) / 2;
    const int CV = C / V;
    const long long total = static_cast<long long>(N) * H * W * CV;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const unsigned iu = static_cast<unsigned>(i);
        const int c0 = static_cast<int>(iu % static_cast<unsigned>(CV)) * V;
        unsigned t = iu / static_cast<unsigned>(CV);
        const int ix = static_cast<int>(t % static_cast<unsigned>(W));
        t /= static_cast<unsigned>(W);
        const int iy = static_cast<int>(t % static_cast<unsigned>(H)), n = static_cast<int>(t / static_cast<unsigned>(H));
        float acc[V];
#pragma unroll
        for (int v = 0; v < V; ++v) acc[v] = 0.f;
        const int py = (iy + pad) & 1, px = (ix + pad) & 1;
        const T* dyn = dy + static_cast<long long>(n) * OH * OW * lddy + c0;
#pragma unroll
        for (int a = 0; a < NT; ++a) {
            const int ky = py + 2 * a, ty = iy + pad - ky, oy = ty >> 1;
            if (ky >= K || ty < 0 || oy >= OH) continue;
#pragma unroll
            for (int b = 0; b < NT; ++b) {
                const int kx = px + 2 * b, tx = ix + pad - kx, ox = tx >> 1;
                if (kx >= K || tx < 0 || ox >= OW) continue;
                float g[V];
                ldv(dyn + (static_cast<long long>(oy) * OW + ox) * lddy, g);
                const float4* wp = reinterpret_cast<const float4*>(w + (ky * K + kx) * C + c0);
#pragma unroll
                for (int v4 = 0; v4 < V / 4; ++v4) {
                    const float4 wv = __ldg(wp + v4);
                    acc[4 * v4] = fmaf(g[4 * v4], wv.x, acc[4 * v4]);
                    acc[4 * v4 + 1] = fmaf(g[4 * v4 + 1], wv.y, acc[4 * v4 + 1]);
                    acc[4 * v4 + 2] = fmaf(g[4 * v4 + 2], wv.z, acc[4 * v4 + 2]);
                    acc[4 * v4 + 3] = fmaf(g[4 * v4 + 3], wv.w, acc[4 * v4 + 3]);
                }
            }
        }
        T* o = dx + ((static_cast<long long>(n) * H + iy) * W + ix) * lddx + c0;
        if (accumulate) {
            float old[V];
            ldv(o, old);
#pragma unroll
            for (int v = 0; v < V; ++v) acc[v] += old[v];
        }
        stv(o, acc);
    }
}

// partial[b][tap][c] = sum over the block's output pixels of dy[pix][c] * x[pix shifted by tap][c]
template <typename T, int KK>
__global__ void __launch_bounds__(RED_THREADS)
dw_wgrad_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ x, long long ldx, int H, int W, int C,
                int stride, int OH, int OW, long long M, long long rpb, float* __restrict__ partial) {
    constexpr int K = KK;
    const int pad = (K - 1) / 2;
    col_reduce_block<K * K>(M, C, rpb, partial, [&](long long m, int c, float* acc) {
        // 32-bit index arithmetic (the host checks N*OH*OW < 2^31): a 64-bit division costs ~100 instructions
        const unsigned mu = static_cast<unsigned>(m);
        const int ox = static_cast<int>(mu % static_cast<unsigned>(OW));
        const unsigned t = mu / static_cast<unsigned>(OW);
        const int oy = static_cast<int>(t % static_cast<unsigned>(OH)), n = static_cast<int>(t / static_cast<unsigned>(OH));
        const float g = ldf(dy + m * lddy + c);
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
            const int iy = oy * stride - pad + ky;
#pragma unroll
            for (int kx = 0; kx < K; ++kx) {
                const int ix = ox * stride - pad + kx;
                if (iy >= 0 && iy < H && ix >= 0 && ix < W)
                    acc[ky * K + kx] = fmaf(g, ldf(x + ((static_cast<long long>(n) * H + iy) * W + ix) * ldx + c), acc[ky * K + kx]);
            }
        }
    });
}

// channel-pair variant (4-byte bf16x2 / 8-byte float2 accesses: a warp reads 128 / 256 contiguous bytes per tap)
template <typename T> __device__ __forceinline__ float2 ld2(const T* p);
template <> __device__ __forceinline__ float2 ld2<float>(const float* p) { return *reinterpret_cast<const float2*>(p); }
template <> __device__ __forceinline__ float2 ld2<bf16>(const bf16* p) { return cab_unpack2<bf16>(*reinterpret_cast<const uint32_t*>(p)); }
template <> __device__ __forceinline__ float2 ld2<f16>(const f16* p) { return cab_unpack2<f16>(*reinterpret_cast<const uint32_t*>(p)); }

template <typename T, int KK>
__global__ void __launch_bounds__(RED_THREADS)
dw_wgrad_v2_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ x, long long ldx, int H, int W, int C,
                   int stride, int OH, int OW, long long M, long long rpb, float* __restrict__ partial) {
    constexpr int K = KK;
    const int pad = (K - 1) / 2;
    col_reduce_block_v<K * K, 2>(M, C, rpb, partial, [&](long long m, int c0, float* acc) {
        // 32-bit index arithmetic (the host checks N*OH*OW < 2^31): a 64-bit division costs ~100 instructions
        const unsigned mu = static_cast<unsigned>(m);
        const int ox = static_cast<int>(mu % static_cast<unsigned>(OW));
        const unsigned t = mu / static_cast<unsigned>(OW);
        const int oy = static_cast<int>(t % static_cast<unsigned>(OH)), n = static_cast<int>(t / static_cast<unsigned>(OH));
        const float2 g = ld2(dy + m * lddy + c0);
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
            const int iy = oy * stride - pad + ky;
#pragma unroll
            for (int kx = 0; kx < K; ++kx) {
                const int ix = ox * stride - pad + kx;
                if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
                    const float2 xv = ld2(x + ((static_cast<long long>(n) * H + iy) * W + ix) * ldx + c0);
                    acc[(ky * K + kx) * 2] = fmaf(g.x, xv.x, acc[(ky * K + kx) * 2]);
                    acc[(ky * K + kx) * 2 + 1] = fmaf(g.y, xv.y, acc[(ky * K + kx) * 2 + 1]);
                }
            }
        }
    });
}

// Line-walking variant: one thread = one segment of an output line (n, oy) x one channel pair; it slides a K x K
// register window of x along the segment, so a step costs K * S new 4-byte loads instead of K * K (and no per-pixel
// index arithmetic).  Lines are cut into `nseg` segments of `seg_len` pixels so that even a 256-line layer fills the
// machine (whole lines left 128 blocks of dependent 256-step walks: latency bound, 13x the HBM floor).
template <typename T, int KK, int S>
__global__ void __launch_bounds__(RED_THREADS)
dw_wgrad_line_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ x, long long ldx, int H, int W, int C,
                     int OH, int OW, long long n_items, int nseg, int seg_len, long long rpb, float* __restrict__ partial) {
    constexpr int K = KK;
    constexpr int pad = (K - 1) / 2;
    col_reduce_block_v<K * K, 2, false>(n_items, C, rpb, partial, [&](long long item, int c0, float* acc) {
        const unsigned iu = static_cast<unsigned>(item);
        const unsigned lu = iu / static_cast<unsigned>(nseg);
        const int ox0 = static_cast<int>(iu - lu * static_cast<unsigned>(nseg)) * seg_len, ox1 = min(OW, ox0 + seg_len);
        const long long line = lu;
        const int oy = static_cast<int>(lu % static_cast<unsigned>(OH)), n = static_cast<int>(lu / static_cast<unsigned>(OH));
        const T* xrow[K];
        bool rv[K];
#pragma unroll
        for (int ky = 0; ky < K; ++ky) {
            const int iy = oy * S - pad + ky;
            rv[ky] = iy >= 0 && iy < H;
            xrow[ky] = x + (static_cast<long long>(n) * H + (rv[ky] ? iy : 0)) * W * ldx + c0;
        }
        float2 win[K][K];
#pragma unroll
        for (int ky = 0; ky < K; ++ky)
#pragma unroll
            for (int kx = 0; kx < K; ++kx) {
                const int ix = ox0 * S + kx - pad;
                win[ky][kx] = (rv[ky] && ix >= 0 && ix < W) ? ld2(xrow[ky] + static_cast<long long>(ix) * ldx) : make_float2(0.f, 0.f);
            }
        const T* dyp = dy + line * OW * lddy + c0;
        for (int ox = ox0; ox < ox1; ++ox) {
            const float2 g = ld2(dyp + static_cast<long long>(ox) * lddy);
#pragma unroll
            for (int ky = 0; ky < K; ++ky)
#pragma unroll
                for (int kx = 0; kx < K; ++kx) {
                    acc[(ky * K + kx) * 2] = fmaf(g.x, win[ky][kx].x, acc[(ky * K + kx) * 2]);
                    acc[(ky * K + kx) * 2 + 1] = fmaf(g.y, win[ky][kx].y, acc[(ky * K + kx) * 2 + 1]);
                }
            if (ox + 1 < ox1) {
#pragma unroll
                for (int ky = 0; ky < K; ++ky) {
#pragma unroll
                    for (int kx = 0; kx + S < K; ++kx) win[ky][kx] = win[ky][kx + S];
#pragma unroll
                    for (int j = 0; j < S; ++j) {
                        if (K - S + j < 0) continue;
                        const int ix = (ox + 1) * S - pad + K - S + j;
                        win[ky][K - S + j] = (rv[ky] && ix >= 0 && ix < W) ? ld2(xrow[ky] + static_cast<long long>(ix) * ldx) : make_float2(0.f, 0.f);
                    }
                }
            }
        }
    });
}

// Row-tap variant: one thread = (channel pair, filter row ky, segment of an output line).  It owns the K taps of ONE
// filter row, i.e. K accumulator pairs and a sliding window over ONE input row: ~50 registers instead of ~130, so 5-6
// blocks per SM are resident, and it moves U = 4 output pixels per iteration with the 4 S + 4 loads of the NEXT
// iteration already in flight (the line walker above had one dependent batch of loads per pixel and two blocks per SM:
// latency bound at 0.2-0.6 TB/s).  Lanes: `cw` channel pairs x 32 / cw segments per warp, warps = K filter rows x 2.
// Block (bx, by) writes partial[bx][tap][channels of chunk by]; fixed summation order (deterministic).
template <typename T> struct Raw2;
template <> struct Raw2<float> {
    typedef float2 type;
    static __device__ __forceinline__ float2 zero() { return make_float2(0.f, 0.f); }
    static __device__ __forceinline__ float2 load(const float* p) { return *reinterpret_cast<const float2*>(p); }
    static __device__ __forceinline__ float2 cvt(float2 r) { return r; }
};
template <typename T> struct Raw2Half {  // T = bf16 or f16: two packed elements in one 32-bit word
    typedef uint32_t type;
    static __device__ __forceinline__ uint32_t zero() { return 0u; }
    static __device__ __forceinline__ uint32_t load(const T* p) { return *reinterpret_cast<const uint32_t*>(p); }
    static __device__ __forceinline__ float2 cvt(uint32_t r) { return cab_unpack2<T>(r); }
};
template <> struct Raw2<bf16> : Raw2Half<bf16> {};
template <> struct Raw2<f16> : Raw2Half<f16> {};

constexpr int DWR_SL = 2;  // segment lanes (warps per filter row) of a block

template <typename T, int K, int S>
__global__ void __launch_bounds__(32 * K * DWR_SL)
dw_wgrad_row_kernel(const T* __restrict__ dy, long long lddy, const T* __restrict__ x, long long ldx, int H, int W, int C,
                    int OH, int OW, int n_items, int nseg, int seg_len, int items_per_block, int cw_log2,
                    float* __restrict__ partial) {
    constexpr int pad = (K - 1) / 2, U = 4, NCOL = (U - 1) * S + K, NEW = U * S, KEEP = NCOL - NEW;
    typedef Raw2<T> R;
    typedef typename R::type raw_t;
    __shared__ float s_red[K][K][64];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ky = warp % K, sl = warp / K;
    const int cw = 1 << cw_log2, nsub = 32 >> cw_log2;
    const int pl = lane & (cw - 1), sub = lane >> cw_log2;
    const int c0 = (static_cast<int>(blockIdx.y) * cw + pl) * 2;
    const bool c_ok = c0 < C;
    float2 acc[K];
#pragma unroll
    for (int kx = 0; kx < K; ++kx) acc[kx] = make_float2(0.f, 0.f);
    const int it0 = static_cast<int>(blockIdx.x) * items_per_block, it1 = min(it0 + items_per_block, n_items);
    for (int item = it0 + sl * nsub + sub; item < it1; item += DWR_SL * nsub) {
        const unsigned lu = static_cast<unsigned>(item) / static_cast<unsigned>(nseg);
        const int ox0 = (item - static_cast<int>(lu) * nseg) * seg_len, ox1 = min(OW, ox0 + seg_len);
        const int oy = static_cast<int>(lu % static_cast<unsigned>(OH)), n = static_cast<int>(lu / static_cast<unsigned>(OH));
        const int iy = oy * S - pad + ky;
        if (!c_ok || iy < 0 || iy >= H || ox0 >= ox1) continue;
        const T* xr = x + (static_cast<long long>(n) * H + iy) * W * ldx + c0;
        const T* dp = dy + static_cast<long long>(lu) * OW * lddy + c0;
        float2 win[NCOL];
#pragma unroll
        for (int j = 0; j < KEEP; ++j) {  // columns ox0 * S - pad + j
            const int ix = ox0 * S - pad + j;
            win[j] = (ix >= 0 && ix < W) ? R::cvt(R::load(xr + static_cast<long long>(ix) * ldx)) : make_float2(0.f, 0.f);
        }
        raw_t rx[NEW], rg[U];
        auto fetch = [&](int ox) {  // the NEW input columns and U gradients of the group starting at output column ox
#pragma unroll
            for (int j = 0; j < NEW; ++j) {
                const int ix = ox * S - pad + KEEP + j;  // >= 0: KEEP = K - S >= pad
                rx[j] = ix < W ? R::load(xr + static_cast<long long>(ix) * ldx) : R::zero();
            }
#pragma unroll
            for (int u = 0; u < U; ++u) rg[u] = ox + u < ox1 ? R::load(dp + static_cast<long long>(ox + u) * lddy) : R::zero();
        };
        fetch(ox0);
        for (int ox = ox0; ox < ox1; ox += U) {
            float2 g[U];
#pragma unroll
            for (int j = 0; j < NEW; ++j) win[KEEP + j] = R::cvt(rx[j]);
#pragma unroll
            for (int u = 0; u < U; ++u) g[u] = R::cvt(rg[u]);
            if (ox + U < ox1) fetch(ox + U);  // in flight under the FMAs below
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int kx = 0; kx < K; ++kx) {
                    acc[kx].x = fmaf(g[u].x, win[u * S + kx].x, acc[kx].x);
                    acc[kx].y = fmaf(g[u].y, win[u * S + kx].y, acc[kx].y);
                }
#pragma unroll
            for (int j = 0; j < KEEP; ++j) win[j] = win[NEW + j];
        }
    }
    // segments of a warp (fixed butterfly), then the two segment lanes through shared memory
#pragma unroll
    for (int kx = 0; kx < K; ++kx)
        for (int o = cw; o < 32; o <<= 1) {
            acc[kx].x += __shfl_xor_sync(0xffffffffu, acc[kx].x, o);
            acc[kx].y += __shfl_xor_sync(0xffffffffu, acc[kx].y, o);
        }
    if (sl == 1 && sub == 0) {
#pragma unroll
        for (int kx = 0; kx < K; ++kx) {
            s_red[ky][kx][2 * pl] = acc[kx].x;
            s_red[ky][kx][2 * pl + 1] = acc[kx].y;
        }
    }
    __syncthreads();
    if (sl == 0 && sub == 0 && c_ok) {
#pragma unroll
        for (int kx = 0; kx < K; ++kx) {
            float* out = partial + (static_cast<long long>(blockIdx.x) * (K * K) + ky * K + kx) * C + c0;
            out[0] = acc[kx].x + s_red[ky][kx][2 * pl];
            out[1] = acc[kx].y + s_red[ky][kx][2 * pl + 1];
        }
    }
}

// dW ([C][1][k][k]) += sum_b partial[b][tap][c]: one warp per output (lane l adds blocks l, l + 32, ... then a fixed
// butterfly: deterministic)
__global__ void dw_wgrad_finalize_kernel(const float* __restrict__ partial, int nb, int C, int taps, float* __restrict__ dw) {
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (i >= C * taps) return;
    const int c = i % C, t = i / C;
    float sum = 0.f;
    for (int b = lane; b < nb; b += 32) sum += partial[(static_cast<long long>(b) * taps + t) * C + c];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) dw[c * taps + t] += sum;
}

// ---------------------------------------------------------------------------------------------------------------
// Separable sparse resampling: out[n][oy][ox][c] (+)= sum_{iy in Ry[oy]} sum_{ix in Rx[ox]} wy * wx * in[n][iy][ix][c].
// The row operators come as CSR tables (start[o], start[o+1]) -> (index, weight).  With the forward matrices of a
// bilinear resize / adaptive average pool this is the forward op; with their transposes it is the exact adjoint, which
// is what the backward of every F.interpolate / AdaptiveAvgPool2d of the network needs.  Generic element strides on
// both sides (NHWC maps and the NCHW logit gradients).
template <typename TI, typename TO>
__global__ void __launch_bounds__(256)
resample_sep_kernel(const TI* __restrict__ in, long long isn, long long isy, long long isx, long long isc,
                    TO* __restrict__ out, long long osn, long long osy, long long osx, long long osc, int N, int OH, int OW,
                    int C, const int* __restrict__ ys, const int* __restrict__ yi, const float* __restrict__ yw,
                    const int* __restrict__ xs, const int* __restrict__ xi, const float* __restrict__ xw, int accumulate) {
    const long long total = static_cast<long long>(N) * OH * OW * C;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        // c fastest when the output is channel-contiguous, x fastest otherwise (coalesced stores either way; x-fastest
        // threads for the x8 adjoint of the planar logit gradients measured 2.8x slower: 1.08 vs 0.39 ms)
        // (32-bit index arithmetic: the host checks total < 2^31)
        int c, ox, oy, n;
        unsigned t = static_cast<unsigned>(i);
        const unsigned uC = C, uW = OW, uH = OH;
        if (osc == 1) {
            c = static_cast<int>(t % uC); t /= uC;
            ox = static_cast<int>(t % uW); t /= uW;
            oy = static_cast<int>(t % uH); n = static_cast<int>(t / uH);
        } else {
            ox = static_cast<int>(t % uW); t /= uW;
            oy = static_cast<int>(t % uH); t /= uH;
            c = static_cast<int>(t % uC); n = static_cast<int>(t / uC);
        }
        float acc = 0.f;
        const TI* base = in + n * isn + c * isc;
        for (int a = ys[oy]; a < ys[oy + 1]; ++a) {
            const TI* row = base + yi[a] * isy;
            float r = 0.f;
            for (int b = xs[ox]; b < xs[ox + 1]; ++b) r = fmaf(xw[b], ldf(row + xi[b] * isx), r);
            acc = fmaf(yw[a], r, acc);
        }
        TO* o = out + n * osn + oy * osy + ox * osx + c * osc;
        if (accumulate) acc += ldf(o);
        *o = from_f32<TO>(acc);
    }
}

// Planar input, many taps per output (the x8 adjoint of the NCHW logit gradients: 16 x 16 taps): one block = one output
// row of one plane.  Phase 1 adds the rows of the band into a shared-memory line (coalesced reads along x: every input
// row is read by two blocks), phase 2 applies the x operator from that line.  Same CSR tables -> same result as the
// generic kernel up to the summation order (fixed).
template <typename TI, typename TO>
__global__ void __launch_bounds__(256)
resample_band_kernel(const TI* __restrict__ in, long long isn, long long isy, long long isc, int W_in, TO* __restrict__ out,
                     long long osn, long long osy, long long osx, long long osc, int C, int OW, const int* __restrict__ ys,
                     const int* __restrict__ yi, const float* __restrict__ yw, const int* __restrict__ xs,
                     const int* __restrict__ xi, const float* __restrict__ xw, int accumulate, int vec) {
    extern __shared__ float s_line[];  // [W_in]
    const int oy = blockIdx.x, n = blockIdx.y / C, c = blockIdx.y - n * C;
    const TI* plane = in + n * isn + c * isc;
    const int a0 = ys[oy], a1 = ys[oy + 1];
    if (vec) {
        // 16-byte loads (8 bf16 / 4 fp32 columns per thread), the band's rows unrolled four at a time: up to 64 bytes in
        // flight per thread instead of one 2-byte load per tap
        constexpr int V = vec_n<TI>();
        for (int x = threadIdx.x * V; x < W_in; x += 256 * V) {
            float acc[V];
#pragma unroll
            for (int v = 0; v < V; ++v) acc[v] = 0.f;
            int a = a0;
            for (; a + 4 <= a1; a += 4) {
                float r[4][V];
#pragma unroll
                for (int u = 0; u < 4; ++u) ldv(plane + yi[a + u] * isy + x, r[u]);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const float w = yw[a + u];
#pragma unroll
                    for (int v = 0; v < V; ++v) acc[v] = fmaf(w, r[u][v], acc[v]);
                }
            }
            for (; a < a1; ++a) {
                float r[V];
                ldv(plane + yi[a] * isy + x, r);
                const float w = yw[a];
#pragma unroll
                for (int v = 0; v < V; ++v) acc[v] = fmaf(w, r[v], acc[v]);
            }
#pragma unroll
            for (int v = 0; v < V; ++v) s_line[x + v] = acc[v];
        }
    } else {
        for (int x = threadIdx.x; x < W_in; x += 256) {
            float acc = 0.f;
            for (int a = a0; a < a1; ++a) acc = fmaf(yw[a], ldf(plane + yi[a] * isy + x), acc);
            s_line[x] = acc;
        }
    }
    __syncthreads();
    for (int ox = threadIdx.x; ox < OW; ox += 256) {
        float acc = 0.f;
        for (int b = xs[ox]; b < xs[ox + 1]; ++b) acc = fmaf(xw[b], s_line[xi[b]], acc);
        TO* o = out + n * osn + oy * osy + ox * osx + c * osc;
        if (accumulate) acc += ldf(o);
        *o = from_f32<TO>(acc);
    }
}

// Channel-contiguous (NHWC -> NHWC) form: one thread = 8 channels of one output pixel, 16-byte loads per tap.
template <typename TI, typename TO>
__global__ void __launch_bounds__(256)
resample_sep_v_kernel(const TI* __restrict__ in, long long isn, long long isy, long long isx, TO* __restrict__ out,
                      long long osn, long long osy, long long osx, int N, int OH, int OW, int C, const int* __restrict__ ys,
                      const int* __restrict__ yi, const float* __restrict__ yw, const int* __restrict__ xs,
                      const int* __restrict__ xi, const float* __restrict__ xw, int accumulate) {
    const unsigned CV = C / 8;
    const long long total = static_cast<long long>(N) * OH * OW * CV;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        unsigned t = static_cast<unsigned>(i);
        const int cv = static_cast<int>(t % CV); t /= CV;
        const int ox = static_cast<int>(t % static_cast<unsigned>(OW)); t /= static_cast<unsigned>(OW);
        const int oy = static_cast<int>(t % static_cast<unsigned>(OH)), n = static_cast<int>(t / static_cast<unsigned>(OH));
        float acc[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = 0.f;
        const TI* base = in + n * isn + cv * 8;
        const int xb0 = xs[ox], xb1 = xs[ox + 1];
        for (int a = ys[oy]; a < ys[oy + 1]; ++a) {
            const TI* row = base + yi[a] * isy;
            const float wy = yw[a];
            for (int b = xb0; b < xb1; ++b) {
                const float w = wy * xw[b];
                float v[8];
                if constexpr (sizeof(TI) == 2) {
                    ldv(row + xi[b] * isx, v);
                } else {
                    ldv(row + xi[b] * isx, v);
                    ldv(row + xi[b] * isx + 4, v + 4);
                }
#pragma unroll
                for (int k = 0; k < 8; ++k) acc[k] = fmaf(w, v[k], acc[k]);
            }
        }
        TO* o = out + n * osn + oy * osy + ox * osx + cv * 8;
        if (accumulate) {
            float p[8];
            if constexpr (sizeof(TO) == 2) {
                ldv(o, p);
            } else {
                ldv(o, p);
                ldv(o + 4, p + 4);
            }
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[k] += p[k];
        }
        if constexpr (sizeof(TO) == 2) {
            stv(o, acc);
        } else {
            stv(o, acc);
            stv(o + 4, acc + 4);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// softmax backward over rows: ds = p * (dp - sum_j dp_j p_j) * alpha
__global__ void __launch_bounds__(256)
softmax_bwd_kernel(const float* __restrict__ p, const float* __restrict__ dp, float* __restrict__ ds, long long rows,
                   int cols, float alpha) {
    const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x % 32;
    if (row >= rows) return;
    const float* pr = p + row * cols;
    const float* dr = dp + row * cols;
    float dot = 0.f;
    for (int c = lane; c < cols; c += 32) dot = fmaf(pr[c], dr[c], dot);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    float* out = ds + row * cols;
    for (int c = lane; c < cols; c += 32) out[c] = pr[c] * (dr[c] - dot) * alpha;
}

// Attention on the tensor cores (training, bf16 / fp16 mode): the GEMMs run as cabinet_conv_tc_imgw / cabinet_conv_wgrad_tc
// calls on 2-byte operands (T); these three passes sit between them.
// p = softmax(scale * s) over rows, written as fp32 (kept for the backward) AND as T (the operand of P V and P^T dO)
template <typename T>
__global__ void __launch_bounds__(256)
attn_softmax_kernel(const float* __restrict__ s, float scale, float* __restrict__ p, T* __restrict__ p16, long long rows,
                    int cols) {
    const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x % 32;
    if (row >= rows) return;
    const float* in = s + row * cols;
    float m = -INFINITY;
    for (int c = lane; c < cols; c += 32) m = fmaxf(m, in[c] * scale);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float sum = 0.f;
    for (int c = lane; c < cols; c += 32) sum += expf(in[c] * scale - m);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv = 1.f / sum;
    for (int c = lane; c < cols; c += 32) {
        const float v = expf(in[c] * scale - m) * inv;
        p[row * cols + c] = v;
        p16[row * cols + c] = from_f32<T>(v);
    }
}

// ds = p * (dp - sum_j dp_j p_j) * alpha as T (the operand of dS K and dS^T Q)
template <typename T>
__global__ void __launch_bounds__(256)
attn_softmax_bwd_kernel(const float* __restrict__ p, const float* __restrict__ dp, T* __restrict__ ds, long long rows,
                        int cols, float alpha) {
    const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x / 32) + threadIdx.x / 32;
    const int lane = threadIdx.x % 32;
    if (row >= rows) return;
    const float* pr = p + row * cols;
    const float* dr = dp + row * cols;
    float dot = 0.f;
    for (int c = lane; c < cols; c += 32) dot = fmaf(pr[c], dr[c], dot);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    for (int c = lane; c < cols; c += 32) ds[row * cols + c] = from_f32<T>(pr[c] * (dr[c] - dot) * alpha);
}

// out[n][c][l] = x[n][l][c] (2-byte T): per-image K^T / V^T as cabinet_conv_tc weight matrices ([rows = channels][k = tokens])
template <typename T>
__global__ void __launch_bounds__(256)
transpose_tokens_kernel(const T* __restrict__ x, long long ldx, T* __restrict__ out, int L, int C) {
    __shared__ T tile[32][34];
    const int n = blockIdx.z, l0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    const T* xin = x + static_cast<long long>(n) * L * ldx;
#pragma unroll
    for (int r = ty; r < 32; r += 8)
        if (l0 + r < L && c0 + tx < C) tile[r][tx] = xin[static_cast<long long>(l0 + r) * ldx + c0 + tx];
    __syncthreads();
    T* o = out + static_cast<long long>(n) * C * L;
#pragma unroll
    for (int r = ty; r < 32; r += 8)
        if (c0 + r < C && l0 + tx < L) o[static_cast<long long>(c0 + r) * L + l0 + tx] = tile[tx][r];
}

// CAB combine backward: out = gamma * g + x + x * sigmoid(r)
template <typename T>
__global__ void __launch_bounds__(RED_THREADS)
cab_combine_bwd_kernel(const T* __restrict__ dout, long long ldo, const T* __restrict__ g, const T* __restrict__ x,
                       const T* __restrict__ r, const float* __restrict__ gamma, T* __restrict__ dg, T* __restrict__ dx,
                       T* __restrict__ dr, long long M, int C, long long rpb, float* __restrict__ partial, int accumulate_dx) {
    const float gm = *gamma;
    // column-reduction helper doubles as the elementwise pass: acc[0] collects dout * g per channel (dgamma = its total)
    col_reduce_block<1>(M, C, rpb, partial, [&](long long m, int c, float* acc) {
        const long long i = m * C + c;
        const float d = ldf(dout + m * ldo + c), xv = ldf(x + i), gv = ldf(g + i);
        const float s = 1.f / (1.f + __expf(-ldf(r + i)));
        acc[0] = fmaf(d, gv, acc[0]);
        dg[i] = from_f32<T>(gm * d);
        float v = d * (1.f + s);
        if (accumulate_dx) v += ldf(dx + i);
        dx[i] = from_f32<T>(v);
        dr[i] = from_f32<T>(d * xv * s * (1.f - s));
    });
}

// total of a [nb][C] partial buffer -> one scalar accumulated into out (dgamma)
__global__ void sum_all_kernel(const float* __restrict__ partial, long long count, float* __restrict__ out) {
    __shared__ float s[256];
    float acc = 0.f;
    for (long long i = threadIdx.x; i < count; i += 256) acc += partial[i];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out += s[0];
}

// out = a + b  (gradient fan-in / residual add), any mix of pixel strides
template <typename T>
__global__ void __launch_bounds__(256)
add_kernel(const T* __restrict__ a, long long lda, const T* __restrict__ b, long long ldb, T* __restrict__ out,
           long long ldo, long long M, int C) {
    const long long total = M * C;
    for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
         i += static_cast<long long>(gridDim.x) * blockDim.x) {
        const long long m = i / C;
        const int c = static_cast<int>(i - m * C);
        out[m * ldo + c] = from_f32<T>(ldf(a + m * lda + c) + ldf(b + m * ldb + c));
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Gate MLP backward (SE: Linear + ReLU + Linear + hard-sigmoid; FFM: 1x1 + ReLU + 1x1 + sigmoid), tiny matrices:
//   a2 = W2 h + b2, s = gate(a2);  h = relu(W1 m + b1)
// phase 0: da2[n][c] = ds[n][c] * gate'(.) (from s); phase 1: dW2, db2; phase 2: da1 = (da2 W2) * (h > 0);
// phase 3: dW1, db1; phase 4: dm = da1 W1.  One launch per phase (the phases depend on each other).
__global__ void gate_bwd_phase_kernel(int phase, int N, int C, int J, int gate, float m_scale, const float* __restrict__ m,
                                      const float* __restrict__ W1, const float* __restrict__ W2, const float* __restrict__ h,
                                      const float* __restrict__ s, const float* __restrict__ ds, float* __restrict__ da2,
                                      float* __restrict__ da1, float* __restrict__ dW1, float* __restrict__ db1,
                                      float* __restrict__ dW2, float* __restrict__ db2, float* __restrict__ dm) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (phase == 0) {
        if (i >= N * C) return;
        const float sv = s[i];
        const float d = gate == CABINET_ACT_SIGMOID ? sv * (1.f - sv) : ((sv > 0.f && sv < 1.f) ? (1.f / 6.f) : 0.f);
        da2[i] = ds[i] * d;
    } else if (phase == 1) {
        if (i >= C * J) return;
        const int c = i / J, j = i - c * J;
        float acc = 0.f;
        for (int n = 0; n < N; ++n) acc = fmaf(da2[n * C + c], h[n * J + j], acc);
        dW2[i] += acc;
        if (j == 0 && db2) {
            float b = 0.f;
            for (int n = 0; n < N; ++n) b += da2[n * C + c];
            db2[c] += b;
        }
    } else if (phase == 2) {
        if (i >= N * J) return;
        const int n = i / J, j = i - n * J;
        float acc = 0.f;
        for (int c = 0; c < C; ++c) acc = fmaf(da2[n * C + c], W2[c * J + j], acc);
        da1[i] = h[i] > 0.f ? acc : 0.f;
    } else if (phase == 3) {
        if (i >= J * C) return;
        const int j = i / C, c = i - j * C;
        float acc = 0.f;
        for (int n = 0; n < N; ++n) acc = fmaf(da1[n * J + j], m[n * C + c] * m_scale, acc);
        dW1[i] += acc;
        if (c == 0 && db1) {
            float b = 0.f;
            for (int n = 0; n < N; ++n) b += da1[n * J + j];
            db1[j] += b;
        }
    } else {
        if (i >= N * C) return;
        const int n = i / C, c = i - n * C;
        float acc = 0.f;
        for (int j = 0; j < J; ++j) acc = fmaf(da1[n * J + j], W1[j * C + c], acc);
        dm[i] = acc;
    }
}

// Phases 2 and 4 with one WARP per output: the lanes stride over the reduction index (C up to 960: a thread per output
// walked it alone, 16 us per launch), fixed butterfly at the end.
__global__ void __launch_bounds__(256)
gate_bwd_dot_kernel(int phase, int N, int C, int J, const float* __restrict__ W1, const float* __restrict__ W2,
                    const float* __restrict__ h, const float* __restrict__ da2, float* __restrict__ da1, float* __restrict__ dm) {
    const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    float acc = 0.f;
    if (phase == 2) {
        if (i >= N * J) return;
        const int n = i / J, j = i - n * J;
        for (int c = lane; c < C; c += 32) acc = fmaf(da2[n * C + c], W2[c * J + j], acc);
    } else {
        if (i >= N * C) return;
        const int n = i / C, c = i - n * C;
        for (int j = lane; j < J; j += 32) acc = fmaf(da1[n * J + j], W1[j * C + c], acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane != 0) return;
    if (phase == 2) da1[i] = h[i] > 0.f ? acc : 0.f;
    else dm[i] = acc;
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline unsigned row_grid(long long M, int lanes) { return static_cast<unsigned>(std::max<long long>(1, std::min<long long>(cab_ceil_div(M, lanes), 148LL * 8))); }
inline unsigned ew_grid(long long total) { return static_cast<unsigned>(std::min<long long>(cab_ceil_div(total, 256), 148LL * 16)); }

}  // namespace

extern "C" int cabinet_pack_conv_weight(const float* w_oihw, int Cout, int Cin, int KH, int KW, void* out, int out_dtype,
                                        int rows_pad, int k_pad, int transpose_flip, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("pack_conv_weight", out_dtype, CAB_DT_ALL);
    CAB_REQUIRE(w_oihw && out && Cout > 0 && Cin > 0 && KH > 0 && KW > 0 && rows_pad >= (transpose_flip ? Cin : Cout) &&
                    k_pad >= (transpose_flip ? Cout : Cin),
                "pack_conv_weight: bad arguments");
    const long long total = static_cast<long long>(rows_pad) * KH * KW * k_pad;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CAB_DISPATCH_DT(out_dtype, T,
                    pack_conv_weight_kernel<T><<<ew_grid(total), 256, 0, s>>>(w_oihw, Cout, Cin, KH * KW, rows_pad, k_pad,
                                                                             transpose_flip, reinterpret_cast<T*>(out)));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_pack_conv_weight_parity(const float* w_oihw, int Cout, int Cin, int K, int pad, int py, int px, int KH2,
                                               int KW2, int pad2, void* out, int rows_pad, int k_pad, cabinet_stream_t stream) {
    return cabinet_pack_conv_weight_parity_dt(w_oihw, Cout, Cin, K, pad, py, px, KH2, KW2, pad2, out, rows_pad, k_pad, CABINET_BF16,
                                              stream);
}

extern "C" int cabinet_pack_conv_weight_parity_dt(const float* w_oihw, int Cout, int Cin, int K, int pad, int py, int px, int KH2,
                                                  int KW2, int pad2, void* out, int rows_pad, int k_pad, int out_dtype,
                                                  cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("pack_conv_weight_parity", out_dtype, CAB_DT_BF16 | CAB_DT_F16);
    CAB_REQUIRE(w_oihw && out && Cout > 0 && Cin > 0 && K > 0 && KH2 > 0 && KW2 > 0 && rows_pad >= Cin && k_pad >= Cout &&
                    (py == 0 || py == 1) && (px == 0 || px == 1),
                "pack_conv_weight_parity: bad arguments");
    const long long total = static_cast<long long>(rows_pad) * KH2 * KW2 * k_pad;
    CAB_DISPATCH_DT_HALF(out_dtype, T,
                    pack_conv_weight_parity_kernel<T><<<ew_grid(total), 256, 0, static_cast<cudaStream_t>(stream)>>>(
                        w_oihw, Cout, Cin, K, pad, py, px, KH2, KW2, pad2, rows_pad, k_pad, reinterpret_cast<T*>(out)));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_pack_dw_weight(const float* w, int C, int k, int flip, float* out, cabinet_stream_t stream) {
    CAB_REQUIRE(w && out && C > 0 && k > 0, "pack_dw_weight: bad arguments");
    pack_dw_weight_kernel<<<static_cast<unsigned>(cab_ceil_div(C * k * k, 256)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        w, C, k * k, flip, out);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_im2col_nchw(const float* x, int N, int Cin, int H, int W, int k, int stride, int pad, void* out,
                                   long long ld, cabinet_stream_t stream) {
    return cabinet_im2col_nchw_dt(x, N, Cin, H, W, k, stride, pad, out, ld, CABINET_BF16, stream);
}

extern "C" int cabinet_im2col_nchw_dt(const float* x, int N, int Cin, int H, int W, int k, int stride, int pad, void* out,
                                      long long ld, int out_dtype, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("im2col_nchw", out_dtype, CAB_DT_BF16 | CAB_DT_F16);
    CAB_REQUIRE(x && out && N >= 0 && Cin > 0 && H > 0 && W > 0 && k > 0 && stride > 0 && ld >= static_cast<long long>(Cin) * k * k &&
                    ld % 8 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0,
                "im2col_nchw: bad arguments (ld must be a multiple of 8 >= Cin*k*k, out 16-byte aligned)");
    if (N == 0) return CABINET_OK;
    const int OH = (H + 2 * pad - k) / stride + 1, OW = (W + 2 * pad - k) / stride + 1;
    const long long total = static_cast<long long>(N) * OH * OW;
    CAB_REQUIRE(total * (ld / 8) < (1LL << 31), "im2col_nchw: too many pixels");
    const size_t smem = (static_cast<size_t>(Cin) * k * (IM2COL_PX * stride + k - stride) + static_cast<size_t>(ld)) * 4;
    const int segs = (OW + IM2COL_PX - 1) / IM2COL_PX;
    CAB_DISPATCH_DT_HALF(out_dtype, T,
        if (smem <= 48 * 1024 && static_cast<long long>(N) * OH * segs < (1LL << 31))
            im2col_nchw_row_kernel<T><<<static_cast<unsigned>(static_cast<long long>(N) * OH * segs), 256, smem, static_cast<cudaStream_t>(stream)>>>(
                x, Cin, H, W, k, stride, pad, OH, OW, reinterpret_cast<T*>(out), static_cast<int>(ld), segs);
        else
            im2col_nchw_kernel<T><<<ew_grid(total * (ld / 8)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
                x, N, Cin, H, W, k, stride, pad, OH, OW, reinterpret_cast<T*>(out), static_cast<int>(ld)));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_embed_filter(float* w_small, int Cout, int Cin, int k, int K, float* w_big, long long ld_big,
                                    int extract_add, cabinet_stream_t stream) {
    CAB_REQUIRE(w_small && w_big && Cout > 0 && Cin > 0 && k > 0 && K >= k && (K - k) % 2 == 0 && ld_big >= static_cast<long long>(Cin) * K * K,
                "embed_filter: bad arguments");
    const int total = Cout * Cin * k * k;
    embed_filter_kernel<<<static_cast<unsigned>(cab_ceil_div(total, 256)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        w_small, Cout, Cin, k, K, w_big, static_cast<int>(ld_big), extract_add);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" long long cabinet_train_scratch_floats(long long M, int C, int nq) {
    long long rpb;
    const int nb = red_blocks(std::max<long long>(M, 1), &rpb);
    return static_cast<long long>(nb) * nq * C;
}

// bench / debug: bit 6 of cabinet_debug_flags keeps the line-walking weight-gradient kernel (A/B against the row-tap one),
// bit 7 the register-fed BatchNorm reductions
static int cabinet_debug_flags_value() {
    const int f = cabinet_debug_flags(0);
    cabinet_debug_flags(f);
    return f;
}

// Plan of the shared-memory-staged reductions: dense bf16 rows, at least 2 MB, at most three blocks per SM
struct RtPlan {
    bool ok;
    int nb, chunk_rows;
    long long rpb;
};
static RtPlan rt_plan(int dtype, long long M, int C, bool dense, int nsrc, int nb_max) {
    RtPlan p = {false, 0, 0, 0};
    if ((dtype != CABINET_BF16 && dtype != CABINET_F16) || !dense || C % 8 != 0 || C / 8 > RED_THREADS || M * C < (1LL << 20) || (cabinet_debug_flags_value() & 128))
        return p;
    const int lanes = RED_THREADS / (C / 8);
    p.chunk_rows = (RT_STAGE_BYTES / nsrc) / (C * 2) / lanes * lanes;
    if (p.chunk_rows < lanes) return p;
    const long long nb = std::min<long long>(nb_max, 148 * (nsrc == 2 ? 2 : 3));  // resident blocks per SM: 91 / 53 registers
    p.rpb = cab_ceil_div(cab_ceil_div(M, nb), p.chunk_rows) * p.chunk_rows;  // whole chunks per block
    p.nb = static_cast<int>(cab_ceil_div(M, p.rpb));
    p.ok = true;
    return p;
}

extern "C" int cabinet_bn_train_stats(const void* x, long long ldx, int dtype, long long M, int C, const float* gamma,
                                      const float* beta, float eps, float momentum, float* running_mean,
                                      float* running_var, float* stats, float* scratch, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("bn_train_stats", dtype, CAB_DT_ALL);
    CAB_REQUIRE(x && stats && scratch && M > 0 && C > 0 && ldx >= C, "bn_train_stats: bad arguments");
    long long rpb;
    const int nb = red_blocks(M, &rpb);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int V = dtype == CABINET_F32 ? 4 : 8;
    const RtPlan tp = rt_plan(dtype, M, C, ldx == C && al16(x), 1, nb);
    if (tp.ok) {
        static bool attr_done = false;
        if (!attr_done) {
            CAB_CUDA(cudaFuncSetAttribute(bn_stats_tma_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, RT_STAGES * RT_STAGE_BYTES));
            CAB_CUDA(cudaFuncSetAttribute(bn_stats_tma_kernel<f16>, cudaFuncAttributeMaxDynamicSharedMemorySize, RT_STAGES * RT_STAGE_BYTES));
            attr_done = true;
        }
        CAB_DISPATCH_DT_HALF(dtype, T,
                        bn_stats_tma_kernel<T><<<tp.nb, RT_THREADS, RT_STAGES * RT_STAGE_BYTES, s>>>(reinterpret_cast<const T*>(x), M, C, tp.rpb,
                                                                                                     tp.chunk_rows, scratch);
                        CAB_LAUNCH_CHECK();
                        bn_finalize_kernel<T><<<static_cast<unsigned>(cab_ceil_div(C, 4)), 128, 0, s>>>(scratch, tp.nb, M, C, reinterpret_cast<const T*>(x),
                                                                                                      gamma, beta, eps, momentum, running_mean,
                                                                                                      running_var, stats));
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    if (C % V == 0 && ldx % V == 0 && al16(x)) {
        CAB_DISPATCH_DT(dtype, T,
                bn_stats_v_kernel<T><<<nb, RED_THREADS, red_smem_v<T>(2), s>>>(reinterpret_cast<const T*>(x), ldx, M, C, rpb, scratch));
    } else {
        CAB_DISPATCH_DT(dtype, T,
                bn_stats_kernel<T><<<nb, RED_THREADS, RED_SMEM, s>>>(reinterpret_cast<const T*>(x), ldx, M, C, rpb, scratch));
    }
    CAB_LAUNCH_CHECK();
    const unsigned g = static_cast<unsigned>(cab_ceil_div(C, 4));  // 4 warps = 4 channels per block
    CAB_DISPATCH_DT(dtype, T,
                bn_finalize_kernel<T><<<g, 128, 0, s>>>(scratch, nb, M, C, reinterpret_cast<const T*>(x), gamma, beta, eps,
                                                       momentum, running_mean, running_var, stats));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_affine_act(const void* z, long long ldz, int z_dtype, const float* scale, const float* shift,
                                  const float* gate, float gate_plus, const void* res, long long ldres, void* y,
                                  long long ldy, int y_dtype, long long M, long long HW, int C, int act,
                                  cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("affine_act", z_dtype, CAB_DT_ALL);
    CAB_REQUIRE_DTYPE("affine_act", y_dtype, CAB_DT_ALL);
    CAB_REQUIRE(z && y && M >= 0 && C > 0 && HW > 0 && (!scale || shift), "affine_act: bad arguments");
    if (M == 0) return CABINET_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (C % 8 == 0 && C <= 2048 && ldz % 8 == 0 && ldy % 8 == 0 && (!res || ldres % 8 == 0) && al16(z) && al16(y) && al16(res)) {
        const int lanes = 256 / (C / 8);
        const unsigned gv = row_grid(M, lanes);
#define CAB_AAV(TZ, TY)                                                                                                  \
    affine_act_v_kernel<TZ, TY><<<gv, 256, 0, s>>>(reinterpret_cast<const TZ*>(z), ldz, scale, shift, gate, gate_plus,   \
                                                   reinterpret_cast<const TY*>(res), ldres, reinterpret_cast<TY*>(y), ldy, \
                                                   M, HW, C, act)
        CAB_DISPATCH_DT_PAIR(z_dtype, y_dtype, CAB_AAV);
#undef CAB_AAV
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    const unsigned g = ew_grid(M * C);
#define CAB_AA(TZ, TY)                                                                                                \
    affine_act_kernel<TZ, TY><<<g, 256, 0, s>>>(reinterpret_cast<const TZ*>(z), ldz, scale, shift, gate, gate_plus,   \
                                                reinterpret_cast<const TY*>(res), ldres, reinterpret_cast<TY*>(y), ldy, \
                                                M, HW, C, act)
    CAB_DISPATCH_DT_PAIR(z_dtype, y_dtype, CAB_AA);
#undef CAB_AA
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_bn_train_backward(const void* dy, long long lddy, const void* z, long long ldz, int dtype,
                                         const float* stats, int act, float* dgamma, float* dbeta, void* dz,
                                         long long lddz, long long M, int C, int accumulate, float* scratch,
                                         cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("bn_train_backward", dtype, CAB_DT_ALL);
    CAB_REQUIRE(dy && z && stats && dz && scratch && M > 0 && C > 0, "bn_train_backward: bad arguments");
    long long rpb;
    const int nb = red_blocks(M, &rpb);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    float* coef = scratch + static_cast<long long>(nb) * 2 * C;
    const int V = dtype == CABINET_F32 ? 4 : 8;
    const bool vec = C % V == 0 && C / V <= 256 && lddy % V == 0 && ldz % V == 0 && lddz % V == 0 && al16(dy) && al16(z) && al16(dz);
    const RtPlan tp = rt_plan(dtype, M, C, vec && lddy == C && ldz == C, 2, nb);
    int nb_red = nb;
    if (tp.ok) {
        static bool attr_done = false;
        if (!attr_done) {
            CAB_CUDA(cudaFuncSetAttribute(bn_bwd_reduce_tma_kernel<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, RT_STAGES * RT_STAGE_BYTES));
            CAB_CUDA(cudaFuncSetAttribute(bn_bwd_reduce_tma_kernel<f16>, cudaFuncAttributeMaxDynamicSharedMemorySize, RT_STAGES * RT_STAGE_BYTES));
            attr_done = true;
        }
        CAB_DISPATCH_DT_HALF(dtype, T,
                        bn_bwd_reduce_tma_kernel<T><<<tp.nb, RT_THREADS, RT_STAGES * RT_STAGE_BYTES, s>>>(reinterpret_cast<const T*>(dy),
                                                                                                          reinterpret_cast<const T*>(z), stats, act, M, C,
                                                                                                          tp.rpb, tp.chunk_rows, scratch));
        nb_red = tp.nb;
    } else if (vec) {
        CAB_DISPATCH_DT(dtype, T,
                bn_bwd_reduce_v_kernel<T><<<nb, RED_THREADS, red_smem_v<T>(2), s>>>(reinterpret_cast<const T*>(dy), lddy,
                                                                                        reinterpret_cast<const T*>(z), ldz, stats, act, M, C, rpb, scratch));
    } else {
        CAB_DISPATCH_DT(dtype, T,
                bn_bwd_reduce_kernel<T><<<nb, RED_THREADS, RED_SMEM, s>>>(reinterpret_cast<const T*>(dy), lddy,
                                                                            reinterpret_cast<const T*>(z), ldz, stats, act, M, C, rpb, scratch));
    }
    CAB_LAUNCH_CHECK();
    bn_bwd_finalize_kernel<<<static_cast<unsigned>(cab_ceil_div(C, 4)), 128, 0, s>>>(scratch, nb_red, M, C, dgamma, dbeta, coef);
    CAB_LAUNCH_CHECK();
    if (vec) {
        const unsigned gv = row_grid(M, 256 / (C / V));
        CAB_DISPATCH_DT(dtype, T,
                bn_bwd_apply_v_kernel<T><<<gv, 256, 0, s>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(z), ldz,
                                                               stats, coef, act, reinterpret_cast<T*>(dz), lddz, M, C, accumulate));
    } else {
        const unsigned g = ew_grid(M * C);
        CAB_DISPATCH_DT(dtype, T,
                bn_bwd_apply_kernel<T><<<g, 256, 0, s>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(z), ldz,
                                                            stats, coef, act, reinterpret_cast<T*>(dz), lddz, M, C, accumulate));
    }
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_bn_frozen_stats(const float* gamma, const float* beta, const float* running_mean,
                                       const float* running_var, float eps, int C, float* stats, cabinet_stream_t stream) {
    CAB_REQUIRE(running_mean && running_var && stats && C > 0 && eps >= 0.f, "bn_frozen_stats: bad arguments");
    bn_frozen_stats_kernel<<<static_cast<unsigned>(cab_ceil_div(C, 256)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
            gamma, beta, running_mean, running_var, eps, C, stats);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_bn_frozen_backward(const void* dy, long long lddy, const void* z, long long ldz, int dtype,
                                          const float* stats, int act, float* dgamma, float* dbeta, void* dz,
                                          long long lddz, long long M, int C, int accumulate, float* scratch,
                                          cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("bn_frozen_backward", dtype, CAB_DT_ALL);
    const bool red = dgamma || dbeta;
    CAB_REQUIRE(dy && z && stats && (red || dz) && (!red || scratch) && M > 0 && C > 0 && lddy >= C && ldz >= C &&
                        (!dz || lddz >= C),
                "bn_frozen_backward: bad arguments");
    long long rpb;
    const int nb = red_blocks(M, &rpb);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int V = dtype == CABINET_F32 ? 4 : 8;
    const bool vec = C % V == 0 && C / V <= RED_THREADS && lddy % V == 0 && ldz % V == 0 && al16(dy) && al16(z) &&
                     (!dz || (lddz % V == 0 && al16(dz)));
#define CAB_FB(KERNEL, RED, GRID, SMEM)                                                                                  \
    CAB_DISPATCH_DT(dtype, T,                                                                                            \
                    KERNEL<T, RED><<<GRID, RED_THREADS, SMEM, s>>>(reinterpret_cast<const T*>(dy), lddy,                 \
                                                                   reinterpret_cast<const T*>(z), ldz, stats, act,       \
                                                                   reinterpret_cast<T*>(dz), lddz, M, C, accumulate, rpb, \
                                                                   scratch))
    if (red) {
        if (vec) {
            CAB_FB(bn_frozen_bwd_v_kernel, true, nb, red_smem_v<T>(2));
        } else {
            CAB_FB(bn_frozen_bwd_kernel, true, nb, RED_SMEM);
        }
        CAB_LAUNCH_CHECK();
        bn_bwd_finalize_kernel<<<static_cast<unsigned>(cab_ceil_div(C, 4)), 128, 0, s>>>(scratch, nb, M, C, dgamma, dbeta,
                                                                                          nullptr);
    } else if (vec) {
        CAB_FB(bn_frozen_bwd_v_kernel, false, row_grid(M, RED_THREADS / (C / V)), 0);
    } else {
        CAB_FB(bn_frozen_bwd_kernel, false, ew_grid(M * C), 0);
    }
#undef CAB_FB
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_gate_apply_backward(const void* dy, long long lddy, const void* v, long long ldv, int dtype,
                                           const float* s, float plus, const float* dm, float inv_hw, int act, void* dv,
                                           long long lddv, int N, long long HW, int C, int accumulate,
                                           cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("gate_apply_backward", dtype, CAB_DT_ALL);
    CAB_REQUIRE(dy && v && dv && N >= 0 && HW > 0 && C > 0, "gate_apply_backward: bad arguments");
    if (N == 0) return CABINET_OK;
    const long long M = static_cast<long long>(N) * HW;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int V = dtype == CABINET_F32 ? 4 : 8;
    if (C % V == 0 && C / V <= 256 && lddy % V == 0 && ldv % V == 0 && lddv % V == 0 && al16(dy) && al16(v) && al16(dv) && N <= 65535) {
        const int lanes = 256 / (C / V);
        const unsigned gx = static_cast<unsigned>(std::max<long long>(1, std::min<long long>(cab_ceil_div(HW, 4LL * lanes), 148LL * 16 / N + 1)));
        dim3 grid(gx, N);
        CAB_DISPATCH_DT(dtype, T,
                gate_bwd_apply_v_kernel<T><<<grid, 256, 0, st>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(v), ldv, s, plus, dm,
                                                                    inv_hw, act, reinterpret_cast<T*>(dv), lddv, HW, C, accumulate));
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    CAB_DISPATCH_DT(dtype, T,
                gate_bwd_apply_kernel<T><<<ew_grid(M * C), 256, 0, st>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(v), ldv, s, plus,
                                                                        dm, inv_hw, act, reinterpret_cast<T*>(dv), lddv, M, HW, C, accumulate));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_gate_scale_backward(const void* dy, long long lddy, const void* v, long long ldv, int dtype,
                                           const float* s, float plus, int act, float* ds, int N, long long HW, int C,
                                           float* scratch, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("gate_scale_backward", dtype, CAB_DT_ALL);
    CAB_REQUIRE(dy && v && s && ds && scratch && N > 0 && HW > 0 && C > 0 && N <= 65535, "gate_scale_backward: bad arguments");
    long long rpb;
    const int nb = red_blocks(HW, &rpb);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    dim3 grid(nb, N);
    const int V = dtype == CABINET_F32 ? 4 : 8;
    if (C % V == 0 && lddy % V == 0 && ldv % V == 0 && al16(dy) && al16(v)) {
        CAB_DISPATCH_DT(dtype, T,
                gate_bwd_reduce_v_kernel<T><<<grid, RED_THREADS, red_smem_v<T>(1), st>>>(reinterpret_cast<const T*>(dy), lddy,
                                                                                               reinterpret_cast<const T*>(v), ldv, s, plus, act, HW, C, rpb, scratch));
        CAB_LAUNCH_CHECK();
        sum_partials_kernel<<<dim3(static_cast<unsigned>(cab_ceil_div(C, 128)), N), 128, 0, st>>>(scratch, nb, C, static_cast<long long>(nb) * C, ds,
                                                                                                   1.f, 0);
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    CAB_DISPATCH_DT(dtype, T,
                gate_bwd_reduce_kernel<T><<<grid, RED_THREADS, RED_SMEM, st>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(v), ldv,
                                                                              s, plus, act, HW, C, rpb, scratch));
    CAB_LAUNCH_CHECK();
    sum_partials_kernel<<<dim3(static_cast<unsigned>(cab_ceil_div(C, 128)), N), 128, 0, st>>>(scratch, nb, C, static_cast<long long>(nb) * C, ds,
                                                                                               1.f, 0);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_col_sum(const void* x, long long ldx, int dtype, long long M, int C, float* out, int accumulate,
                               float* scratch, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("col_sum", dtype, CAB_DT_ALL);
    CAB_REQUIRE(x && out && scratch && M > 0 && C > 0, "col_sum: bad arguments");
    long long rpb;
    const int nb = red_blocks(M, &rpb);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CAB_DISPATCH_DT(dtype, T,
                col_sum_kernel<T><<<nb, RED_THREADS, RED_SMEM, s>>>(reinterpret_cast<const T*>(x), ldx, M, C, rpb, scratch));
    CAB_LAUNCH_CHECK();
    sum_partials_kernel<<<dim3(static_cast<unsigned>(cab_ceil_div(C, 128)), 1), 128, 0, s>>>(scratch, nb, C, 0, out, 1.f, accumulate);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_conv_dgrad(const void* dy, long long lddy, int dtype, const void* w_packed, int w_dtype,
                                  long long w_sco, long long w_stap, void* dx, long long lddx, int N, int H, int W, int Cin,
                                  int Cout, int KH, int KW, int stride, int pad, int OH, int OW, int accumulate,
                                  cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("conv_dgrad", dtype, CAB_DT_ALL);
    CAB_REQUIRE_DTYPE("conv_dgrad", w_dtype, CAB_DT_ALL);
    CAB_REQUIRE(dy && w_packed && dx && N >= 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0 && stride >= 1, "conv_dgrad: bad arguments");
    if (N == 0) return CABINET_OK;
    DgradArgs a;
    a.dy = dy; a.lddy = lddy; a.w = w_packed; a.w_sco = w_sco; a.w_stap = w_stap; a.dx = dx; a.lddx = lddx;
    a.N = N; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.KH = KH; a.KW = KW; a.stride = stride; a.pad = pad;
    a.OH = OH; a.OW = OW; a.accumulate = accumulate;
    a.M = static_cast<long long>(N) * H * W;
    a.K = KH * KW * Cout;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool s2 = stride == 2;
    if (s2) a.M = static_cast<long long>(N) * ((H + 1) / 2) * ((W + 1) / 2);  // the largest parity class
    dim3 grid(static_cast<unsigned>(cab_ceil_div(a.M, GBM)), static_cast<unsigned>(cab_ceil_div(Cin, GBN)), s2 ? 4 : 1);
#define CAB_DG(T, TW)                                                      \
    do {                                                                   \
        if (s2) conv_dgrad_kernel<T, TW, true><<<grid, 256, 0, s>>>(a);    \
        else conv_dgrad_kernel<T, TW, false><<<grid, 256, 0, s>>>(a);      \
    } while (0)
    CAB_DISPATCH_DT_PAIR(dtype, w_dtype, CAB_DG);
#undef CAB_DG
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" long long cabinet_conv_wgrad_scratch_floats(int N, int OH, int OW, int Cin, int Cout, int KH, int KW) {
    const long long M = static_cast<long long>(N) * OH * OW;
    const long long tiles = cab_ceil_div(Cout, GBM) * cab_ceil_div(static_cast<long long>(KH) * KW * Cin, GBN);
    long long splits = std::max<long long>(1, std::min<long long>(cab_ceil_div(148LL * 4, tiles), cab_ceil_div(M, 256)));
    splits = std::min<long long>(splits, 512);
    return splits * Cout * KH * KW * Cin;
}

extern "C" int cabinet_conv_wgrad(const void* dy, long long lddy, int dtype, const void* x, int x_dtype, long long sxn,
                                  long long sxh, long long sxw, long long sxc, float* dw_oihw, int N, int H, int W, int Cin,
                                  int Cout, int KH, int KW, int stride, int pad, int OH, int OW, float* scratch,
                                  cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("conv_wgrad", dtype, CAB_DT_ALL);
    CAB_REQUIRE_DTYPE("conv_wgrad", x_dtype, CAB_DT_ALL);
    CAB_REQUIRE(dy && x && dw_oihw && scratch && N > 0 && Cin > 0 && Cout > 0, "conv_wgrad: bad arguments");
    WgradArgs a;
    a.dy = dy; a.lddy = lddy; a.x = x; a.sxn = sxn; a.sxh = sxh; a.sxw = sxw; a.sxc = sxc; a.partial = scratch;
    a.N = N; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.KH = KH; a.KW = KW; a.stride = stride; a.pad = pad;
    a.OH = OH; a.OW = OW;
    a.M = static_cast<long long>(N) * OH * OW;
    a.Kn = KH * KW * Cin;
    const long long total = static_cast<long long>(Cout) * a.Kn;
    const long long splits = cabinet_conv_wgrad_scratch_floats(N, OH, OW, Cin, Cout, KH, KW) / total;
    a.rows_per_split = cab_ceil_div(cab_ceil_div(a.M, splits), GBK) * GBK;
    const int nz = static_cast<int>(cab_ceil_div(a.M, a.rows_per_split));
    dim3 grid(static_cast<unsigned>(cab_ceil_div(Cout, GBM)), static_cast<unsigned>(cab_ceil_div(a.Kn, GBN)), nz);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
#define CAB_WG(T, TX) conv_wgrad_kernel<T, TX><<<grid, 256, 0, s>>>(a)
    CAB_DISPATCH_DT_PAIR(dtype, x_dtype, CAB_WG);
#undef CAB_WG
    CAB_LAUNCH_CHECK();
    wgrad_finalize_kernel<<<static_cast<unsigned>(cab_ceil_div(total, 256)), 256, 0, s>>>(scratch, nz, Cout, Cin, KH * KW, dw_oihw);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_dwconv_dgrad(const void* dy, long long lddy, int dtype, const float* w_packed, void* dx,
                                    long long lddx, int N, int H, int W, int C, int k, int stride, int OH, int OW,
                                    int accumulate, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("dwconv_dgrad", dtype, CAB_DT_ALL);
    CAB_REQUIRE(dy && w_packed && dx && C > 0 && (k == 3 || k == 5) && stride >= 1, "dwconv_dgrad: bad arguments");
    if (N == 0) return CABINET_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int V = dtype == CABINET_F32 ? 4 : 8;
    if (C % V == 0 && lddy % V == 0 && lddx % V == 0 && al16(dy) && al16(dx) && al16(w_packed) && C % 4 == 0 &&
        static_cast<long long>(N) * H * W * (C / V) < (1LL << 31)) {
        const long long tv = static_cast<long long>(N) * H * W * (C / V);
        if (stride == 2) {
            const unsigned g2 = static_cast<unsigned>(std::min<long long>(cab_ceil_div(tv, 256), 148LL * 32));
#define CAB_DG2(T, KK)                                                                                                          \
    dw_dgrad_s2_kernel<T, KK><<<g2, 256, 0, s>>>(reinterpret_cast<const T*>(dy), lddy, w_packed, reinterpret_cast<T*>(dx), lddx, N, H, W, \
                                                 C, OH, OW, accumulate)
            CAB_DISPATCH_DT(dtype, T, if (k == 3) CAB_DG2(T, 3); else CAB_DG2(T, 5));
#undef CAB_DG2
            CAB_LAUNCH_CHECK();
            return CABINET_OK;
        }
        CAB_DISPATCH_DT(dtype, T,
                dw_dgrad_v_kernel<T><<<ew_grid(tv), 256, 0, s>>>(reinterpret_cast<const T*>(dy), lddy, w_packed, reinterpret_cast<T*>(dx), lddx, N, H,
                                                                    W, C, k, stride, OH, OW, accumulate));
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    const long long total = static_cast<long long>(N) * H * W * C;
    CAB_DISPATCH_DT(dtype, T,
                dw_dgrad_kernel<T><<<ew_grid(total), 256, 0, s>>>(reinterpret_cast<const T*>(dy), lddy, w_packed, reinterpret_cast<T*>(dx), lddx, N, H, W,
                                                                 C, k, stride, OH, OW, accumulate));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_dwconv_wgrad(const void* dy, long long lddy, const void* x, long long ldx, int dtype, float* dw,
                                    int N, int H, int W, int C, int k, int stride, int OH, int OW, float* scratch,
                                    cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("dwconv_wgrad", dtype, CAB_DT_ALL);
    CAB_REQUIRE(dy && x && dw && scratch && N > 0 && C > 0 && (k == 3 || k == 5), "dwconv_wgrad: bad arguments");
    const long long M = static_cast<long long>(N) * OH * OW;
    CAB_REQUIRE(M < (1LL << 31), "dwconv_wgrad: too many pixels");
    long long rpb;
    const int nb = red_blocks(M, &rpb);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (C % 2 == 0 && lddy % 2 == 0 && ldx % 2 == 0 && (reinterpret_cast<uintptr_t>(dy) & 7) == 0 && (reinterpret_cast<uintptr_t>(x) & 7) == 0 &&
        (stride == 1 || stride == 2) && OW >= 8 && !(cabinet_debug_flags_value() & 64)) {
        // row-tap kernel.  Channel pairs per warp: the largest power of two <= 32 that pads the channel count by <= 12 %
        const int pairs = C / 2;
        int cw_log2 = 5;
        while (cw_log2 > 2 && (cab_ceil_div(pairs, 1 << cw_log2) << cw_log2) * 100 > pairs * 112) --cw_log2;
        const int cw = 1 << cw_log2, nsub = 32 / cw, ny = static_cast<int>(cab_ceil_div(pairs, cw));
        // segments: enough items per chunk column to keep ~5 blocks per SM busy twice over, >= 16 pixels each
        const long long n_lines = static_cast<long long>(N) * OH;
        const int want_bx = std::max(1, std::min<int>(nb, (148 * 5 + ny - 1) / ny));
        const long long want_items = 2LL * want_bx * DWR_SL * nsub;
        int nseg = static_cast<int>(std::max<long long>(1, std::min<long long>(OW / 16, cab_ceil_div(want_items, n_lines))));
        const int seg_len = static_cast<int>(cab_ceil_div(cab_ceil_div(OW, nseg), 4) * 4);
        nseg = (OW + seg_len - 1) / seg_len;
        const long long n_items = n_lines * nseg;
        const int bx = static_cast<int>(std::min<long long>(want_bx, cab_ceil_div(n_items, DWR_SL * nsub)));
        const int ipb = static_cast<int>(cab_ceil_div(cab_ceil_div(n_items, bx), DWR_SL * nsub) * DWR_SL * nsub);
        const int nbx = static_cast<int>(cab_ceil_div(n_items, ipb));  // <= bx <= nb: fits the scratch
        dim3 grid(nbx, ny);
#define CAB_DWR(T, KK, SS)                                                                                                \
    dw_wgrad_row_kernel<T, KK, SS><<<grid, 32 * KK * DWR_SL, 0, s>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(x), \
                                                                     ldx, H, W, C, OH, OW, static_cast<int>(n_items), nseg, seg_len, ipb, cw_log2, scratch)
#define CAB_DWR2(T)                                                                                 \
    do {                                                                                            \
        if (k == 3 && stride == 1) CAB_DWR(T, 3, 1); else if (k == 3) CAB_DWR(T, 3, 2);             \
        else if (stride == 1) CAB_DWR(T, 5, 1); else CAB_DWR(T, 5, 2);                              \
    } while (0)
        CAB_DISPATCH_DT(dtype, T, CAB_DWR2(T));
#undef CAB_DWR2
#undef CAB_DWR
        CAB_LAUNCH_CHECK();
        dw_wgrad_finalize_kernel<<<static_cast<unsigned>(cab_ceil_div(C * k * k, 8)), 256, 0, s>>>(scratch, nbx, C, k * k, dw);
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    if (C % 2 == 0 && lddy % 2 == 0 && ldx % 2 == 0 && (reinterpret_cast<uintptr_t>(dy) & 7) == 0 && (reinterpret_cast<uintptr_t>(x) & 7) == 0 &&
        (stride == 1 || stride == 2) && OW >= 8 &&
        cab_ceil_div(static_cast<long long>(N) * OH, 2LL * (RED_THREADS / std::min(RED_THREADS, C / 2))) <= nb) {
        // line walker: a block reduces 2 line segments per pixel lane; as many segments per line as the scratch (sized
        // for `nb` blocks of partial rows) allows, at least 8 pixels each
        const long long n_lines = static_cast<long long>(N) * OH;
        const int cwv = std::min(RED_THREADS, C / 2), lanes = RED_THREADS / cwv;
        const long long rpb2 = 2LL * lanes;
        int nseg = static_cast<int>(std::max<long long>(1, std::min<long long>(OW / 8, nb * rpb2 / n_lines)));
        const int seg_len = (OW + nseg - 1) / nseg;
        nseg = (OW + seg_len - 1) / seg_len;
        const long long n_items = n_lines * nseg;
        const int nb2 = static_cast<int>(cab_ceil_div(n_items, rpb2));
        const size_t smem2 = RED_THREADS * 2 * k * k * sizeof(float);
        static bool attr_done = false;
        if (!attr_done) {
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_line_kernel<float, 5, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_line_kernel<float, 5, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_line_kernel<bf16, 5, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_line_kernel<bf16, 5, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_line_kernel<f16, 5, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_line_kernel<f16, 5, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            attr_done = true;
        }
#define CAB_DWL(T, KK, SS)                                                                                                     \
    dw_wgrad_line_kernel<T, KK, SS><<<nb2, RED_THREADS, smem2, s>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(x), \
                                                                    ldx, H, W, C, OH, OW, n_items, nseg, seg_len, rpb2, scratch)
#define CAB_DWL2(T)                                                                                 \
    do {                                                                                            \
        if (k == 3 && stride == 1) CAB_DWL(T, 3, 1); else if (k == 3) CAB_DWL(T, 3, 2);             \
        else if (stride == 1) CAB_DWL(T, 5, 1); else CAB_DWL(T, 5, 2);                              \
    } while (0)
        CAB_DISPATCH_DT(dtype, T, CAB_DWL2(T));
#undef CAB_DWL2
#undef CAB_DWL
        CAB_LAUNCH_CHECK();
        dw_wgrad_finalize_kernel<<<static_cast<unsigned>(cab_ceil_div(C * k * k, 8)), 256, 0, s>>>(scratch, nb2, C, k * k, dw);
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    if (C % 2 == 0 && lddy % 2 == 0 && ldx % 2 == 0 && (reinterpret_cast<uintptr_t>(dy) & 7) == 0 && (reinterpret_cast<uintptr_t>(x) & 7) == 0) {
        const size_t smem2 = RED_THREADS * 2 * k * k * sizeof(float);
        static bool attr_done = false;
        if (!attr_done) {
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_v2_kernel<float, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_v2_kernel<bf16, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            CAB_CUDA(cudaFuncSetAttribute(dw_wgrad_v2_kernel<f16, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            attr_done = true;
        }
#define CAB_DWV(T, KK)                                                                                                       \
    dw_wgrad_v2_kernel<T, KK><<<nb, RED_THREADS, smem2, s>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(x), \
                                                            ldx, H, W, C, stride, OH, OW, M, rpb, scratch)
        CAB_DISPATCH_DT(dtype, T, if (k == 3) CAB_DWV(T, 3); else CAB_DWV(T, 5));
#undef CAB_DWV
        CAB_LAUNCH_CHECK();
        dw_wgrad_finalize_kernel<<<static_cast<unsigned>(cab_ceil_div(C * k * k, 8)), 256, 0, s>>>(scratch, nb, C, k * k, dw);
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    const size_t smem = RED_THREADS * k * k * sizeof(float);
#define CAB_DWW(T, KK)                                                                                                   \
    dw_wgrad_kernel<T, KK><<<nb, RED_THREADS, smem, s>>>(reinterpret_cast<const T*>(dy), lddy, reinterpret_cast<const T*>(x), \
                                                         ldx, H, W, C, stride, OH, OW, M, rpb, scratch)
    CAB_DISPATCH_DT(dtype, T, if (k == 3) CAB_DWW(T, 3); else CAB_DWW(T, 5));
#undef CAB_DWW
    CAB_LAUNCH_CHECK();
    dw_wgrad_finalize_kernel<<<static_cast<unsigned>(cab_ceil_div(C * k * k, 8)), 256, 0, s>>>(scratch, nb, C, k * k, dw);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_resample_sep(const void* in, int in_dtype, long long isn, long long isy, long long isx,
                                    long long isc, void* out, int out_dtype, long long osn, long long osy, long long osx,
                                    long long osc, int N, int OH, int OW, int C, const int* y_start, const int* y_index,
                                    const float* y_weight, const int* x_start, const int* x_index, const float* x_weight,
                                    int accumulate, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("resample_sep", in_dtype, CAB_DT_ALL);
    CAB_REQUIRE_DTYPE("resample_sep", out_dtype, CAB_DT_ALL);
    CAB_REQUIRE(in && out && y_start && y_index && y_weight && x_start && x_index && x_weight && OH > 0 && OW > 0 && C > 0,
                "resample_sep: bad arguments");
    if (N == 0) return CABINET_OK;
    const long long total = static_cast<long long>(N) * OH * OW * C;
    CAB_REQUIRE(total < (1LL << 31), "resample_sep: too many output elements");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    const int band = (accumulate >> 1) & 1;       // bit 1: planar input with many taps per output -> row-band kernel
    const int few_taps = (accumulate >> 2) & 1;   // bit 2: few taps per output (an upsample, the adjoint of a pool): the
    accumulate &= 1;                              //        8-channel vector kernel pays (with many taps it starves: 8x fewer threads)
    if (band && isx == 1 && static_cast<long long>(N) * C <= 65535) {
        // the input line length is not an argument: it is what the x operator indexes, i.e. the row pitch of a dense plane
        const int W_in = static_cast<int>(isy);
        CAB_REQUIRE(W_in > 0 && W_in * sizeof(float) <= 48 * 1024, "resample_sep: input line too long for the band kernel");
        dim3 grid(OH, N * C);
        const size_t smem = W_in * sizeof(float);
#define CAB_RB(TI, TO)                                                                                                       \
    resample_band_kernel<TI, TO><<<grid, 256, smem, s>>>(reinterpret_cast<const TI*>(in), isn, isy, isc, W_in,               \
                                                         reinterpret_cast<TO*>(out), osn, osy, osx, osc, C, OW, y_start, y_index, \
                                                         y_weight, x_start, x_index, x_weight, accumulate & 1, vec)
        const int vw = in_dtype == CABINET_F32 ? 4 : 8;  // columns per 16-byte load
        const int vec = (W_in % vw == 0 && isn % vw == 0 && isc % vw == 0 && al16(in)) ? 1 : 0;
        CAB_DISPATCH_DT_PAIR(in_dtype, out_dtype, CAB_RB);
#undef CAB_RB
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
    if (few_taps && isc == 1 && osc == 1 && C % 8 == 0 && isn % 8 == 0 && isy % 8 == 0 && isx % 8 == 0 && osn % 8 == 0 && osy % 8 == 0 &&
        osx % 8 == 0 && al16(in) && al16(out)) {
#define CAB_RSV(TI, TO)                                                                                                        \
    resample_sep_v_kernel<TI, TO><<<ew_grid(total / 8), 256, 0, s>>>(reinterpret_cast<const TI*>(in), isn, isy, isx,             \
                                                                     reinterpret_cast<TO*>(out), osn, osy, osx, N, OH, OW, C,    \
                                                                     y_start, y_index, y_weight, x_start, x_index, x_weight, accumulate)
        CAB_DISPATCH_DT_PAIR(in_dtype, out_dtype, CAB_RSV);
#undef CAB_RSV
        CAB_LAUNCH_CHECK();
        return CABINET_OK;
    }
#define CAB_RS(TI, TO)                                                                                                   \
    resample_sep_kernel<TI, TO><<<ew_grid(total), 256, 0, s>>>(reinterpret_cast<const TI*>(in), isn, isy, isx, isc,      \
                                                               reinterpret_cast<TO*>(out), osn, osy, osx, osc, N, OH, OW, C, \
                                                               y_start, y_index, y_weight, x_start, x_index, x_weight, accumulate)
    CAB_DISPATCH_DT_PAIR(in_dtype, out_dtype, CAB_RS);
#undef CAB_RS
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_softmax_backward(const float* p, const float* dp, float* ds, long long rows, int cols, float alpha,
                                        cabinet_stream_t stream) {
    CAB_REQUIRE(p && dp && ds && cols > 0, "softmax_backward: bad arguments");
    if (rows == 0) return CABINET_OK;
    softmax_bwd_kernel<<<static_cast<unsigned>(cab_ceil_div(rows, 8)), 256, 0, static_cast<cudaStream_t>(stream)>>>(p, dp, ds, rows, cols, alpha);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_attn_softmax(const float* s, float scale, float* p, void* p_bf16, long long rows, int cols,
                                    cabinet_stream_t stream) {
    return cabinet_attn_softmax_dt(s, scale, p, p_bf16, rows, cols, CABINET_BF16, stream);
}

extern "C" int cabinet_attn_softmax_dt(const float* s, float scale, float* p, void* p_half, long long rows, int cols,
                                       int op_dtype, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("attn_softmax", op_dtype, CAB_DT_BF16 | CAB_DT_F16);
    CAB_REQUIRE(s && p && p_half && cols > 0, "attn_softmax: bad arguments");
    if (rows == 0) return CABINET_OK;
    CAB_DISPATCH_DT_HALF(op_dtype, T,
                    attn_softmax_kernel<T><<<static_cast<unsigned>(cab_ceil_div(rows, 8)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
                        s, scale, p, reinterpret_cast<T*>(p_half), rows, cols));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_attn_softmax_backward(const float* p, const float* dp, void* ds_bf16, long long rows, int cols,
                                             float alpha, cabinet_stream_t stream) {
    return cabinet_attn_softmax_backward_dt(p, dp, ds_bf16, rows, cols, alpha, CABINET_BF16, stream);
}

extern "C" int cabinet_attn_softmax_backward_dt(const float* p, const float* dp, void* ds_half, long long rows, int cols,
                                                float alpha, int op_dtype, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("attn_softmax_backward", op_dtype, CAB_DT_BF16 | CAB_DT_F16);
    CAB_REQUIRE(p && dp && ds_half && cols > 0, "attn_softmax_backward: bad arguments");
    if (rows == 0) return CABINET_OK;
    CAB_DISPATCH_DT_HALF(op_dtype, T,
                    attn_softmax_bwd_kernel<T><<<static_cast<unsigned>(cab_ceil_div(rows, 8)), 256, 0, static_cast<cudaStream_t>(stream)>>>(
                        p, dp, reinterpret_cast<T*>(ds_half), rows, cols, alpha));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_transpose_tokens(const void* x, long long ldx, void* out, int N, int L, int C,
                                        cabinet_stream_t stream) {
    return cabinet_transpose_tokens_dt(x, ldx, out, N, L, C, CABINET_BF16, stream);
}

extern "C" int cabinet_transpose_tokens_dt(const void* x, long long ldx, void* out, int N, int L, int C, int op_dtype,
                                           cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("transpose_tokens", op_dtype, CAB_DT_BF16 | CAB_DT_F16);
    CAB_REQUIRE(x && out && N >= 0 && L > 0 && C > 0 && ldx >= C && N <= 65535, "transpose_tokens: bad arguments");
    if (N == 0) return CABINET_OK;
    dim3 grid(static_cast<unsigned>(cab_ceil_div(L, 32)), static_cast<unsigned>(cab_ceil_div(C, 32)), N);
    CAB_DISPATCH_DT_HALF(op_dtype, T,
                    transpose_tokens_kernel<T><<<grid, 256, 0, static_cast<cudaStream_t>(stream)>>>(reinterpret_cast<const T*>(x), ldx,
                                                                                                  reinterpret_cast<T*>(out), L, C));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_cab_combine_backward(const void* dout, long long ldo, const void* g, const void* x, const void* r,
                                            const float* gamma, int dtype, void* dg, void* dx, void* dr, float* dgamma,
                                            long long n_pixels, int C, int accumulate_dx, float* scratch,
                                            cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("cab_combine_backward", dtype, CAB_DT_ALL);
    CAB_REQUIRE(dout && g && x && r && gamma && dg && dx && dr && dgamma && scratch && n_pixels > 0 && C > 0,
                "cab_combine_backward: bad arguments");
    long long rpb;
    const int nb = red_blocks(n_pixels, &rpb);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CAB_DISPATCH_DT(dtype, T,
                cab_combine_bwd_kernel<T><<<nb, RED_THREADS, RED_SMEM, s>>>(reinterpret_cast<const T*>(dout), ldo, reinterpret_cast<const T*>(g),
                                                                          reinterpret_cast<const T*>(x), reinterpret_cast<const T*>(r), gamma,
                                                                          reinterpret_cast<T*>(dg), reinterpret_cast<T*>(dx), reinterpret_cast<T*>(dr),
                                                                          n_pixels, C, rpb, scratch, accumulate_dx));
    CAB_LAUNCH_CHECK();
    sum_all_kernel<<<1, 256, 0, s>>>(scratch, static_cast<long long>(nb) * C, dgamma);
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_add(const void* a, long long lda, const void* b, long long ldb, void* out, long long ldo, int dtype,
                           long long M, int C, cabinet_stream_t stream) {
    CAB_REQUIRE_DTYPE("add", dtype, CAB_DT_ALL);
    CAB_REQUIRE(a && b && out && C > 0, "add: bad arguments");
    if (M == 0) return CABINET_OK;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    CAB_DISPATCH_DT(dtype, T,
                add_kernel<T><<<ew_grid(M * C), 256, 0, s>>>(reinterpret_cast<const T*>(a), lda, reinterpret_cast<const T*>(b), ldb,
                                                            reinterpret_cast<T*>(out), ldo, M, C));
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}

extern "C" int cabinet_gate_mlp_backward(const float* mean, float mean_scale, const float* w1, const float* w2, const float* hidden,
                                         const float* s, const float* ds, int gate, int N, int C, int J, float* dw1,
                                         float* db1, float* dw2, float* db2, float* dmean, float* scratch,
                                         cabinet_stream_t stream) {
    CAB_REQUIRE(mean && w1 && w2 && hidden && s && ds && dw1 && dw2 && dmean && scratch && N > 0 && C > 0 && J > 0,
                "gate_mlp_backward: bad arguments");
    float* da2 = scratch;
    float* da1 = scratch + static_cast<long long>(N) * C;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int sizes[5] = {N * C, C * J, N * J, J * C, N * C};
    for (int ph = 0; ph < 5; ++ph) {
        if (ph == 2 || ph == 4)
            gate_bwd_dot_kernel<<<static_cast<unsigned>(cab_ceil_div(sizes[ph], 8)), 256, 0, st>>>(ph, N, C, J, w1, w2, hidden, da2, da1, dmean);
        else
            gate_bwd_phase_kernel<<<static_cast<unsigned>(cab_ceil_div(sizes[ph], 128)), 128, 0, st>>>(ph, N, C, J, gate, mean_scale, mean, w1, w2, hidden, s, ds, da2, da1,
                                                                                                        dw1, db1, dw2, db2, dmean);
        CAB_LAUNCH_CHECK();
    }
    return CABINET_OK;
}
