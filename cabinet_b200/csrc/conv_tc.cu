// Implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05.mma, fp32 accumulators in TMEM), bf16 NHWC (fp16 for
// the plain convolution forms of the fp16 training mode: same tiles, only the operand format bits and the map type change).
//
//   D[128 pixels x block_n couts] = sum over (tap, 64-channel block)  A_tap[128 x 64] * W_tap[block_n x 64]^T
//
// * A tiles are fetched by TMA straight from the NHWC activation: the 128 output pixels of a tile are a TH x TW
//   patch of one image, each filter tap is ONE 4-D box load {64 ch, TW, TH, 1} at a shifted coordinate, and the
//   zero padding of the convolution is TMA's out-of-bounds zero fill (negative / past-the-end coordinates).
//   Stride-2 convolutions use one tensor map per input parity (py, px): map(py,px)[h][w] = x[2h+py][2w+px], so a
//   tap is again a plain shifted box.  1x1 convolutions view the tensor as [N*H*W][C] (no tile waste).
// * W tiles ([Cout_pad][taps*Cin_pad] bf16, K-major, BN folded) come through a 2-D tensor map; when the whole
//   weight matrix is <= 64 KB (every memory-bound 1x1 layer) it is loaded ONCE per CTA and stays resident.
// * Both land in 128-byte-swizzled shared memory = the canonical K-major SWIZZLE_128B UMMA layout, so MMA
//   descriptors are the stage base + 32 B per K=16 step.
// * PERSISTENT and pipelined across tiles: one CTA per SM walks tiles blockIdx.x, +gridDim.x, ...; the smem ring
//   never drains between tiles and two TMEM accumulator stages let the MMAs of tile i+1 run under the epilogue of
//   tile i.  Warp roles (320 threads): warp 0 = TMA producer, warp 1 = TMEM allocator + MMA issuer,
//   warps 2-5 / 6-9 = two epilogue warpgroups (even / odd tiles).
// * Epilogue: tcgen05.ld -> +bias -> act -> (+residual) -> bf16 -> 128B-swizzled smem staging -> TMA store
//   (full-line writes, image-border and channel clipping by the tensor map); fp32 outputs (class logits) are
//   stored directly.
#include <stdlib.h>

#include <type_traits>

#include "tc_common.cuh"

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // bf16 elements: 128 bytes = one swizzle row
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;
constexpr int C_STAGE_BYTES = BLOCK_M * 128;  // one [128 rows x 64 ch] bf16 store box
constexpr int MAX_STAGES = 8;
constexpr int NUM_THREADS = 320;
constexpr int PRO_THREADS = 256;                 // A-operand prologue warps (PRO variants): 8 warps, 4 chunks of a row each
// (16 warps were measured: 10 % faster without a residual, 30-40 % slower with one -- 72 registers per thread spill the epilogue)
constexpr int PRO_CHUNKS = 8 * 128 / PRO_THREADS;  // 16-byte chunks of its A row per prologue thread
constexpr int B_RESIDENT_MAX = 80 * 1024;  // sb.conv2 (3x3, 64 -> 64: 72 KB) stays resident
constexpr int SMEM_LIMIT = 220 * 1024;

struct TcConvParams {
    int OH, OW, Cin, Cout;
    int KW, stride, pad;
    int TW, TH, tiles_w, tiles_h;
    int cin_blocks, num_k_blocks;
    int block_n, n_tiles, num_tiles, tmem_cols, stages, b_resident;
    int act, y_dtype, debug;
    int act_cols;             // the activation applies to output channels < act_cols only (merged q|k|v projection)
    int reverse;              // walk the tiles back to front (start on the part of the input its producer left in L2)
    int b_per_image;          // weights differ per image (cabinet_conv_tc_imgw): B tiles are fetched with the tile's image index
    int c_bufs;               // store staging buffers per epilogue warpgroup: 2, or 1 when a tile is a single 64-column group
    int a_act, hw;            // A-operand prologue: x <- act(x * a_scale[image][channel]); hw = pixels per image
    const float* a_scale;     // [N][Cin] fp32 or nullptr
    const float* bias;
    const void* res;          // residual: the operand type (bf16 / fp16)
    long long ldres;
    void* y;
    long long ldy;
    // UP4 epilogue: v += bilinear(up -> output size)[pixel] before the activation.  up: fp32 [N][up_h][up_w][Cout];
    // img_h x img_w = true output size of one image (the tile walk of a 1x1 conv is flat over all pixels)
    const float* up;
    int up_h, up_w, img_h, img_w, up_flat;
};

__device__ long long g_dbg[8192];  // clock64 stamps of CTA 0's MMA warp when debug bit 8 is set

struct TileCoord {
    int img, oh0, ow0, n0;
};

__device__ __forceinline__ TileCoord decode_tile(const TcConvParams& p, int tile) {
    TileCoord c;
    if (p.reverse) tile = p.num_tiles - 1 - tile;
    const int m = tile / p.n_tiles;
    c.n0 = (tile - m * p.n_tiles) * p.block_n;
    const int tw_i = m % p.tiles_w;
    const int t = m / p.tiles_w;
    c.ow0 = tw_i * p.TW;
    c.oh0 = (t % p.tiles_h) * p.TH;
    c.img = t / p.tiles_h;
    return c;
}

template <int ACT, bool HAS_RES, bool OUT_F32, bool PRO, bool UP4 = false, typename T = bf16>
__global__ void __launch_bounds__(PRO ? NUM_THREADS + PRO_THREADS : NUM_THREADS, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
               const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmA3,
               const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmY,
               const TcConvParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[MAX_STAGES];
    __shared__ __align__(8) uint64_t empty_bar[MAX_STAGES];
    __shared__ __align__(8) uint64_t ready_bar[MAX_STAGES];  // PRO: A tile transformed in place, MMA may read it
    __shared__ __align__(8) uint64_t acc_full[2], acc_empty[2], bres_bar;
    __shared__ uint32_t tmem_base_smem;
    __shared__ __align__(16) float s_bias[2][256];  // per epilogue warpgroup: bias slice of its current cout tile
    __shared__ __align__(16) float s_ascale[PRO ? 1024 : 4];  // PRO: the A-operand scale row of the tile's image

    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int b_stage_bytes = p.block_n * BLOCK_K * 2;
    uint8_t* sC = smem;                                   // 2 x c_bufs x 16 KB store staging (c_bufs per epilogue warpgroup)
    uint8_t* sA = sC + 2 * p.c_bufs * C_STAGE_BYTES;      // ring: stages x 16 KB
    uint8_t* sB = sA + p.stages * A_STAGE_BYTES;          // ring (stages x b_stage) or resident (num_k_blocks x b_stage)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        tc::prefetch_tmap(&tmA0);
        tc::prefetch_tmap(&tmB);
        tc::prefetch_tmap(&tmY);
        for (int s = 0; s < p.stages; ++s) {
            tc::mbar_init(&full_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
            tc::mbar_init(&ready_bar[s], PRO_THREADS / 32);
        }
        for (int s = 0; s < 2; ++s) {
            tc::mbar_init(&acc_full[s], 1);
            tc::mbar_init(&acc_empty[s], 4);
        }
        tc::mbar_init(&bres_bar, 1);
        tc::mbar_fence_init();
        tc::fence_proxy_async();
    }
    if (warp == 1) tc::tmem_alloc(&tmem_base_smem, p.tmem_cols);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = tmem_base_smem;
    const int acc_stride = p.tmem_cols >> 1;  // columns per accumulator stage (>= block_n)

    if (warp == 0) {
        if (lane == 0) {
            // ================= TMA producer =================
            if (p.b_resident) {
                tc::mbar_expect_tx(&bres_bar, p.num_k_blocks * b_stage_bytes);
                for (int kb = 0; kb < p.num_k_blocks; ++kb)
                    tc::tma_load_3d(sB + kb * b_stage_bytes, &tmB, &bres_bar, kb * BLOCK_K, 0, 0);
            }
            const uint32_t tx_bytes = A_STAGE_BYTES + (p.b_resident ? 0 : b_stage_bytes);
            int s = 0;
            uint32_t ph = 0;
            for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
                const TileCoord tcd = decode_tile(p, tile);
                int tap = 0, cb = 0, ky = 0, kx = 0;
                for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                    tc::mbar_wait(&empty_bar[s], ph ^ 1);
                    if (p.debug & 4) {
                        tc::mbar_arrive(&full_bar[s]);
                    } else {
                    tc::mbar_expect_tx(&full_bar[s], tx_bytes);
                    const int ty = ky - p.pad, tx = kx - p.pad;
                    const CUtensorMap* map = &tmA0;
                    int dy = ty, dx = tx;
                    if (p.stride == 2) {
                        const int py = ty & 1, px = tx & 1;
                        dy = (ty - py) >> 1;
                        dx = (tx - px) >> 1;
                        const int id = py * 2 + px;
                        map = id == 0 ? &tmA0 : id == 1 ? &tmA1 : id == 2 ? &tmA2 : &tmA3;
                    }
                    tc::tma_load_4d(sA + s * A_STAGE_BYTES, map, &full_bar[s], cb * BLOCK_K, tcd.ow0 + dx, tcd.oh0 + dy,
                                    tcd.img);
                    if (!p.b_resident) {
                        // per-image weights: spatial tiles carry the image index, flat (1x1) tiles cover 128 consecutive
                        // pixels of ONE image (the host checks H * W % 128 == 0)
                        const int bimg = !p.b_per_image ? 0 : (p.tiles_h == 1 && p.OH == 1 ? tcd.ow0 / p.hw : tcd.img);
                        tc::tma_load_3d(sB + s * b_stage_bytes, &tmB, &full_bar[s], kb * BLOCK_K, tcd.n0, bimg);
                    }
                    }
                    if (++cb == p.cin_blocks) {
                        cb = 0;
                        ++tap;
                        if (++kx == p.KW) { kx = 0; ++ky; }
                    }
                    if (++s == p.stages) { s = 0; ph ^= 1; }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ================= MMA issuer: warp-uniform control flow, one elected lane issues =================
        const uint32_t leader = tc::elect_one();
        const uint32_t idesc = tc::make_idesc<T>(BLOCK_M, p.block_n);
        const uint64_t a_desc0 = tc::make_desc_sw128(tc::smem_u32(sA));
        const uint64_t b_desc0 = tc::make_desc_sw128(tc::smem_u32(sB));
        const uint32_t a_step = A_STAGE_BYTES >> 4, b_step = static_cast<uint32_t>(b_stage_bytes) >> 4;
        if (p.b_resident) tc::mbar_wait(&bres_bar, 0);
        int g = 0, it = 0, s = 0;
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x, ++it) {
            const int acc = it & 1;
            tc::mbar_wait(&acc_empty[acc], ((it >> 1) & 1) ^ 1);
            tc::tc_fence_after();
            const uint32_t d = tmem + acc * acc_stride;
            int cb = 0;
            for (int kb = 0; kb < p.num_k_blocks; ++kb, ++g) {
                const bool rec = (p.debug & 8) && blockIdx.x == 0 && g < 2000 && lane == 0;
                if (rec) g_dbg[4 * g + 0] = clock64();
                tc::mbar_wait(PRO ? &ready_bar[s] : &full_bar[s], ph);
                tc::tc_fence_after();
                if (rec) g_dbg[4 * g + 1] = clock64();
                const int ksteps = min(BLOCK_K / 16, (p.Cin - cb * BLOCK_K + 15) / 16);  // skip all-zero K tails
                const uint64_t a_desc = a_desc0 + static_cast<uint64_t>(s * a_step);
                const uint64_t b_desc = b_desc0 + static_cast<uint64_t>((p.b_resident ? kb : s) * b_step);
                tc::umma_bf16_if(leader, d, a_desc, b_desc, idesc, kb != 0 ? 1u : 0u);
                if (ksteps > 1) tc::umma_bf16_if(leader, d, a_desc + 2, b_desc + 2, idesc, 1u);
                if (ksteps > 2) tc::umma_bf16_if(leader, d, a_desc + 4, b_desc + 4, idesc, 1u);
                if (ksteps > 3) tc::umma_bf16_if(leader, d, a_desc + 6, b_desc + 6, idesc, 1u);
                if (rec) g_dbg[4 * g + 2] = clock64();
                tc::umma_commit_if(leader, &empty_bar[s]);  // ring slot is free once these MMAs have read it
                if (rec) g_dbg[4 * g + 3] = clock64();
                if (++cb == p.cin_blocks) cb = 0;
                if (++s == p.stages) { s = 0; ph ^= 1; }
            }
            tc::umma_commit_if(leader, &acc_full[acc]);     // accumulator of this tile complete
        }
        __syncwarp();
    } else if (PRO && warp >= 10) {
        // ================= A-operand prologue (SE): x <- act(x * scale[image][channel]) in place =================
        // reference: src/models/mobilenetv3.py:83 (x * y) followed by the activation at :143, fused in front of the
        // project 1x1 so the depthwise output is read from HBM once and never rewritten.
        // 8 warps: thread = (A row = pixel of the tile, half of its eight 16-byte chunks).  All shared / global loads of
        // a stage are issued before the first dependent instruction.
        const int r = (threadIdx.x - NUM_THREADS) & 127, half = (threadIdx.x - NUM_THREADS) >> 7;  // half = part of the row
        int s = 0;
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
            const TileCoord tcd = decode_tile(p, tile);
            // image of this row: flat tiles index pixels of all images, spatial tiles belong to one image
            const long long pixrow = static_cast<long long>(tcd.ow0) + r;
            const int img = p.tiles_h == 1 && p.OH == 1 ? static_cast<int>(min(pixrow, static_cast<long long>(p.OW) - 1) / p.hw)
                                                        : tcd.img;
            const float* sc = p.a_scale + static_cast<long long>(img) * p.Cin;
            // The scale row is read once per tile into shared memory when all rows of the tile belong to one image
            // (always, except flat tiles that straddle an image boundary): per-stage __ldg's of it were the dominant
            // stall of this path (long scoreboard), 11 stages x 8 loads per thread and tile.
            bool sc_smem = p.Cin <= 1024 && (p.Cin & 3) == 0;
            if (p.tiles_h == 1 && p.OH == 1) {
                const long long last = min(static_cast<long long>(tcd.ow0) + 127, static_cast<long long>(p.OW) - 1);
                sc_smem = sc_smem && (tcd.ow0 / p.hw == last / p.hw);
            }
            tc::named_bar_sync(3, PRO_THREADS);  // the previous tile's stages no longer read s_ascale
            if (sc_smem) {
                const float* sc0 = p.a_scale + static_cast<long long>(p.tiles_h == 1 && p.OH == 1 ? tcd.ow0 / p.hw : tcd.img) * p.Cin;
                for (int i = threadIdx.x - NUM_THREADS; i < (p.Cin >> 2); i += PRO_THREADS)
                    reinterpret_cast<float4*>(s_ascale)[i] = __ldg(reinterpret_cast<const float4*>(sc0) + i);
            }
            tc::named_bar_sync(3, PRO_THREADS);
            int cb = 0;
            for (int kb = 0; kb < p.num_k_blocks; ++kb) {
                tc::mbar_wait(&full_bar[s], ph);
                const uint32_t rowa = tc::smem_u32(sA) + s * A_STAGE_BYTES + r * 128;
                {
                uint4 raw[PRO_CHUNKS];
                float4 s0[PRO_CHUNKS], s1[PRO_CHUNKS];
#pragma unroll
                for (int jj = 0; jj < PRO_CHUNKS; ++jj) {
                    // walk LOGICAL chunks: the 8 rows of a quarter-warp then touch 8 different physical chunks
                    // (conflict-free; walking physical chunks is an 8-way bank conflict) and share the scale address
                    const int l = half * PRO_CHUNKS + jj;
                    const int j = l ^ (r & 7);
                    const int c = cb * BLOCK_K + (l << 3);
                    if (c < p.Cin) {
                        raw[jj] = tc::lds128(rowa + (j << 4));
                        if (sc_smem) {
                            s0[jj] = *reinterpret_cast<const float4*>(s_ascale + c);
                            s1[jj] = *reinterpret_cast<const float4*>(s_ascale + c + 4);
                        } else {
                            s0[jj] = __ldg(reinterpret_cast<const float4*>(sc + c));
                            s1[jj] = __ldg(reinterpret_cast<const float4*>(sc + c) + 1);
                        }
                    }
                }
#pragma unroll
                for (int jj = 0; jj < PRO_CHUNKS; ++jj) {
                    const int l = half * PRO_CHUNKS + jj;
                    const int j = l ^ (r & 7);
                    const int c = cb * BLOCK_K + (l << 3);
                    if (c < p.Cin) {
                        Vec16<T> v;
                        v.raw = raw[jj];
                        float f[8];
                        v.unpack(f);
                        f[0] *= s0[jj].x; f[1] *= s0[jj].y; f[2] *= s0[jj].z; f[3] *= s0[jj].w;
                        f[4] *= s1[jj].x; f[5] *= s1[jj].y; f[6] *= s1[jj].z; f[7] *= s1[jj].w;
                        cab_act_vec<8>(f, p.a_act);
                        v.pack(f);
                        tc::sts128(rowa + (j << 4), v.raw);
                    }
                }
                }
                tc::fence_proxy_async();
                __syncwarp();
                if (lane == 0) tc::mbar_arrive(&ready_bar[s]);
                if (++cb == p.cin_blocks) cb = 0;
                if (++s == p.stages) { s = 0; ph ^= 1; }
            }
        }
    } else {
        // ================= epilogue warpgroup e (tiles it = e, e+2, ...) =================
        const int e = (warp - 2) >> 2;
        const int q = warp & 3;  // TMEM lane quarter this warp may access
        const int row = q * 32 + lane;
        const int gtid = threadIdx.x - 64 - e * 128;  // 0..127 inside the warpgroup
        const bool leader = gtid == 0;
        uint8_t* myC = sC + e * p.c_bufs * C_STAGE_BYTES;
        float* myBias = s_bias[e];
        uint32_t store_seq = 0;
        int it = e, bias_n0 = -1;
        for (int tile = blockIdx.x + e * gridDim.x; tile < p.num_tiles; tile += 2 * gridDim.x, it += 2) {
            const TileCoord tcd = decode_tile(p, tile);
            const int oh = tcd.oh0 + row / p.TW, ow = tcd.ow0 + row % p.TW;
            const bool valid = oh < p.OH && ow < p.OW;
            const long long pix = (static_cast<long long>(tcd.img) * p.OH + oh) * p.OW + ow;
            [[maybe_unused]] const float* up00 = nullptr;
            [[maybe_unused]] long long up_dx = 0, up_dy = 0;
            [[maybe_unused]] float uw00 = 0.f, uw01 = 0.f, uw10 = 0.f, uw11 = 0.f;
            if constexpr (UP4) {
                if (valid) {  // bilinear taps of this thread's pixel in the low-resolution map (align_corners=False)
                    int un = tcd.img, uoh = oh, uow = ow;
                    if (p.up_flat) {
                        un = static_cast<int>(pix / p.hw);
                        const int rem = static_cast<int>(pix - static_cast<long long>(un) * p.hw);
                        uoh = rem / p.img_w;
                        uow = rem - uoh * p.img_w;
                    }
                    int y0, y1, x0, x1;
                    float wy, wx;
                    cab_bilinear_tap(uoh, static_cast<float>(p.up_h) / static_cast<float>(p.img_h), p.up_h, y0, y1, wy);
                    cab_bilinear_tap(uow, static_cast<float>(p.up_w) / static_cast<float>(p.img_w), p.up_w, x0, x1, wx);
                    up00 = p.up + ((static_cast<long long>(un) * p.up_h + y0) * p.up_w + x0) * p.Cout;
                    up_dx = static_cast<long long>(x1 - x0) * p.Cout;
                    up_dy = static_cast<long long>(y1 - y0) * p.up_w * p.Cout;
                    uw00 = (1.f - wy) * (1.f - wx); uw01 = (1.f - wy) * wx; uw10 = wy * (1.f - wx); uw11 = wy * wx;
                }
            }
            if (tcd.n0 != bias_n0) {  // (re)load this cout tile's bias slice, zero padded
                tc::named_bar_sync(1 + e, 128);  // everyone is done reading the previous slice
                for (int i = gtid; i < p.block_n; i += 128) myBias[i] = (tcd.n0 + i < p.Cout) ? __ldg(p.bias + tcd.n0 + i) : 0.f;
                bias_n0 = tcd.n0;
                tc::named_bar_sync(1 + e, 128);
            }
            tc::mbar_wait(&acc_full[e], (it >> 1) & 1);
            tc::tc_fence_after();
            const uint32_t taddr = tmem + e * acc_stride + (static_cast<uint32_t>(q * 32) << 16);
            const int ngroups = (p.block_n + 63) >> 6;
            for (int grp = 0; grp < ngroups; ++grp) {
                uint8_t* buf = myC + (p.c_bufs == 2 ? (store_seq & 1) : 0) * C_STAGE_BYTES;
                const int nch = min(4, (p.block_n - grp * 64) >> 4);  // 16-column chunks in this 64-column group
                // issue all TMEM loads of the group, then one wait: 64 independent values per thread
                uint32_t r[64];
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (c < nch) tc::tmem_ld16(taddr + grp * 64 + c * 16, r + 16 * c);
                tc::tmem_ld_wait();
                if (grp == ngroups - 1) {
                    // all TMEM reads of this accumulator stage are done: hand it back to the MMA warp
                    tc::tc_fence_before();
                    __syncwarp();
                    if (lane == 0) tc::mbar_arrive(&acc_empty[e]);
                }
                if constexpr (!OUT_F32) {
                    // the TMA store that used this staging buffer two groups ago must have finished reading it
                    if (leader) {
                        if (p.c_bufs == 2) tc::bulk_wait_read<1>();
                        else tc::bulk_wait_read<0>();  // single buffer: its previous store (two tiles ago) must be done
                    }
                    tc::named_bar_sync(1 + e, 128);
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (c >= nch) break;
                    const int c0 = grp * 64 + c * 16;
                    const int co0 = tcd.n0 + c0;
                    float v[16];
#pragma unroll
                    for (int j4 = 0; j4 < 4; ++j4) {
                        const float4 b = *reinterpret_cast<const float4*>(myBias + c0 + 4 * j4);
                        v[4 * j4 + 0] = __uint_as_float(r[16 * c + 4 * j4 + 0]) + b.x;
                        v[4 * j4 + 1] = __uint_as_float(r[16 * c + 4 * j4 + 1]) + b.y;
                        v[4 * j4 + 2] = __uint_as_float(r[16 * c + 4 * j4 + 2]) + b.z;
                        v[4 * j4 + 3] = __uint_as_float(r[16 * c + 4 * j4 + 3]) + b.w;
                    }
                    if constexpr (UP4) {
                        if (valid && co0 + 16 <= p.Cout) {
                            const float* t = up00 + co0;
#pragma unroll
                            for (int j4 = 0; j4 < 4; ++j4) {
                                const float4 a = __ldg(reinterpret_cast<const float4*>(t) + j4);
                                const float4 b = __ldg(reinterpret_cast<const float4*>(t + up_dx) + j4);
                                const float4 c2 = __ldg(reinterpret_cast<const float4*>(t + up_dy) + j4);
                                const float4 d = __ldg(reinterpret_cast<const float4*>(t + up_dy + up_dx) + j4);
                                v[4 * j4 + 0] += uw00 * a.x + uw01 * b.x + uw10 * c2.x + uw11 * d.x;
                                v[4 * j4 + 1] += uw00 * a.y + uw01 * b.y + uw10 * c2.y + uw11 * d.y;
                                v[4 * j4 + 2] += uw00 * a.z + uw01 * b.z + uw10 * c2.z + uw11 * d.z;
                                v[4 * j4 + 3] += uw00 * a.w + uw01 * b.w + uw10 * c2.w + uw11 * d.w;
                            }
                        }
                    }
                    constexpr bool RELU_ON_CVT = ACT == CABINET_ACT_RELU && !HAS_RES && !OUT_F32;  // cvt.rn.relu.{bf16,f16}x2
                    const bool do_act = co0 < p.act_cols;  // uniform per 16-column chunk (act_cols % 16 == 0)
                    if constexpr (ACT == CABINET_ACT_RELU && !RELU_ON_CVT) {
                        if (do_act) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
                        }
                    } else if constexpr (ACT == CABINET_ACT_HSWISH) {
                        if (do_act) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) v[j] *= __saturatef(fmaf(v[j], 1.f / 6.f, 0.5f));  // relu6(v+3)/6
                        }
                    }
                    if constexpr (HAS_RES) {
                        if (valid && co0 < p.Cout) {
                            const T* rp = reinterpret_cast<const T*>(p.res) + pix * p.ldres + co0;
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                if (co0 + 8 * h + 8 <= p.Cout) {
                                    Vec16<T> rv;
                                    rv.load(rp + 8 * h);
                                    float rf[8];
                                    rv.unpack(rf);
#pragma unroll
                                    for (int j = 0; j < 8; ++j) v[8 * h + j] += rf[j];
                                } else {
                                    for (int j = 0; j < 8; ++j)
                                        if (co0 + 8 * h + j < p.Cout) v[8 * h + j] += to_f32<T>(rp[8 * h + j]);
                                }
                            }
                        }
                    }
                    if constexpr (!OUT_F32) {
                        Vec16<T> o0, o1;
                        if (RELU_ON_CVT && do_act) {
                            // never .satfinite: an fp16 overflow stays inf (a loss-scale overflow must reach the gradients)
                            uint32_t w[8];
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                if constexpr (std::is_same<T, f16>::value)
                                    asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(w[j]) : "f"(v[2 * j + 1]), "f"(v[2 * j]));
                                else
                                    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(w[j]) : "f"(v[2 * j + 1]), "f"(v[2 * j]));
                            }
                            o0.raw = make_uint4(w[0], w[1], w[2], w[3]);
                            o1.raw = make_uint4(w[4], w[5], w[6], w[7]);
                        } else {
                            o0.pack(v);
                            o1.pack(v + 8);
                        }
                        const uint32_t rowa = tc::smem_u32(buf) + row * 128;
                        tc::sts128(rowa + (((2 * c) ^ (row & 7)) << 4), o0.raw);
                        tc::sts128(rowa + (((2 * c + 1) ^ (row & 7)) << 4), o1.raw);
                    } else if (valid) {
                        float* yp = reinterpret_cast<float*>(p.y) + pix * p.ldy + co0;
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            if (co0 + j < p.Cout) yp[j] = v[j];
                    }
                }
                if constexpr (!OUT_F32) {
                    tc::fence_proxy_async();
                    tc::named_bar_sync(1 + e, 128);
                    if (leader && !(p.debug & 1)) {
                        tc::tma_store_4d(&tmY, buf, tcd.n0 + grp * 64, tcd.ow0, tcd.oh0, tcd.img);
                        tc::bulk_commit();
                    }
                    ++store_seq;
                }
            }
        }
        if (leader) tc::bulk_wait_read<0>();  // smem must outlive the reads; global visibility comes with grid completion
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem, p.tmem_cols);
    }
}

int g_debug = 0;

}  // namespace

cab_encode_tiled_fn cab_get_encode_tiled() {
    static cab_encode_tiled_fn fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<cab_encode_tiled_fn>(sym);
    }
    return fn;
}

int cab_make_tmap_2b(CUtensorMap* map, int elem_dtype, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_bytes, const uint32_t* box, CUtensorMapL2promotion promo,
                     CUtensorMapSwizzle swizzle) {
    CAB_REQUIRE_DTYPE("tensor map", elem_dtype, CAB_DT_BF16 | CAB_DT_F16);
    cab_encode_tiled_fn enc = cab_get_encode_tiled();
    if (!enc) {
        cabinet_set_error("cuTensorMapEncodeTiled is unavailable (driver too old or no driver)");
        return CABINET_ERR_CUDA;
    }
    cuuint64_t gdim[5], gstr[4];
    cuuint32_t bdim[5], estr[5];
    for (int i = 0; i < rank; ++i) {
        gdim[i] = dims[i];
        bdim[i] = box[i];
        estr[i] = 1;
        if (i > 0) gstr[i - 1] = strides_bytes[i - 1];
    }
    CUresult r = enc(map, elem_dtype == CABINET_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), gdim, gstr, bdim, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, promo, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        cabinet_set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d dims %llu,%llu,%llu,%llu box %u,%u,%u,%u)",
                          static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
                          (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0), box[0],
                          rank > 1 ? box[1] : 0, rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
        return CABINET_ERR_CUDA;
    }
    return CABINET_OK;
}

extern "C" int cabinet_debug_read(long long* host_out, int n) {
    CAB_CUDA(cudaMemcpyFromSymbol(host_out, g_dbg, sizeof(long long) * n));
    return CABINET_OK;
}

extern "C" int cabinet_debug_flags(int flags) {
    const int old = g_debug;
    g_debug = flags;
    return old;
}

static int conv_tc_impl(const void* x, long long ldx, int N, int H, int W, int Cin, const float* a_scale, int a_act,
                        const void* w_packed, long long w_image_stride, int Cout, int KH, int KW, int stride, int pad,
                        const float* bias, const void* res, long long ldres, void* y, int y_dtype, long long ldy,
                        int OH, int OW, int act, int op_dtype, cabinet_stream_t stream, int act_cols = 1 << 30,
                        const float* up = nullptr, int up_h = 0, int up_w = 0, long long y_sw = 1, long long y_sh = 0,
                        long long y_sn = 0);

extern "C" int cabinet_conv_tc_view(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed,
                                    int Cout, int KH, int KW, int pad, const float* bias, void* y, long long ldy, int OH,
                                    int OW, long long y_sw, long long y_sh, long long y_sn, cabinet_stream_t stream) {
    return cabinet_conv_tc_view_dt(x, ldx, N, H, W, Cin, w_packed, Cout, KH, KW, pad, bias, y, ldy, OH, OW, y_sw, y_sh, y_sn,
                                   CABINET_BF16, stream);
}

extern "C" int cabinet_conv_tc_view_dt(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed,
                                       int Cout, int KH, int KW, int pad, const float* bias, void* y, long long ldy, int OH,
                                       int OW, long long y_sw, long long y_sh, long long y_sn, int op_dtype,
                                       cabinet_stream_t stream) {
    return conv_tc_impl(x, ldx, N, H, W, Cin, nullptr, CABINET_ACT_NONE, w_packed, 0, Cout, KH, KW, 1, pad, bias, nullptr, 0,
                        y, op_dtype, ldy, OH, OW, CABINET_ACT_NONE, op_dtype, stream, 1 << 30, nullptr, 0, 0, y_sw, y_sh, y_sn);
}

extern "C" int cabinet_conv_tc_se(const void* x, long long ldx, int N, int H, int W, int Cin, const float* a_scale,
                                  int a_act, const void* w_packed, int Cout, int KH, int KW, int stride, int pad,
                                  const float* bias, const void* res, long long ldres, void* y, int y_dtype,
                                  long long ldy, int OH, int OW, int act, cabinet_stream_t stream) {
    return conv_tc_impl(x, ldx, N, H, W, Cin, a_scale, a_act, w_packed, 0, Cout, KH, KW, stride, pad, bias, res, ldres, y,
                        y_dtype, ldy, OH, OW, act, CABINET_BF16, stream);
}

extern "C" int cabinet_conv_tc_imgw(const void* x, long long ldx, int N, int H, int W, int Cin,
                                    const void* w_packed_per_image, long long w_image_stride, int Cout, int KH, int KW,
                                    int stride, int pad, const float* bias, const void* res, long long ldres, void* y,
                                    int y_dtype, long long ldy, int OH, int OW, int act, cabinet_stream_t stream) {
    return cabinet_conv_tc_imgw_dt(x, ldx, N, H, W, Cin, w_packed_per_image, w_image_stride, Cout, KH, KW, stride, pad, bias,
                                   res, ldres, y, y_dtype, ldy, OH, OW, act, CABINET_BF16, stream);
}

extern "C" int cabinet_conv_tc_imgw_dt(const void* x, long long ldx, int N, int H, int W, int Cin,
                                       const void* w_packed_per_image, long long w_image_stride, int Cout, int KH, int KW,
                                       int stride, int pad, const float* bias, const void* res, long long ldres, void* y,
                                       int y_dtype, long long ldy, int OH, int OW, int act, int op_dtype,
                                       cabinet_stream_t stream) {
    CAB_REQUIRE(w_image_stride > 0 && w_image_stride % 8 == 0, "conv_tc_imgw: weight image stride must be a positive multiple of 8");
    CAB_REQUIRE(!(KH == 1 && KW == 1 && stride == 1 && pad == 0) || (static_cast<long long>(H) * W) % 128 == 0,
                "conv_tc_imgw: a 1x1 convolution needs H * W %% 128 == 0 (a 128-pixel tile must not straddle two images)");
    return conv_tc_impl(x, ldx, N, H, W, Cin, nullptr, CABINET_ACT_NONE, w_packed_per_image, w_image_stride, Cout, KH, KW,
                        stride, pad, bias, res, ldres, y, y_dtype, ldy, OH, OW, act, op_dtype, stream);
}

extern "C" int cabinet_conv_tc_split_act(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed,
                                         int Cout, int KH, int KW, int stride, int pad, const float* bias, void* y,
                                         int y_dtype, long long ldy, int OH, int OW, int act, int act_cols,
                                         cabinet_stream_t stream) {
    CAB_REQUIRE(act_cols >= 0 && act_cols % 16 == 0, "conv_tc_split_act: act_cols must be a multiple of 16");
    return conv_tc_impl(x, ldx, N, H, W, Cin, nullptr, CABINET_ACT_NONE, w_packed, 0, Cout, KH, KW, stride, pad, bias,
                        nullptr, 0, y, y_dtype, ldy, OH, OW, act, CABINET_BF16, stream, act_cols);
}

extern "C" int cabinet_conv_tc(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed,
                               int Cout, int KH, int KW, int stride, int pad, const float* bias, const void* res,
                               long long ldres, void* y, int y_dtype, long long ldy, int OH, int OW, int act,
                               cabinet_stream_t stream) {
    return cabinet_conv_tc_dt(x, ldx, N, H, W, Cin, w_packed, Cout, KH, KW, stride, pad, bias, res, ldres, y, y_dtype, ldy,
                              OH, OW, act, CABINET_BF16, stream);
}

extern "C" int cabinet_conv_tc_dt(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed,
                                  int Cout, int KH, int KW, int stride, int pad, const float* bias, const void* res,
                                  long long ldres, void* y, int y_dtype, long long ldy, int OH, int OW, int act, int op_dtype,
                                  cabinet_stream_t stream) {
    return conv_tc_impl(x, ldx, N, H, W, Cin, nullptr, CABINET_ACT_NONE, w_packed, 0, Cout, KH, KW, stride, pad, bias, res,
                        ldres, y, y_dtype, ldy, OH, OW, act, op_dtype, stream);
}

extern "C" int cabinet_conv_tc_up(const void* x, long long ldx, int N, int H, int W, int Cin, const void* w_packed,
                                  int Cout, int KH, int KW, int stride, int pad, const float* bias, const float* up,
                                  int up_h, int up_w, void* y, long long ldy, int OH, int OW, int act,
                                  cabinet_stream_t stream) {
    CAB_REQUIRE(up != nullptr, "conv_tc_up: null low-resolution map");
    return conv_tc_impl(x, ldx, N, H, W, Cin, nullptr, CABINET_ACT_NONE, w_packed, 0, Cout, KH, KW, stride, pad, bias,
                        nullptr, 0, y, CABINET_BF16, ldy, OH, OW, act, CABINET_BF16, stream, 1 << 30, up, up_h, up_w);
}

static int conv_tc_impl(const void* x, long long ldx, int N, int H, int W, int Cin, const float* a_scale, int a_act,
                        const void* w_packed, long long w_image_stride, int Cout, int KH, int KW, int stride, int pad,
                        const float* bias, const void* res, long long ldres, void* y, int y_dtype, long long ldy,
                        int OH, int OW, int act, int op_dtype, cabinet_stream_t stream, int act_cols, const float* up, int up_h,
                        int up_w, long long y_sw, long long y_sh, long long y_sn) {
    // y_sw / y_sh / y_sn (pixels): the output is a strided VIEW (pixel, row, image pitch) of a larger NHWC tensor -- e.g.
    // one input-parity class of the data gradient of a stride-2 convolution.  Defaults: a dense [N][OH][OW] tensor.
    // op_dtype: the 2-byte type of x, w_packed, res and a 2-byte y (bf16, or fp16 for the plain convolution forms)
    CAB_REQUIRE_DTYPE("conv_tc", op_dtype, CAB_DT_BF16 | CAB_DT_F16);
    CAB_REQUIRE_DTYPE("conv_tc (output)", y_dtype, CAB_DT_F32 | (1 << op_dtype));
    CAB_REQUIRE(op_dtype == CABINET_BF16 || (!a_scale && !up), "conv_tc: the prologue / upsample epilogues are built for bf16");
    CAB_REQUIRE(x && w_packed && bias && y, "conv_tc: null pointer");
    const bool out_view = y_sw != 1 || y_sh != 0 || y_sn != 0;
    CAB_REQUIRE(!out_view || (y_dtype == op_dtype && !res && !up && y_sw >= 1 && y_sh >= OW && y_sn >= OH),
                "conv_tc: a strided output view needs a 2-byte output and no residual");
    const int reverse = (act & CABINET_CONV_REVERSE_TILES) ? 1 : 0;
    act &= ~CABINET_CONV_REVERSE_TILES;
    CAB_REQUIRE(!up || (up_h > 0 && up_w > 0 && Cout % 16 == 0 && (reinterpret_cast<uintptr_t>(up) & 15) == 0 && !res &&
                        !a_scale && y_dtype == CABINET_BF16 && w_image_stride == 0),
                "conv_tc_up: the upsample-add epilogue needs Cout %% 16 == 0, an aligned fp32 map, bf16 output, no residual");
    CAB_REQUIRE(!a_scale || (Cin % 8 == 0 && (reinterpret_cast<uintptr_t>(a_scale) & 15) == 0),
                "conv_tc: the A-operand scale needs Cin %% 8 == 0 and a 16-byte aligned pointer");
    CAB_REQUIRE(N >= 0 && H > 0 && W > 0 && Cin > 0 && Cout > 0 && KH > 0 && KW > 0 && OH > 0 && OW > 0,
                "conv_tc: bad sizes");
    CAB_REQUIRE(stride == 1 || stride == 2, "conv_tc: stride must be 1 or 2");
    CAB_REQUIRE(stride == 1 || (H >= 2 && W >= 2), "conv_tc: stride-2 needs H, W >= 2");
    CAB_REQUIRE(ldx % 8 == 0 && ldx >= Cin && (reinterpret_cast<uintptr_t>(x) & 15) == 0,
                "conv_tc: input needs 16-byte aligned pixels (ldx %% 8 == 0)");
    CAB_REQUIRE(ldy >= Cout && (y_dtype == CABINET_F32 || (ldy % 8 == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0)),
                "conv_tc: a 2-byte output needs 16-byte aligned pixels");
    CAB_REQUIRE(!res || (ldres % 8 == 0 && (reinterpret_cast<uintptr_t>(res) & 15) == 0), "conv_tc: residual alignment");
    CAB_REQUIRE((reinterpret_cast<uintptr_t>(w_packed) & 15) == 0, "conv_tc: weight alignment");
    if (N == 0) return CABINET_OK;

    TcConvParams p;
    const bool flat = KH == 1 && KW == 1 && stride == 1 && pad == 0 && !out_view;
    const int taps = KH * KW;
    p.Cin = Cin; p.Cout = Cout; p.KW = KW; p.stride = stride; p.pad = pad;
    p.cin_blocks = (Cin + BLOCK_K - 1) / BLOCK_K;
    p.num_k_blocks = taps * p.cin_blocks;
    const int n16 = ((Cout + 15) / 16) * 16;
    // one cout tile when it fits an accumulator stage (<= 256 columns), else 256-wide tiles (a multiple of the
    // 64-channel store box, so the boxes of neighbouring tiles never overlap; the tail is clipped by the map)
    p.n_tiles = (n16 + 255) / 256;
    p.block_n = p.n_tiles == 1 ? n16 : 256;
    p.tmem_cols = 32;
    while (p.tmem_cols < 2 * p.block_n) p.tmem_cols *= 2;
    const int b_stage_bytes = p.block_n * BLOCK_K * 2;
    p.act_cols = act_cols;
    p.reverse = reverse;
    p.b_per_image = w_image_stride > 0 ? 1 : 0;
    p.b_resident = (!p.b_per_image && p.n_tiles == 1 && p.num_k_blocks * b_stage_bytes <= B_RESIDENT_MAX) ? 1 : 0;
    p.c_bufs = (y_dtype != CABINET_F32 && p.block_n > 64) ? 2 : 1;
    const int fixed = 2 * p.c_bufs * C_STAGE_BYTES + (p.b_resident ? p.num_k_blocks * b_stage_bytes : 0) + 1024;
    const int stage_bytes = A_STAGE_BYTES + (p.b_resident ? 0 : b_stage_bytes);
    // experiment hook: CAB_SMEM_CAP_KB caps the dynamic smem of kernels whose accumulators need <= 256 TMEM columns, so
    // that two CTAs (e.g. from two streams) can share an SM
    static const int cap_kb = getenv("CAB_SMEM_CAP_KB") ? atoi(getenv("CAB_SMEM_CAP_KB")) : 0;
    const int limit = (cap_kb > 0 && p.tmem_cols <= 256) ? std::max(cap_kb * 1024, fixed + 2 * stage_bytes) : SMEM_LIMIT;
    // the prologue variants keep a 4 KB scale row in static shared memory: leave room for it under the 227 KB CTA limit
    p.stages = std::max(2, std::min(MAX_STAGES, (std::min(limit, SMEM_LIMIT) - (a_scale ? 4096 : 0) - fixed) / stage_bytes));
    p.act = act; p.y_dtype = y_dtype; p.bias = bias; p.res = res; p.ldres = ldres;
    p.y = y; p.ldy = ldy; p.debug = g_debug;
    p.a_scale = a_scale; p.a_act = a_act; p.hw = H * W;
    p.up = up; p.up_h = up_h; p.up_w = up_w; p.img_h = OH; p.img_w = OW; p.up_flat = 0;

    CUtensorMap tmA[4], tmB, tmY;
    const uint64_t es = 2;
    int Ng = N;
    if (flat) {
        const long long P = static_cast<long long>(N) * H * W;
        CAB_REQUIRE(P < (1LL << 31), "conv_tc: too many pixels");
        Ng = 1; p.OH = 1; p.OW = static_cast<int>(P); p.up_flat = 1;
        p.TW = BLOCK_M; p.TH = 1; p.tiles_w = static_cast<int>(cab_ceil_div(P, BLOCK_M)); p.tiles_h = 1;
        const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)P, 1, 1};
        const uint64_t strides[3] = {(uint64_t)ldx * es, (uint64_t)ldx * es * P, (uint64_t)ldx * es * P};
        const uint32_t box[4] = {BLOCK_K, BLOCK_M, 1, 1};
        int rc = cab_make_tmap_2b(&tmA[0], op_dtype, x, 4, dims, strides, box);
        if (rc) return rc;
        tmA[1] = tmA[2] = tmA[3] = tmA[0];
    } else {
        p.OH = OH; p.OW = OW;
        // pick the TH x TW = 128 patch shape that wastes the fewest pixels (ties: wider)
        long long best = -1;
        for (int tw = 128; tw >= 4; tw >>= 1) {
            const int th = BLOCK_M / tw;
            const long long cover = cab_ceil_div(OW, tw) * tw * cab_ceil_div(OH, th) * th;
            if (best < 0 || cover < best) { best = cover; p.TW = tw; p.TH = th; }
        }
        p.tiles_w = static_cast<int>(cab_ceil_div(OW, p.TW));
        p.tiles_h = static_cast<int>(cab_ceil_div(OH, p.TH));
        const uint32_t box[4] = {BLOCK_K, (uint32_t)p.TW, (uint32_t)p.TH, 1};
        const uint16_t* xb = reinterpret_cast<const uint16_t*>(x);  // 2-byte elements of either type
        for (int py = 0; py < stride; ++py)
            for (int px = 0; px < stride; ++px) {
                const uint64_t dims[4] = {(uint64_t)Cin, (uint64_t)((W - px + stride - 1) / stride),
                                          (uint64_t)((H - py + stride - 1) / stride), (uint64_t)N};
                const uint64_t strides[3] = {(uint64_t)ldx * es * stride, (uint64_t)ldx * es * W * stride,
                                             (uint64_t)ldx * es * W * H};
                int rc = cab_make_tmap_2b(&tmA[py * stride + px], op_dtype, xb + (static_cast<long long>(py) * W + px) * ldx, 4,
                                            dims, strides, box);
                if (rc) return rc;
            }
        if (stride == 1) tmA[1] = tmA[2] = tmA[3] = tmA[0];
    }
    {
        const uint64_t ktot = static_cast<uint64_t>(taps) * p.cin_blocks * BLOCK_K;
        CAB_REQUIRE(!p.b_per_image || static_cast<uint64_t>(w_image_stride) >= ktot * n16, "conv_tc_imgw: weight image stride too small");
        const uint64_t dims[3] = {ktot, (uint64_t)n16, (uint64_t)(p.b_per_image ? N : 1)};
        const uint64_t strides[2] = {ktot * es, (p.b_per_image ? static_cast<uint64_t>(w_image_stride) : ktot * n16) * es};
        const uint32_t box[3] = {BLOCK_K, (uint32_t)p.block_n, 1};
        int rc = cab_make_tmap_2b(&tmB, op_dtype, w_packed, 3, dims, strides, box, CU_TENSOR_MAP_L2_PROMOTION_L2_256B);
        if (rc) return rc;
    }
    if (y_dtype != CABINET_F32) {
        // store map: {Cout (true extent: clips padded / foreign channels), OW, OH, N}, 64-channel boxes
        const uint64_t dims[4] = {(uint64_t)Cout, (uint64_t)p.OW, (uint64_t)p.OH, (uint64_t)Ng};
        const uint64_t strides[3] = {(uint64_t)ldy * es * (uint64_t)y_sw, (uint64_t)ldy * es * (uint64_t)(y_sh ? y_sh : p.OW),
                                     (uint64_t)ldy * es * (uint64_t)(y_sn ? y_sn : (long long)p.OW * p.OH)};
        const uint32_t box[4] = {64, (uint32_t)p.TW, (uint32_t)p.TH, 1};
        int rc = cab_make_tmap_2b(&tmY, op_dtype, y, 4, dims, strides, box);
        if (rc) return rc;
    } else {
        tmY = tmB;  // unused
    }
    const size_t smem = static_cast<size_t>(fixed) + static_cast<size_t>(p.stages) * stage_bytes;

    const long long m_tiles = static_cast<long long>(Ng) * p.tiles_h * p.tiles_w;
    const long long tiles = m_tiles * p.n_tiles;
    CAB_REQUIRE(tiles < (1LL << 31), "conv_tc: too many tiles");
    p.num_tiles = static_cast<int>(tiles);
    int dev = 0, sms = 148;
    CAB_CUDA(cudaGetDevice(&dev));
    CAB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // experiment hook: CAB_TC_MAX_CTAS caps the persistent grid (leaves SMs to kernels of a concurrent stream)
    static const int max_ctas = getenv("CAB_TC_MAX_CTAS") ? atoi(getenv("CAB_TC_MAX_CTAS")) : 0;
    const int grid = static_cast<int>(std::min<long long>(tiles, max_ctas > 0 ? std::min(max_ctas, sms) : sms));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
#define CAB_TC_LAUNCH_T(ACT_, RES_, F32_, PRO_, T_)                                                                  \
    do {                                                                                                             \
        static bool attr_done = false;                                                                               \
        if (!attr_done) {                                                                                            \
            CAB_CUDA(cudaFuncSetAttribute(conv_tc_kernel<ACT_, RES_, F32_, PRO_, false, T_>,                         \
                                          cudaFuncAttributeMaxDynamicSharedMemorySize,                               \
                                          SMEM_LIMIT + 1024 - ((PRO_) ? 4096 : 0)));                                 \
            attr_done = true;                                                                                        \
        }                                                                                                            \
        conv_tc_kernel<ACT_, RES_, F32_, PRO_, false, T_>                                                            \
            <<<grid, (PRO_) ? NUM_THREADS + PRO_THREADS : NUM_THREADS, smem, st>>>(tmA[0], tmA[1], tmA[2], tmA[3], tmB, tmY, p); \
    } while (0)
#define CAB_TC_LAUNCH(ACT_, RES_, F32_, PRO_)                                                                        \
    do {                                                                                                             \
        if (op_dtype == CABINET_F16) CAB_TC_LAUNCH_T(ACT_, RES_, F32_, PRO_, f16);                                   \
        else CAB_TC_LAUNCH_T(ACT_, RES_, F32_, PRO_, bf16);                                                          \
    } while (0)
#define CAB_TC_LAUNCH_UP(ACT_)                                                                                       \
    do {                                                                                                             \
        static bool attr_done = false;                                                                               \
        if (!attr_done) {                                                                                            \
            CAB_CUDA(cudaFuncSetAttribute(conv_tc_kernel<ACT_, false, false, false, true>,                           \
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT + 1024));          \
            attr_done = true;                                                                                        \
        }                                                                                                            \
        conv_tc_kernel<ACT_, false, false, false, true><<<grid, NUM_THREADS, smem, st>>>(tmA[0], tmA[1], tmA[2],     \
                                                                                         tmA[3], tmB, tmY, p);       \
    } while (0)
    const bool f32 = y_dtype == CABINET_F32;
    if (up) {
        if (act == CABINET_ACT_RELU) CAB_TC_LAUNCH_UP(CABINET_ACT_RELU);
        else if (act == CABINET_ACT_NONE) CAB_TC_LAUNCH_UP(CABINET_ACT_NONE);
        else {
            cabinet_set_error("conv_tc_up: activation %d not built (ReLU / none)", act);
            return CABINET_ERR_INVALID;
        }
    } else if (a_scale) {
        CAB_REQUIRE(!f32 && act == CABINET_ACT_NONE, "conv_tc: the A-operand prologue is built for the linear project conv");
        if (res) CAB_TC_LAUNCH_T(CABINET_ACT_NONE, true, false, true, bf16);
        else CAB_TC_LAUNCH_T(CABINET_ACT_NONE, false, false, true, bf16);
    } else if (f32 && !res && act == CABINET_ACT_NONE) CAB_TC_LAUNCH(CABINET_ACT_NONE, false, true, false);
    else if (!f32 && !res && act == CABINET_ACT_NONE) CAB_TC_LAUNCH(CABINET_ACT_NONE, false, false, false);
    else if (!f32 && !res && act == CABINET_ACT_RELU) CAB_TC_LAUNCH(CABINET_ACT_RELU, false, false, false);
    else if (!f32 && !res && act == CABINET_ACT_HSWISH) CAB_TC_LAUNCH(CABINET_ACT_HSWISH, false, false, false);
    else if (!f32 && res && act == CABINET_ACT_NONE) CAB_TC_LAUNCH(CABINET_ACT_NONE, true, false, false);
    else {
        cabinet_set_error("conv_tc: unsupported epilogue combination (act %d, residual %d, fp32 out %d)", act,
                          res != nullptr, (int)f32);
        return CABINET_ERR_INVALID;
    }
#undef CAB_TC_LAUNCH
#undef CAB_TC_LAUNCH_T
#undef CAB_TC_LAUNCH_UP
    CAB_LAUNCH_CHECK();
    return CABINET_OK;
}
