// Implicit-GEMM convolution on tcgen05/TMEM for the KL-autoencoder decoder (sm_100a).
//
//   out[b, y, x, n] = epilogue( sum_{tap, c} src0[b, y + dy(tap), x + dx(tap), c] * W[n, tap*C0 + c]
//                             + sum_{c}      src1[b, y, x, c]                     * W[n, taps*C0 + c] )
//
// Replaces every torch.nn.Conv2d of the reference decoder (models/utils/autoencoder.py:320-449): the 3x3 convolutions
// of ResnetBlock (:95-106, :116-137), conv_in / conv_out (:363-365, :410-412), Upsample.conv (:47-56) and the 1x1
// convolutions q/k/v/proj_out of AttnBlock (:152-163); ResnetBlock.nin_shortcut (:112-114) rides along as a second K
// source of conv2 (the same trick as the U-ViT's long-skip GEMM), so `x + h` never needs its own pass.  The two
// batched matrix products of AttnBlock.forward (:174-186) run through the same kernel with per-sample "weights".
//
// Activations are NHWC bf16.  One M tile is 128 pixels = BH rows x BW columns of one sample; the A operand of tap
// (dy, dx) is ONE 4-D TMA box {64 channels, BW, BH, 1} at the shifted coordinate -- TMA zero-fills whatever falls
// outside the image, which is exactly the convolution's padding = 1, so there is no im2col buffer and no halo logic.
// The box lands in shared memory as a K-major 128 x 64 tile with the 128-byte swizzle, i.e. exactly the layout the
// U-ViT GEMMs feed to tcgen05.mma.
//
// Nearest-neighbour 2x upsampling followed by a 3x3 convolution (Upsample.forward, :52-56) is evaluated WITHOUT
// materialising the upsampled tensor: output pixels of parity class (py, px) only ever see a 2x2 neighbourhood of the
// low-resolution source, so the layer is four 2x2-tap convolutions with pre-summed weights (2.25x fewer FLOPs); each
// class stores its tile through a 5-D tensor map {n, px, x, py, b*H + y} of the high-resolution output.
//
// The encoder's Downsample (F.pad(h, (0,1,0,1)) then a 3x3 stride-2 convolution) is the same idea on the load side:
// the tile walk stays on the half-resolution output grid and the source is read through a 5-D tensor map
// {(q, c), x, p, y, b} with source pixel (2y + p, 2x + q), so every tap is again ONE box (ConvArgs::stride2).
//
// Roles (384 threads, 1 CTA / SM, persistent over tiles): warp 0 TMA producer, warp 1 MMA issuer, warp 2 TMEM
// allocator, warps 4-11 epilogue (two warpgroups, 64-column chunks, double-buffered TMEM accumulator).
// The epilogue can also emit the GroupNorm statistics of the NEXT layer: per (tile, group) sums of x and x^2 of the
// bf16 values it stores, reduced in a fixed order (deterministic; merged per sample by gn_finalize_kernel).
#pragma once
#include "gemm.cuh"

namespace ddb {

enum ConvEpilogue : int {
    CEPI_BIAS = 0,  // out = acc + bias                       (bf16, TMA store)
    CEPI_RES = 1,   // out = residual + acc + bias            (bf16, TMA store)
    CEPI_F32 = 2,   // out = scale * acc                      (fp32 row-major [M, N]; attention scores)
    CEPI_IMG = 3,   // out = acc + bias, first img_C columns  (fp32 NCHW image; conv_out)
};

struct ConvArgs {
    CUtensorMap tmA0;   // src0 NHWC bf16: dims {C0, W, H, B}, box {64, BW, BH, 1}
    CUtensorMap tmA1;   // src1 NHWC bf16 (1x1 K-extension), same box; unused when C1 == 0
    CUtensorMap tmB;    // weights [nw][N][Ktot] bf16, box {64, BN, 1}
    CUtensorMap tmOut;  // [M, N] bf16 box {64, 128}; sub-pixel mode: 5-D {N, 2, W, 2, B*H}, box {64, 1, BW, 1, BH}
    CUtensorMap tmRes;  // [M, N] bf16 residual, box {64, 128}
    int B, H, W;        // source grid
    int C0, C1, N;
    int tw, taps, dy0, dx0;  // tap t reads the source at (y + dy0 + t / tw, x + dx0 + t % tw)
    int BW, BH;              // pixel tile: BH rows x BW columns = 128 pixels
    int wmode;               // 0 one weight set, 1 one per sample (batched matmul), 2 one per sub-pixel class
    int subpixel;            // fused nearest-2x upsample: 4 parity classes, taps 2x2, dy0/dx0 derived per class
    int stride2;             // stride-2 3x3 conv over a 2H x 2W source (Downsample); tmA0 is then the 5-D view
                             // {2*C0 (q*C0 + c), W, 2 (p), H, B} of it and tap (ky, kx) is one box at
                             // (kx&1, x + (kx>>1), ky&1, y + (ky>>1)); the zero fill past the right / bottom edge is
                             // F.pad(h, (0, 1, 0, 1))
    const float* bias;       // [N] or nullptr
    float2* gn_part;         // optional [B][slots][32] (sum, sum of squares) of the stored values per GroupNorm group
    int cpg;                 // output channels per group (N / 32)
    float* out_f32;          // CEPI_F32
    float scale;
    float* img;              // CEPI_IMG: [B, img_C, H, W] fp32
    int img_C;
};

// MT = pixel tiles per work unit.  With MT = 2 a CTA computes two 128-pixel tiles against the SAME weight tile: per
// 64-channel K chunk it stages 2 x 16 KB of activations + BN x 128 B of weights for 2 x 4 MMAs.  For the N = 128 layers
// (the 256 x 256 level, 40 % of the decoder's FLOPs) that is 6 KB of shared-memory fill per MMA instead of 8 KB; those
// layers are paced by the SM's TMA fill rate (ncu: tensor pipe 41 % active with MT = 1), not by the tensor pipe.
template <int BN, int MT = 1>
struct ConvCfg {
    static constexpr int BM = 128;
    static constexpr int BK = 64;
    static constexpr int A_BYTES = BM * BK * 2;
    static constexpr int B_BYTES = BN * BK * 2;
    static constexpr int STAGE_BYTES = MT * A_BYTES + B_BYTES;
    static constexpr int STAGES = (144 * 1024) / STAGE_BYTES;  // 144 KB of operand ring: 3 / 4 / 6 stages
    static constexpr int OUT_BUF_BYTES = 128 * 128;  // 128 rows x 64 bf16
    static constexpr int NUM_OUT_BUFS = 4;           // 2 per epilogue warpgroup
    static constexpr int ACC_COLS = MT * BN;         // TMEM columns of one accumulator stage
    static constexpr int TMEM_COLS = (2 * ACC_COLS <= 128) ? 128 : (2 * ACC_COLS <= 256 ? 256 : 512);
    static constexpr int OFF_A = 0;
    static constexpr int OFF_B = OFF_A + STAGES * MT * A_BYTES;
    static constexpr int OFF_OUT = OFF_B + STAGES * B_BYTES;
    static constexpr int OFF_BAR = OFF_OUT + NUM_OUT_BUFS * OUT_BUF_BYTES;
    static constexpr int OFF_RED = OFF_BAR + 256;
    static constexpr int SMEM_BYTES = OFF_RED + 2 * 4 * 32 * 8 + 1024;  // + alignment slack
    static_assert(2 * ACC_COLS <= 512, "TMEM budget");
    static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

template <int BN, int EPI, int MT = 1>
__global__ void __launch_bounds__(384, 1) conv_igemm_kernel(const __grid_constant__ ConvArgs a) {
    using Cfg = ConvCfg<BN, MT>;
    constexpr int STAGES = Cfg::STAGES;
    constexpr bool kTmaStore = (EPI == CEPI_BIAS || EPI == CEPI_RES);

    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sA = smem + Cfg::OFF_A;
    uint8_t* sB = smem + Cfg::OFF_B;
    uint8_t* sOut = smem + Cfg::OFF_OUT;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
    uint64_t* full_bar = bars;
    uint64_t* empty_bar = bars + STAGES;
    uint64_t* tfull_bar = bars + 2 * STAGES;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint64_t* res_bar = tempty_bar + 2;  // [4]
    uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(res_bar + 4);
    float2* red = reinterpret_cast<float2*>(smem + Cfg::OFF_RED);  // [2 warpgroups][4 warps][32 lanes]

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    pdl_launch_dependents();
    const int ncls = a.subpixel ? 4 : 1;
    const int tps = (a.H * a.W) >> 7;  // source-grid tiles per sample
    const int nblk_n = a.N / BN;
    const int nblk_m = a.B * tps * ncls;            // pixel tiles (MT > 1: host guarantees nblk_m % MT == 0)
    const int num_units = (nblk_m / MT) * nblk_n;   // work units: MT consecutive pixel tiles x one N tile
    const int cpk = a.C0 / Cfg::BK;  // 64-channel chunks per tap
    const int nkb0 = a.taps * cpk;
    const int nkb = nkb0 + a.C1 / Cfg::BK;

    if (warp == 0 && lane == 0) {
        tma_prefetch_desc(&a.tmA0);
        tma_prefetch_desc(&a.tmB);
        if (a.C1 > 0) tma_prefetch_desc(&a.tmA1);
        if (kTmaStore) tma_prefetch_desc(&a.tmOut);
        if (EPI == CEPI_RES) tma_prefetch_desc(&a.tmRes);
    }
    if (warp == 1 && lane == 0) {
        for (int i = 0; i < STAGES; ++i) {
            mbar_init(&full_bar[i], 1);
            mbar_init(&empty_bar[i], 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(&tfull_bar[i], 1);
            mbar_init(&tempty_bar[i], 8);
        }
        for (int i = 0; i < 4; ++i) mbar_init(&res_bar[i], 1);
        fence_mbar_init();
    }
    if (warp == 2) tmem_alloc<Cfg::TMEM_COLS>(tmem_holder);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;
    pdl_wait();

    if (warp == 0) {
        // ===================================================================== TMA producer
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x) {
                const int mb0 = (unit / nblk_n) * MT, n_blk = unit % nblk_n;
                int tb[MT], ty0[MT], tx0[MT];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    const int rem = (mb0 + mt) / ncls;
                    const int p0 = (rem % tps) << 7;
                    tb[mt] = rem / tps, ty0[mt] = p0 / a.W, tx0[mt] = p0 % a.W;
                }
                const int cls = mb0 % ncls;  // (MT > 1 only without sub-pixel classes)
                const int dy0 = a.subpixel ? (cls >> 1) - 1 : a.dy0;
                const int dx0 = a.subpixel ? (cls & 1) - 1 : a.dx0;
                const int wz = a.wmode == 1 ? tb[0] : (a.wmode == 2 ? cls : 0);
                int tap = 0, cc = 0;
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(&empty_bar[stage], phase ^ 1);
                    mbar_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
                    uint8_t* dA = sA + stage * (MT * Cfg::A_BYTES);
                    if (kb < nkb0) {
                        const int ty = tap / a.tw, tx = tap - ty * a.tw;
                        if (a.stride2) {
#pragma unroll
                            for (int mt = 0; mt < MT; ++mt)
                                tma_load_5d(dA + mt * Cfg::A_BYTES, &a.tmA0, &full_bar[stage],
                                            cc * Cfg::BK + (tx & 1) * a.C0, tx0[mt] + (tx >> 1), ty & 1,
                                            ty0[mt] + (ty >> 1), tb[mt]);
                        } else {
#pragma unroll
                            for (int mt = 0; mt < MT; ++mt)
                                tma_load_4d(dA + mt * Cfg::A_BYTES, &a.tmA0, &full_bar[stage], cc * Cfg::BK,
                                            tx0[mt] + dx0 + tx, ty0[mt] + dy0 + ty, tb[mt]);
                        }
                        if (++cc == cpk) cc = 0, ++tap;
                    } else {
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt)
                            tma_load_4d(dA + mt * Cfg::A_BYTES, &a.tmA1, &full_bar[stage], (kb - nkb0) * Cfg::BK,
                                        tx0[mt], ty0[mt], tb[mt]);
                    }
                    tma_load_3d(sB + stage * Cfg::B_BYTES, &a.tmB, &full_bar[stage], kb * Cfg::BK, n_blk * BN, wz);
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================================================================== MMA issuer (one thread)
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_bf16(Cfg::BM, BN);
            int stage = 0;
            uint32_t phase = 0;
            int it = 0;
            for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x, ++it) {
                const int as = it & 1;
                const uint32_t aph = (it >> 1) & 1;
                mbar_wait(&tempty_bar[as], aph ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + as * Cfg::ACC_COLS;
                for (int kb = 0; kb < nkb; ++kb) {
                    mbar_wait(&full_bar[stage], phase);
                    tc_fence_after();
                    const uint64_t b_desc = umma_desc_kmajor_sw128(smem_u32(sB + stage * Cfg::B_BYTES));
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) {
                        const uint64_t a_desc =
                            umma_desc_kmajor_sw128(smem_u32(sA + stage * (MT * Cfg::A_BYTES) + mt * Cfg::A_BYTES));
#pragma unroll
                        for (int k = 0; k < Cfg::BK / 16; ++k)
                            umma_f16_ss(d_tmem + mt * BN, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0);
                    }
                    umma_commit(&empty_bar[stage]);
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
                umma_commit(&tfull_bar[as]);
            }
        }
    } else if (warp >= 4) {
        // ===================================================================== epilogue (2 warpgroups)
        const int g = (warp - 4) >> 2;
        const int quarter = warp & 3;
        const int et = threadIdx.x - 128 - g * 128;
        const int row_in_tile = quarter * 32 + lane;
        const uint32_t bar_id = 1 + g;
        uint8_t* my_bufs = sOut + g * 2 * Cfg::OUT_BUF_BYTES;
        float2* my_red = red + g * 128;
        constexpr int NCH = BN / 64;      // 64-column chunks per pixel tile
        constexpr int UCH = MT * NCH;     // chunks per work unit; warpgroup g takes chunks g, g+2, ...
        const int my_chunks = (UCH > g) ? (UCH - g + 1) / 2 : 0;
        uint32_t q = 0;

        // chunk k of this warpgroup inside a unit -> (pixel tile mb, column chunk c)
        auto res_coords = [&](int unit, int k, int& col, int& row0) {
            const int ch = g + 2 * k;
            col = (unit % nblk_n) * BN + (ch % NCH) * 64;
            row0 = ((unit / nblk_n) * MT + ch / NCH) * Cfg::BM;
        };
        if (EPI == CEPI_RES && et == 0 && my_chunks > 0 && (int)blockIdx.x < num_units) {
            int col, row0;
            res_coords(blockIdx.x, 0, col, row0);
            mbar_expect_tx(&res_bar[g * 2 + 0], Cfg::OUT_BUF_BYTES);
            tma_load_2d(my_bufs, &a.tmRes, &res_bar[g * 2 + 0], col, row0);
        }

        int it = 0;
        for (int unit = blockIdx.x; unit < num_units; unit += gridDim.x, ++it) {
            const int mb0 = (unit / nblk_n) * MT, n_blk = unit % nblk_n;
            const int as = it & 1;
            const uint32_t aph = (it >> 1) & 1;

            mbar_wait(&tfull_bar[as], aph);
            tc_fence_after();
            const uint32_t t_row = tmem_base + (uint32_t(quarter * 32) << 16) + as * Cfg::ACC_COLS;

            if (my_chunks == 0) {  // BN == 64, MT == 1: the second warpgroup has no columns
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty_bar[as]);
                continue;
            }
#pragma unroll 1
            for (int cc = 0; cc < my_chunks; ++cc) {
                const int ch = g + 2 * cc;
                const int mt = ch / NCH, c = ch % NCH;
                const int mb = mb0 + mt;
                const int cls = mb % ncls, rem = mb / ncls;
                const int b = rem / tps, r = rem % tps;
                const int p0 = r << 7;
                const int col0 = n_blk * BN + c * 64;
                uint32_t acc[2][32];
                tmem_ld_32x32b_x32(t_row + mt * BN + c * 64, acc[0]);
                tmem_ld_32x32b_x32(t_row + mt * BN + c * 64 + 32, acc[1]);

                if constexpr (kTmaStore) {
                    const int buf = q & 1;
                    uint8_t* sbuf = my_bufs + buf * Cfg::OUT_BUF_BYTES;
                    if constexpr (EPI == CEPI_RES) {
                        mbar_wait(&res_bar[g * 2 + buf], (q >> 1) & 1);
                    } else {
                        if (et == 0) tma_store_wait_read<1>();
                        named_bar_sync(bar_id, 128);
                    }
                    tmem_ld_wait();
                    if (cc == my_chunks - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty_bar[as]);
                    }
                    uint8_t* srow = sbuf + row_in_tile * 128;
                    const float* bias = a.bias + col0;  // never null on this path (zero vector for plain matmuls)
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float v[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) v[e] = __uint_as_float(acc[j >> 2][(j & 3) * 8 + e]);
                        const float4 b0 = __ldg(reinterpret_cast<const float4*>(bias + j * 8));
                        const float4 b1 = __ldg(reinterpret_cast<const float4*>(bias + j * 8 + 4));
                        v[0] += b0.x, v[1] += b0.y, v[2] += b0.z, v[3] += b0.w;
                        v[4] += b1.x, v[5] += b1.y, v[6] += b1.z, v[7] += b1.w;
                        uint4* sp = reinterpret_cast<uint4*>(srow + ((j ^ (row_in_tile & 7)) << 4));
                        if constexpr (EPI == CEPI_RES) {
                            const uint4 rr = *sp;
                            v[0] += bf16_lo(rr.x), v[1] += bf16_hi(rr.x);
                            v[2] += bf16_lo(rr.y), v[3] += bf16_hi(rr.y);
                            v[4] += bf16_lo(rr.z), v[5] += bf16_hi(rr.z);
                            v[6] += bf16_lo(rr.w), v[7] += bf16_hi(rr.w);
                        }
                        uint4 o;
                        o.x = pack_bf16(v[0], v[1]);
                        o.y = pack_bf16(v[2], v[3]);
                        o.z = pack_bf16(v[4], v[5]);
                        o.w = pack_bf16(v[6], v[7]);
                        *sp = o;
                    }
                    fence_proxy_async_smem();
                    named_bar_sync(bar_id, 128);
                    if (et == 0) {
                        if (a.subpixel)
                            tma_store_5d(&a.tmOut, sbuf, col0, cls & 1, p0 % a.W, cls >> 1, b * a.H + p0 / a.W);
                        else
                            tma_store_2d(&a.tmOut, sbuf, col0, mb * Cfg::BM);
                        tma_store_commit();
                        if constexpr (EPI == CEPI_RES) {
                            int ncc = cc + 1, nunit = unit;
                            if (ncc == my_chunks) {
                                ncc = 0;
                                nunit = unit + gridDim.x;
                            }
                            if (nunit < num_units) {
                                tma_store_wait_read<1>();
                                int col, row0;
                                res_coords(nunit, ncc, col, row0);
                                uint64_t* rb = &res_bar[g * 2 + (buf ^ 1)];
                                mbar_expect_tx(rb, Cfg::OUT_BUF_BYTES);
                                tma_load_2d(my_bufs + (buf ^ 1) * Cfg::OUT_BUF_BYTES, &a.tmRes, rb, col, row0);
                            }
                        }
                    }
                    if (a.gn_part) {
                        // GroupNorm partials of the stored (bf16-rounded) tile: lane = column pair, warp = 32-row band
                        float s = 0.f, ss = 0.f;
#pragma unroll 8
                        for (int rr = 0; rr < 32; ++rr) {
                            const int row = quarter * 32 + rr;
                            const uint32_t u = *reinterpret_cast<const uint32_t*>(
                                sbuf + row * 128 + (((lane >> 2) ^ (row & 7)) << 4) + (lane & 3) * 4);
                            const float lo = bf16_lo(u), hi = bf16_hi(u);
                            s += lo + hi;
                            ss = fmaf(lo, lo, fmaf(hi, hi, ss));
                        }
                        const int lpg = a.cpg >> 1;  // lanes per group
                        for (int off = 1; off < lpg; off <<= 1) {
                            s += __shfl_xor_sync(0xffffffffu, s, off);
                            ss += __shfl_xor_sync(0xffffffffu, ss, off);
                        }
                        my_red[quarter * 32 + lane] = make_float2(s, ss);
                        named_bar_sync(bar_id, 128);
                        if (quarter == 0 && (lane % lpg) == 0) {
                            float2 t0 = my_red[lane], t1 = my_red[32 + lane], t2 = my_red[64 + lane],
                                   t3 = my_red[96 + lane];
                            const float2 t = make_float2((t0.x + t1.x) + (t2.x + t3.x), (t0.y + t1.y) + (t2.y + t3.y));
                            const int group = (col0 + 2 * lane) / a.cpg;
                            const int slot = r * ncls + cls;
                            a.gn_part[((size_t)b * (tps * ncls) + slot) * 32 + group] = t;
                        }
                    }
                    ++q;
                } else {
                    tmem_ld_wait();
                    if (cc == my_chunks - 1) {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&tempty_bar[as]);
                    }
                    if constexpr (EPI == CEPI_F32) {
                        float* dst = a.out_f32 + ((size_t)mb * Cfg::BM + row_in_tile) * a.N + col0;
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            float4 o;
                            o.x = a.scale * __uint_as_float(acc[j >> 3][(j & 7) * 4 + 0]);
                            o.y = a.scale * __uint_as_float(acc[j >> 3][(j & 7) * 4 + 1]);
                            o.z = a.scale * __uint_as_float(acc[j >> 3][(j & 7) * 4 + 2]);
                            o.w = a.scale * __uint_as_float(acc[j >> 3][(j & 7) * 4 + 3]);
                            reinterpret_cast<float4*>(dst)[j] = o;
                        }
                    } else {  // CEPI_IMG: consecutive lanes are consecutive pixels of one channel plane
                        // (img_C <= 8: out_ch of the decoder, 2 * embed_dim moments of the encoder)
                        const size_t plane = (size_t)a.H * a.W;
                        float* dst = a.img + (size_t)b * a.img_C * plane + p0 + row_in_tile;
#pragma unroll
                        for (int chn = 0; chn < 8; ++chn) {
                            if (col0 + chn < a.img_C)
                                dst[(size_t)(col0 + chn) * plane] =
                                    __uint_as_float(acc[0][chn]) + __ldg(a.bias + col0 + chn);
                        }
                    }
                }
            }
        }
        if (kTmaStore && et == 0) tma_store_wait_all<0>();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Memory-bound companions (NHWC bf16, 128-bit accesses).

// z [B, Cz, H, W] fp32 -> post_quant_conv(z / scale_factor) as NHWC bf16 with the channel dimension zero-padded to
// 64 (one K chunk of conv_in).  FrozenAutoencoderKL.decode, models/utils/autoencoder.py:486-488.
__global__ void ae_prep_kernel(const float* __restrict__ z, const float* __restrict__ w, const float* __restrict__ bias,
                               float inv_scale, int B, int Cz, int HW, __nv_bfloat16* __restrict__ out) {
    pdl_launch_dependents();
    pdl_wait();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;  // pixel over B*HW
    if (p >= B * HW) return;
    const int b = p / HW, i = p % HW;
    float zin[8], zo[8];
    for (int c = 0; c < Cz; ++c) zin[c] = z[((size_t)b * Cz + c) * HW + i] * inv_scale;
    for (int o = 0; o < Cz; ++o) {
        float acc = bias[o];
        for (int c = 0; c < Cz; ++c) acc = fmaf(w[o * Cz + c], zin[c], acc);
        zo[o] = acc;
    }
    uint4* dst = reinterpret_cast<uint4*>(out + (size_t)p * 64);
    for (int j = 0; j < 8; ++j) {
        float v[8];
        for (int e = 0; e < 8; ++e) v[e] = (j * 8 + e < Cz) ? zo[j * 8 + e] : 0.f;
        uint4 o;
        o.x = pack_bf16(v[0], v[1]), o.y = pack_bf16(v[2], v[3]), o.z = pack_bf16(v[4], v[5]),
        o.w = pack_bf16(v[6], v[7]);
        dst[j] = o;
    }
}

// Encoder conv_in over the caller's image x [B, Cin, H, W] fp32 (Cin <= 7): im2col rows [B*H*W, 64] bf16 with column
// (ky*3 + kx)*Cin + c = x[b, c, y + ky - 1, x + kx - 1] (zero outside the image, zero in columns >= 9*Cin), so that
// conv_in runs as a one-tap convolution with K = 64 instead of nine taps over 64 zero-padded channels.
__global__ void ae_im2col_kernel(const float* __restrict__ img, int B, int Cin, int H, int W,
                                 __nv_bfloat16* __restrict__ out) {
    pdl_launch_dependents();
    pdl_wait();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;  // pixel over B*H*W
    if (p >= B * H * W) return;
    const int b = p / (H * W), i = p % (H * W), y = i / W, x = i % W;
    const float* src = img + (size_t)b * Cin * H * W;
    float v[64];  // compile-time indices only: stays in registers
    int t = 0, c = 0, ky = 0, kx = 0;
#pragma unroll
    for (int k = 0; k < 64; ++k) {
        const int yy = y + ky - 1, xx = x + kx - 1;
        v[k] = (t < 9 && yy >= 0 && yy < H && xx >= 0 && xx < W) ? src[((size_t)c * H + yy) * W + xx] : 0.f;
        if (++c == Cin) {
            c = 0, ++t;
            if (++kx == 3) kx = 0, ++ky;
        }
    }
    uint4* dst = reinterpret_cast<uint4*>(out + (size_t)p * 64);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        uint4 o;
        o.x = pack_bf16(v[j * 8 + 0], v[j * 8 + 1]), o.y = pack_bf16(v[j * 8 + 2], v[j * 8 + 3]);
        o.z = pack_bf16(v[j * 8 + 4], v[j * 8 + 5]), o.w = pack_bf16(v[j * 8 + 6], v[j * 8 + 7]);
        dst[j] = o;
    }
}

// DiagonalGaussian sample of FrozenAutoencoderKL.sample: moments [B, 2E, HW] fp32 (mean | logvar), noise [B, E, HW]
//   z = scale * (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise)
// in torch's operation order, without FMA contraction.
__global__ void ae_sample_kernel(const float* __restrict__ moments, const float* __restrict__ noise, int B, int E,
                                 int HW, float scale, float* __restrict__ z) {
    const size_t n = (size_t)B * E * HW;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const size_t b = i / ((size_t)E * HW), r = i % ((size_t)E * HW);
    const float mean = moments[b * 2 * E * HW + r];
    const float logvar = fminf(fmaxf(moments[b * 2 * E * HW + (size_t)E * HW + r], -30.f), 20.f);
    const float stdv = expf(__fmul_rn(0.5f, logvar));
    z[i] = __fmul_rn(scale, __fadd_rn(mean, __fmul_rn(stdv, noise[i])));
}

// quant_conv (1x1, Nj -> No) folded into the preceding conv (w [Nj, K], b [Nj]) in fp32:
//   w'[o, k] = sum_j wq[o, j] w[j, k],  b'[o] = bq[o] + sum_j wq[o, j] b[j]
__global__ void fold_1x1_kernel(const float* __restrict__ wq, const float* __restrict__ bq,
                                const float* __restrict__ w, const float* __restrict__ b, int No, int Nj, int K,
                                float* __restrict__ w_out, float* __restrict__ b_out) {
    const int o = blockIdx.x;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        float acc = 0.f;
        for (int j = 0; j < Nj; ++j) acc = fmaf(wq[o * Nj + j], w[(size_t)j * K + k], acc);
        w_out[(size_t)o * K + k] = acc;
    }
    if (threadIdx.x == 0) {
        float acc = bq[o];
        for (int j = 0; j < Nj; ++j) acc = fmaf(wq[o * Nj + j], b[j], acc);
        b_out[o] = acc;
    }
}

// (sum, sumsq) partials [B][slots][32] -> per-(sample, channel) affine  y = x * sc + sh  with
// sc = rstd * gamma, sh = beta - mean * rstd * gamma  (torch.nn.GroupNorm(32, C, eps=1e-6), autoencoder.py:37-40).
// One CTA per sample, 256 threads: 8 fixed slices of the slot range per group, combined in a fixed order.
__global__ void gn_finalize_kernel(const float2* __restrict__ part, int slots, int C, int cpg, float count, float eps,
                                   const float* __restrict__ gamma, const float* __restrict__ beta,
                                   float2* __restrict__ affine) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float2 sred[8][32];
    __shared__ float2 smr[32];
    const int b = blockIdx.x, g = threadIdx.x & 31, sl = threadIdx.x >> 5;
    const float2* p = part + (size_t)b * slots * 32 + g;
    double s = 0.0, ss = 0.0;
    for (int i = sl; i < slots; i += 8) {
        const float2 v = p[(size_t)i * 32];
        s += v.x, ss += v.y;
    }
    sred[sl][g] = make_float2((float)s, (float)ss);
    __syncthreads();
    if (sl == 0) {
        double ts = 0.0, tss = 0.0;
        for (int i = 0; i < 8; ++i) ts += sred[i][g].x, tss += sred[i][g].y;
        const double mean = ts / count;
        double var = tss / count - mean * mean;
        if (var < 0.0) var = 0.0;
        smr[g] = make_float2((float)mean, (float)(1.0 / sqrt(var + (double)eps)));
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const float2 mr = smr[c / cpg];
        const float sc = mr.y * gamma[c];
        affine[(size_t)b * C + c] = make_float2(sc, beta[c] - mr.x * sc);
    }
}

// y = swish(x * sc + sh) (or just the affine when swish == 0: AttnBlock.norm), NHWC bf16.  A CTA owns a contiguous slab
// of `rows_per_cta` pixels of one sample; every thread keeps four independent 16-byte loads in flight.
// swish(v) = v * sigmoid(v) = h + h * tanh(h) with h = v / 2: the 1/2 is folded into the affine and the sigmoid costs
// one MUFU op (tanh.approx) instead of two (ex2 + rcp) -- at 8 elements per 16 bytes the MUFU pipe (16 / clk / SM)
// would otherwise cap the kernel below the HBM rate.
// kFixed: 256 % (C / 8) == 0, so a thread sees the same 8 channels in every iteration and keeps their affine in
// registers (every decoder width of the reference); otherwise the affine is looked up in shared memory.
template <bool kFixed>
__global__ void __launch_bounds__(256) gn_apply_kernel(const __nv_bfloat16* __restrict__ x,
                                                       const float2* __restrict__ affine, int HW, int C,
                                                       int rows_per_cta, int swish, __nv_bfloat16* __restrict__ y) {
    pdl_launch_dependents();
    extern __shared__ float2 saff[];  // [C]
    const int b = blockIdx.y;
    const float fold = swish ? 0.5f : 1.f;
    const int units = C >> 3;
    pdl_wait();
    float2 aff[8];
    if constexpr (kFixed) {
        const float2* ap = affine + (size_t)b * C + (threadIdx.x % units) * 8;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float2 t = __ldg(ap + e);
            aff[e] = make_float2(t.x * fold, t.y * fold);
        }
    } else {
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            const float2 t = affine[(size_t)b * C + c];
            saff[c] = make_float2(t.x * fold, t.y * fold);
        }
        __syncthreads();
    }
    const int row0 = blockIdx.x * rows_per_cta;
    const int rows = min(rows_per_cta, HW - row0);
    const int total = rows * units;  // 16-byte units of this slab (contiguous in memory)
    const size_t base = ((size_t)b * HW + row0) * C;
    const uint4* __restrict__ src = reinterpret_cast<const uint4*>(x + base);
    uint4* __restrict__ dst = reinterpret_cast<uint4*>(y + base);
    for (int i0 = threadIdx.x; i0 < total; i0 += 4 * 256) {
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = i0 + k * 256;
            if (i < total) v[k] = __ldcs(src + i);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int i = i0 + k * 256;
            if (i >= total) break;
            if constexpr (!kFixed) {
                const float2* sp = saff + (i % units) * 8;
#pragma unroll
                for (int e = 0; e < 8; ++e) aff[e] = sp[e];
            }
            const uint32_t w[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
            uint32_t o[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                float lo = fmaf(bf16_lo(w[e]), aff[2 * e].x, aff[2 * e].y);
                float hi = fmaf(bf16_hi(w[e]), aff[2 * e + 1].x, aff[2 * e + 1].y);
                if (swish) {
                    lo = fmaf(lo, tanh_approx(lo), lo);
                    hi = fmaf(hi, tanh_approx(hi), hi);
                }
                o[e] = pack_bf16(lo, hi);
            }
            dst[i] = make_uint4(o[0], o[1], o[2], o[3]);
        }
    }
}

// P = softmax(S) over rows of S [rows, n] fp32 (already scaled) -> bf16.  One warp per row.
__global__ void softmax_rows_kernel(const float* __restrict__ S, int rows, int n, __nv_bfloat16* __restrict__ P) {
    pdl_launch_dependents();
    pdl_wait();
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float* s = S + (size_t)row * n;
    float m = -INFINITY;
    for (int i = lane * 4; i < n; i += 128) {
        const float4 v = *reinterpret_cast<const float4*>(s + i);
        m = fmaxf(fmaxf(m, fmaxf(v.x, v.y)), fmaxf(v.z, v.w));
    }
    for (int off = 16; off; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    float sum = 0.f;
    for (int i = lane * 4; i < n; i += 128) {
        const float4 v = *reinterpret_cast<const float4*>(s + i);
        sum += __expf(v.x - m) + __expf(v.y - m) + __expf(v.z - m) + __expf(v.w - m);
    }
    for (int off = 16; off; off >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, off);
    const float inv = 1.f / sum;
    for (int i = lane * 4; i < n; i += 128) {
        const float4 v = *reinterpret_cast<const float4*>(s + i);
        uint2 o;
        o.x = pack_bf16(__expf(v.x - m) * inv, __expf(v.y - m) * inv);
        o.y = pack_bf16(__expf(v.z - m) * inv, __expf(v.w - m) * inv);
        *reinterpret_cast<uint2*>(P + (size_t)row * n + i) = o;
    }
}

// vT[b][c][t] = qkv[b][t][v_off + c]   (32 x 32 shared-memory tiles)
__global__ void transpose_v_kernel(const __nv_bfloat16* __restrict__ qkv, int T, int C, int pitch, int v_off,
                                   __nv_bfloat16* __restrict__ vT) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ __nv_bfloat16 tile[32][33];
    const int b = blockIdx.z, t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
    for (int i = threadIdx.y; i < 32; i += blockDim.y)
        tile[i][threadIdx.x] = qkv[((size_t)b * T + t0 + i) * pitch + v_off + c0 + threadIdx.x];
    __syncthreads();
    for (int i = threadIdx.y; i < 32; i += blockDim.y)
        vT[((size_t)b * C + c0 + i) * T + t0 + threadIdx.x] = tile[threadIdx.x][i];
}

// Weight packing.  conv [N, C, kh, kw] fp32 -> bf16 [N_pad][taps*C_pad (+ C1)] with k = tap*C_pad + c; rows >= N and
// channels >= C are zero.  mode 0: plain taps (kh*kw); mode 1..4: sub-pixel class (py, px) = ((mode-1)>>1, (mode-1)&1)
// of a nearest-2x upsample followed by this 3x3 convolution: the 2x2 taps are sums of the original taps that read the
// same low-resolution pixel.
__global__ void pack_conv_kernel(const float* __restrict__ w, int N, int C, int kh, int kw, int N_pad, int C_pad,
                                 int ktot, int k_off, int mode, __nv_bfloat16* __restrict__ out) {
    const int n = blockIdx.x;
    const int taps = mode == 0 ? kh * kw : 4;
    for (int i = threadIdx.x; i < taps * C_pad; i += blockDim.x) {
        const int tap = i / C_pad, c = i % C_pad;
        float v = 0.f;
        if (n < N && c < C) {
            const float* wp = w + ((size_t)n * C + c) * kh * kw;
            if (mode == 0) {
                v = wp[tap];
            } else {
                const int py = (mode - 1) >> 1, px = (mode - 1) & 1;
                const int ty = tap >> 1, tx = tap & 1;
                // class parity 0: source offset -1 <- k = 0; offset 0 <- k = 1, 2.  parity 1: 0 <- k = 0, 1; +1 <- k = 2
                int ky0, ky1, kx0, kx1;
                if (py == 0) ky0 = ty == 0 ? 0 : 1, ky1 = ty == 0 ? 0 : 2;
                else ky0 = ty == 0 ? 0 : 2, ky1 = ty == 0 ? 1 : 2;
                if (px == 0) kx0 = tx == 0 ? 0 : 1, kx1 = tx == 0 ? 0 : 2;
                else kx0 = tx == 0 ? 0 : 2, kx1 = tx == 0 ? 1 : 2;
                for (int ky = ky0; ky <= ky1; ++ky)
                    for (int kx = kx0; kx <= kx1; ++kx) v += wp[ky * 3 + kx];
            }
        }
        out[(size_t)n * ktot + k_off + i] = __float2bfloat16(v);
    }
}

// bias[n] = b0[n] (+ b1[n]) for n < N, 0 for the padding rows
__global__ void add_bias_kernel(const float* __restrict__ b0, const float* __restrict__ b1, int N, int N_pad,
                                float* __restrict__ out) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n < N_pad) out[n] = n < N ? b0[n] + (b1 ? b1[n] : 0.f) : 0.f;
}

}  // namespace ddb
