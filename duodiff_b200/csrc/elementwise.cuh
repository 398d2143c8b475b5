// HBM-bound kernels of the sampling path: token assembly + patch embed, LayerNorm row statistics (+ early-exit
// probe), 3x3 final conv, DDPM update, weight re-packing, early-exit selection / compaction, output layout.
#pragma once
#include "ptx.cuh"

namespace ddb {

// =====================================================================================================
// Weight re-packing (once per model load)
// =====================================================================================================
// W'[n,k] = bf16(W[n,k] * gamma[k]);  colsum[n] = sum_k float(W'[n,k]);  bias'[n] = bias[n] + sum_k W[n,k]*beta[k]
// gamma/beta may be null (plain cast).  Rows n >= N_src are zero-filled (decoder padding).
__global__ void pack_linear_kernel(const float* __restrict__ W, const float* __restrict__ bias,
                                   const float* __restrict__ gamma, const float* __restrict__ beta, int N_src, int K,
                                   __nv_bfloat16* __restrict__ Wp, float* __restrict__ colsum,
                                   float* __restrict__ bias_out) {
    const int n = blockIdx.x;
    float cs = 0.f, bs = 0.f;
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
        float w = (n < N_src) ? W[(size_t)n * K + k] : 0.f;
        float wg = gamma ? w * gamma[k] : w;
        __nv_bfloat16 q = __float2bfloat16_rn(wg);
        Wp[(size_t)n * K + k] = q;
        cs += __bfloat162float(q);
        if (beta) bs += w * beta[k];
    }
    __shared__ float red[2][32];
    for (int o = 16; o > 0; o >>= 1) {
        cs += __shfl_xor_sync(0xffffffffu, cs, o);
        bs += __shfl_xor_sync(0xffffffffu, bs, o);
    }
    if ((threadIdx.x & 31) == 0) red[0][threadIdx.x >> 5] = cs, red[1][threadIdx.x >> 5] = bs;
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, b = 0.f;
        for (int i = 0; i < (int)(blockDim.x >> 5); ++i) a += red[0][i], b += red[1][i];
        if (colsum) colsum[n] = a;
        if (bias_out) bias_out[n] = ((bias && n < N_src) ? bias[n] : 0.f) + b;
    }
}

// patch-embed conv weight [D, C, p, p] -> transposed fp32 [pd, D] (k = (c, p1, p2) as in the conv weight)
__global__ void transpose_pe_kernel(const float* __restrict__ W, int D, int pd, float* __restrict__ Wt) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < D * pd) {
        int e = i / pd, k = i % pd;
        Wt[(size_t)k * D + e] = W[i];
    }
}

constexpr int EMB_TOK = 16;  // patches per image row (every reference config: img_size / patch_size == 16)

// =====================================================================================================
// Tensor-core patch embed (the model path): the per-patch linear runs on the CTA-pair tcgen05 GEMM.
//   patch_gather_kernel  x_img fp32 -> A [B*256, 128] bf16: columns [0,64) = bf16(x) of the patch vector (c, p1, p2),
//                        zero-padded; columns [64,128) = bf16(x - bf16(x)).  With W duplicated along K the GEMM
//                        computes W_bf16 . (x_hi + x_lo): the input keeps ~16 mantissa bits, only the weights are bf16
//                        like every other Linear of the path.
//   token_extras_kernel  time / label token rows (+ pos_embed) and their 64-column LayerNorm partials.
// The GEMM epilogue adds bias + pos_embed and writes the token rows and their LayerNorm partials (GemmArgs embed_mode).
// =====================================================================================================
// two horizontally adjacent pixels -> bf16 hi pair at dst, lo pair (x - bf16(x)) at dst + 64
__device__ __forceinline__ void patch_store_pair(__nv_bfloat16* dst, float v0, float v1) {
    const __nv_bfloat162 hi = __floats2bfloat162_rn(v0, v1);
    const __nv_bfloat162 lo = __floats2bfloat162_rn(v0 - __low2float(hi), v1 - __high2float(hi));
    *reinterpret_cast<__nv_bfloat162*>(dst) = hi;
    *reinterpret_cast<__nv_bfloat162*>(dst + 64) = lo;
}
// address of element (c, p1, p2) of patch (hh, ww) of sample b in the patch matrix A [B * Hp * Wp, 128]
__device__ __forceinline__ __nv_bfloat16* patch_elem(__nv_bfloat16* A, int b, int c, int yy, int xx, int P, int Hp,
                                                      int Wp) {
    const int hh = yy / P, p1 = yy % P, ww = xx / P, p2 = xx % P;
    return A + ((size_t)b * (Wp * Hp) + hh * Wp + ww) * 128 + (c * P + p1) * P + p2;
}
__global__ void __launch_bounds__(256) patch_gather_kernel(const float* __restrict__ x_img,
                                                           __nv_bfloat16* __restrict__ A, int B, int C, int H, int W,
                                                           int P) {
    pdl_launch_dependents();
    pdl_wait();
    // one thread per (sample, channel, image row, patch column): P contiguous pixels
    const int Wp = W / P;
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)B * C * H * Wp) return;
    const int ww = i % Wp;
    size_t r = i / Wp;
    const int yy = r % H;
    r /= H;
    const int c = r % C, b = r / C;
    const float* src = x_img + (((size_t)b * C + c) * H + yy) * W + ww * P;
    __nv_bfloat16* dst = patch_elem(A, b, c, yy, ww * P, P, H / P, Wp);
    for (int p2 = 0; p2 < P; p2 += 2) {
        const float2 v = *reinterpret_cast<const float2*>(src + p2);
        patch_store_pair(dst + p2, v.x, v.y);
    }
}

// 256 threads write the extras rows (label token, time token; + pos_embed) of sample b and their D/64 LayerNorm
// partials (warp w handles chunks w, w+8, ...).  tau = raw timestep (models/uvit.py:352-360).
__device__ __forceinline__ void write_token_extras(int b, float tau, const long long* __restrict__ y,
                                                   const float* __restrict__ pos, const float* __restrict__ label_emb,
                                                   __nv_bfloat16* __restrict__ tokens, float2* __restrict__ stats_p,
                                                   int D, int L, int extras, int normalize_t, int num_classes,
                                                   const float* __restrict__ time_row = nullptr) {
    // time_row (mlp_time_embed = True, models/uvit.py:264-272): the time token after its MLP, from time_mlp_kernel
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int half = D / 2;
    if (normalize_t) tau = tau / 1000.f;
    for (int row = 0; row < extras; ++row) {
        const bool is_time = (row == extras - 1);
        // labels are validated on the host (the reference raises IndexError); the clamp only keeps a bad label from
        // reading outside the embedding table
        long long cls = is_time ? 0 : y[b];
        cls = cls < 0 ? 0 : (cls >= num_classes ? num_classes - 1 : cls);
        const float* src = is_time ? nullptr : label_emb + (size_t)cls * D;
        for (int ch = warp; ch < D / 64; ch += 8) {
            float v[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const int e = ch * 64 + lane * 2 + u;
                float x;
                if (is_time && time_row) {
                    x = time_row[e];
                } else if (is_time) {
                    // time token: [cos(tau f_i) | sin(tau f_i)], f_i = exp(-ln(1e4) i / half)
                    const int i = (e < half) ? e : e - half;
                    const float f = expf((-9.210340371976184f * (float)i) / (float)half);
                    x = (e < half) ? cosf(tau * f) : sinf(tau * f);
                } else {
                    x = src[e];
                }
                v[u] = x + pos[(size_t)row * D + e];
            }
            const uint32_t pk = pack_bf16(v[0], v[1]);
            *reinterpret_cast<uint32_t*>(tokens + ((size_t)b * L + row) * D + ch * 64 + lane * 2) = pk;
            const float r0 = bf16_lo(pk), r1 = bf16_hi(pk);
            float s = r0 + r1;
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            const float mean = s * (1.f / 64.f);
            float q = (r0 - mean) * (r0 - mean) + (r1 - mean) * (r1 - mean);
            for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
            if (lane == 0 && stats_p) stats_p[((size_t)b * L + row) * (D / 64) + ch] = make_float2(mean, q);
        }
    }
}
// grid = B, 256 threads.  The timestep comes from the caller's float vector (UViT.forward) or, inside the sampler, from
// the device-side step counter.
__global__ void __launch_bounds__(256) token_extras_kernel(const float* __restrict__ tsteps,
                                                           const int* __restrict__ t_dev,
                                                           const long long* __restrict__ y,
                                                           const float* __restrict__ pos,
                                                           const float* __restrict__ label_emb,
                                                           __nv_bfloat16* __restrict__ tokens,
                                                           float2* __restrict__ stats_p, int D, int L, int extras,
                                                           int normalize_t, int num_classes,
                                                           const float* __restrict__ time_rows /*[B, D] or null*/,
                                                           const float* __restrict__ time_tab /*[1000, D] or null*/) {
    pdl_launch_dependents();
    pdl_wait();
    const int b = blockIdx.x;
    const float tau = t_dev ? (float)ld_state(t_dev) : tsteps[b];
    const float* tr = nullptr;  // mlp_time_embed: per-sample rows (caller's timesteps) or the table row of the step
    if (time_rows && !t_dev) tr = time_rows + (size_t)b * D;
    else if (time_tab && t_dev) tr = time_tab + (size_t)min(max((int)tau, 0), 999) * D;
    write_token_extras(b, tau, y, pos, label_emb, tokens, stats_p, D, L, extras, normalize_t, num_classes, tr);
}

// mlp_time_embed = True (models/uvit.py:264-272, 358): time token = Linear(4D, D)(SiLU(Linear(D, 4D)(emb(tau)))).
// Row r: tau = tsteps[r] (the caller's timesteps) or, with tsteps == null, tau = r (the table of the 1000 integer
// timesteps, built once at model creation: inside the sampler the time token is a table row).  The same kernel fills
// both, so a table row and a per-sample row of the same timestep are the same bits.  256 threads, smem 5 D floats.
__global__ void __launch_bounds__(256) time_mlp_kernel(const float* __restrict__ tsteps, int normalize_t, int D,
                                                       const float* __restrict__ w1 /*[4D, D]*/,
                                                       const float* __restrict__ b1, const float* __restrict__ w2 /*[D, 4D]*/,
                                                       const float* __restrict__ b2, float* __restrict__ out /*[rows, D]*/) {
    extern __shared__ float tm_smem[];
    float* emb = tm_smem;      // [D]
    float* hid = tm_smem + D;  // [4D]
    pdl_launch_dependents();
    pdl_wait();
    const int r = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, half = D / 2;
    float tau = tsteps ? tsteps[r] : (float)r;
    if (normalize_t) tau = tau / 1000.f;
    for (int e = threadIdx.x; e < D; e += blockDim.x) {
        const int i = (e < half) ? e : e - half;
        const float f = expf((-9.210340371976184f * (float)i) / (float)half);
        emb[e] = (e < half) ? cosf(tau * f) : sinf(tau * f);
    }
    __syncthreads();
    for (int j = warp; j < 4 * D; j += 8) {
        float d = 0.f;
        for (int k = lane; k < D; k += 32) d = fmaf(w1[(size_t)j * D + k], emb[k], d);
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        const float z = d + b1[j];
        if (lane == 0) hid[j] = z / (1.f + expf(-z));
    }
    __syncthreads();
    for (int j = warp; j < D; j += 8) {
        float d = 0.f;
        for (int k = lane; k < 4 * D; k += 32) d = fmaf(w2[(size_t)j * 4 * D + k], hid[k], d);
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        if (lane == 0) out[(size_t)r * D + j] = d + b2[j];
    }
}

// W_pe [D, pd] fp32 (conv weight flattened (c, p1, p2)) -> [D, 128] bf16: [W | 0 | W | 0]
__global__ void pack_patch_embed_kernel(const float* __restrict__ W, int D, int pd, __nv_bfloat16* __restrict__ Wp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= D * 128) return;
    const int e = i / 128, k = i % 128, kk = k & 63;
    Wp[i] = __float2bfloat16_rn(kk < pd ? W[(size_t)e * pd + kk] : 0.f);
}
__global__ void cast_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = __float2bfloat16_rn(src[i]);
}

// =====================================================================================================
// LayerNorm row statistics (nn.LayerNorm, eps 1e-5; models/uvit.py:206-207,377) as (mean, M2) per row, and --
// optionally -- the early-exit MLP probe's per-token dot product w.x (models/early_exit.py:34-37) in the layout the
// GEMM epilogues use for it: probe_p[row, D/64] partial dots (here: the whole dot in part 0, zeros elsewhere).  Only the
// first layer needs this pass; the input of every later block comes with its statistics and probe partials from the
// fc2 GEMM that produced it.  One warp per row, 16-byte loads, exact two-pass statistics in registers.
// =====================================================================================================
template <int D>
__global__ void __launch_bounds__(256) ln_stats_kernel(const __nv_bfloat16* __restrict__ x, int M,
                                                       const int* __restrict__ m_dev, float2* __restrict__ stats,
                                                       const float* __restrict__ probe_w,
                                                       float* __restrict__ probe_p) {
    constexpr int CH = D / 256;  // 16-byte chunks per lane
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    pdl_launch_dependents();
    pdl_wait();
    const int Mr = m_dev ? ld_state(m_dev) : M;
    if (row >= Mr) return;
    const uint4* xr = reinterpret_cast<const uint4*>(x + (size_t)row * D);
    float v[CH][8];
    float sum = 0.f;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
        const uint4 u = __ldg(xr + c * 32 + lane);
        v[c][0] = bf16_lo(u.x), v[c][1] = bf16_hi(u.x), v[c][2] = bf16_lo(u.y), v[c][3] = bf16_hi(u.y);
        v[c][4] = bf16_lo(u.z), v[c][5] = bf16_hi(u.z), v[c][6] = bf16_lo(u.w), v[c][7] = bf16_hi(u.w);
#pragma unroll
        for (int e = 0; e < 8; ++e) sum += v[c][e];
    }
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float mean = sum / (float)D;
    float m2 = 0.f, dot = 0.f;
#pragma unroll
    for (int c = 0; c < CH; ++c) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            const float d = v[c][e] - mean;
            m2 = fmaf(d, d, m2);
        }
        if (probe_w) {
            const float4 w0 = __ldg(reinterpret_cast<const float4*>(probe_w) + (c * 32 + lane) * 2);
            const float4 w1 = __ldg(reinterpret_cast<const float4*>(probe_w) + (c * 32 + lane) * 2 + 1);
            dot += v[c][0] * w0.x + v[c][1] * w0.y + v[c][2] * w0.z + v[c][3] * w0.w + v[c][4] * w1.x +
                   v[c][5] * w1.y + v[c][6] * w1.z + v[c][7] * w1.w;
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        m2 += __shfl_xor_sync(0xffffffffu, m2, o);
        dot += __shfl_xor_sync(0xffffffffu, dot, o);
    }
    if (lane == 0) stats[row] = make_float2(mean, m2);
    if (probe_w && lane < D / 64) probe_p[(size_t)row * (D / 64) + lane] = lane == 0 ? dot : 0.f;
}

// =====================================================================================================
// final_layer: 3x3 conv, pad 1 (models/uvit.py:329-333,382).  in/out [B,C,H,W] fp32.
// =====================================================================================================
constexpr int CONV_BAND = 16;
// One CTA per (sample, 16-row band): the band (+1 halo row each side) of all C channels is staged in shared memory
// with 128-bit loads, then every thread produces 4 horizontally adjacent pixels of every output channel from
// registers (a 3 x 6 window per input channel) and stores them as one float4 per channel.  Requires W % 4 == 0.
// n_dev / slot_map (early-exit compaction): only the first *n_dev input images are live and image b is written to
// output slot slot_map[b].  layer_idx (grouped mode, the leavers' heads in one launch): image b uses the weights of
// head layer_idx[b] from the stacked arrays wgt [depth][C*C*9] / bias [depth][C]; images with layer_idx[b] >= depth are
// skipped.
template <int C>
__device__ __forceinline__ void conv_stage_band(float* __restrict__ conv_smem, const float* __restrict__ in, int b,
                                                int y0, int H, int W) {
    const int SW = W + 8, SH = CONV_BAND + 2;
    const int w4 = W / 4;
    // interior: rows y0-1 .. y0+16, float4 granularity; halo columns are zero
    for (int i = threadIdx.x; i < C * SH * (w4 + 2); i += blockDim.x) {
        const int q = i % (w4 + 2), r = (i / (w4 + 2)) % SH, c = i / ((w4 + 2) * SH);
        const int yy = y0 - 1 + r;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q >= 1 && q <= w4 && yy >= 0 && yy < H)
            v = __ldg(reinterpret_cast<const float4*>(in + (((size_t)b * C + c) * H + yy) * W) + (q - 1));
        *reinterpret_cast<float4*>(conv_smem + (c * SH + r) * SW + q * 4) = v;
    }
}
// output pixels (y0 + yy, 4*xq .. 4*xq+3) of every output channel; sw = [C*C*9 weights | C biases] in shared memory
template <int C>
__device__ __forceinline__ void conv_pixels4(const float* __restrict__ conv_smem, const float* __restrict__ sw, int yy,
                                             int xq, int W, float (&acc)[C][4]) {
    const int SW = W + 8, SH = CONV_BAND + 2;
#pragma unroll
    for (int co = 0; co < C; ++co) acc[co][0] = acc[co][1] = acc[co][2] = acc[co][3] = sw[C * C * 9 + co];
#pragma unroll
    for (int ci = 0; ci < C; ++ci) {
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            // smem column of pixel x is x + 4; the window needs x-1 .. x+4 -> columns 4*xq+3 .. 4*xq+8
            const float* rp = conv_smem + (ci * SH + yy + dy) * SW + 4 * xq;
            const float4 m = *reinterpret_cast<const float4*>(rp + 4);
            const float l = rp[3], r = rp[8];
            const float win[6] = {l, m.x, m.y, m.z, m.w, r};
#pragma unroll
            for (int co = 0; co < C; ++co) {
                const float* wp = sw + (co * C + ci) * 9 + dy * 3;
                const float w0 = wp[0], w1 = wp[1], w2 = wp[2];
#pragma unroll
                for (int p = 0; p < 4; ++p)
                    acc[co][p] = fmaf(w0, win[p], fmaf(w1, win[p + 1], fmaf(w2, win[p + 2], acc[co][p])));
            }
        }
    }
}
// the same four pixels of ONE output channel: per accumulator the FMA order over (ci, dy) is that of conv_pixels4, so
// both give the same bits; one channel per work item keeps the register count low enough for 3-4 CTAs per SM
template <int C>
__device__ __forceinline__ void conv_pixels4_one(const float* __restrict__ conv_smem, const float* __restrict__ sw,
                                                 int co, int yy, int xq, int W, float (&acc)[4]) {
    const int SW = W + 8, SH = CONV_BAND + 2;
    acc[0] = acc[1] = acc[2] = acc[3] = sw[C * C * 9 + co];
#pragma unroll
    for (int ci = 0; ci < C; ++ci) {
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const float* rp = conv_smem + (ci * SH + yy + dy) * SW + 4 * xq;
            const float4 m = *reinterpret_cast<const float4*>(rp + 4);
            const float l = rp[3], r = rp[8];
            const float win[6] = {l, m.x, m.y, m.z, m.w, r};
            const float* wp = sw + (co * C + ci) * 9 + dy * 3;
            const float w0 = wp[0], w1 = wp[1], w2 = wp[2];
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[p] = fmaf(w0, win[p], fmaf(w1, win[p + 1], fmaf(w2, win[p + 2], acc[p])));
        }
    }
}
template <int C>
__global__ void __launch_bounds__(256) conv3x3_kernel(const float* __restrict__ in, const float* __restrict__ wgt,
                                                      const float* __restrict__ bias, float* __restrict__ out, int H,
                                                      int W, const int* __restrict__ n_dev,
                                                      const int* __restrict__ slot_map,
                                                      const int* __restrict__ layer_idx, int depth) {
    extern __shared__ __align__(16) float conv_smem[];  // [C][CONV_BAND+2][W+8] (4 pad floats left and right)
    __shared__ float sw[C * C * 9 + C];
    const int bands = H / CONV_BAND;
    const int b = blockIdx.x / bands, y0 = (blockIdx.x % bands) * CONV_BAND;
    pdl_launch_dependents();
    if (!layer_idx)
        for (int i = threadIdx.x; i < C * C * 9 + C; i += blockDim.x)
            sw[i] = (i < C * C * 9) ? wgt[i] : bias[i - C * C * 9];
    pdl_wait();
    if (n_dev && b >= ld_state(n_dev)) return;
    if (layer_idx) {
        const int layer = ld_state(layer_idx + b);
        if (layer >= depth) return;
        for (int i = threadIdx.x; i < C * C * 9 + C; i += blockDim.x)
            sw[i] = (i < C * C * 9) ? wgt[(size_t)layer * C * C * 9 + i] : bias[layer * C + i - C * C * 9];
    }
    const int ob = slot_map ? ld_state(slot_map + b) : b;
    const int w4 = W / 4;
    conv_stage_band<C>(conv_smem, in, b, y0, H, W);
    __syncthreads();
    for (int i = threadIdx.x; i < C * CONV_BAND * w4; i += blockDim.x) {
        const int xq = i % w4, yy = (i / w4) % CONV_BAND, co = i / (w4 * CONV_BAND);
        float acc[4];
        conv_pixels4_one<C>(conv_smem, sw, co, yy, xq, W, acc);
        *(reinterpret_cast<float4*>(out + (((size_t)ob * C + co) * H + y0 + yy) * W) + xq) =
            make_float4(acc[0], acc[1], acc[2], acc[3]);
    }
}

// =====================================================================================================
// DDPM update (sampler.py:47-79, eesampler.py:74-82, ddpm_core.py:190-193), one kernel, 128-bit accesses:
//   x' = ca[t]*x + cb[t]*model_out + cs[t]*z        (z ~ N(0,I), absent at t == 0)
// The three per-timestep coefficients are tabulated on the host with the reference's own torch expressions:
//   predict_noise:    x' = sqrt(1/a)*(x - ((1-a)/sqrt(1-abar))*eps) + sigma*z is evaluated in that exact order
//   (mode 0) to stay within 1 ulp of the reference; mode 1 uses the generic two-term form for the other rules;
//   mode 2 is the DDIM update (sampler.py:112-120) with a fourth coefficient d.
// coef layout: [1000][4] = {c0, c1, sigma, d}
// Noise: injected tensor z_all[t] (parity) or Philox4x32-10 + Box-Muller keyed by (seed, t, GLOBAL float4 index): the
// index carries the shard's offset into the global batch, so N data-parallel shards draw exactly the noise a single
// process would draw for the whole batch.
// =====================================================================================================
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t (&out)[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0, c1 = n1, c2 = n2, c3 = n3;
        k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
    }
    out[0] = c0, out[1] = c1, out[2] = c2, out[3] = c3;
}
__device__ __forceinline__ void box_muller(uint32_t u0, uint32_t u1, float& n0, float& n1) {
    const float a = ((float)u0 + 0.5f) * 2.3283064365386963e-10f;  // (0,1)
    const float b = ((float)u1 + 0.5f) * 2.3283064365386963e-10f;
    const float r = sqrtf(-2.f * logf(a));
    float s, c;
    sincosf(6.283185307179586f * b, &s, &c);
    n0 = r * c, n1 = r * s;
}
// the four normals of float4 number `idx4` (global index) at timestep t
__device__ __forceinline__ float4 philox_normal4(unsigned long long idx4, int t, unsigned long long seed) {
    uint32_t r[4];
    philox4x32_10((uint32_t)idx4, (uint32_t)(idx4 >> 32), (uint32_t)t, 0x5eedu, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    float4 z;
    box_muller(r[0], r[1], z.x, z.y);
    box_muller(r[2], r[3], z.z, z.w);
    return z;
}
struct StepCoef {
    float c0, c1, sg, d;
};
__device__ __forceinline__ float ddpm_update1(int mode, const StepCoef& k, float x, float e, float z) {
    if (mode == 0)  // sqrt(1/alpha) * (x - coeff*eps) + sigma*z, evaluated like the reference (no contraction)
        return __fadd_rn(__fmul_rn(k.c0, __fsub_rn(x, __fmul_rn(k.c1, e))), __fmul_rn(k.sg, z));
    if (mode == 2)  // DDIM (sampler.py:112-120): mean = c0*(x - c1*eps); mean += d*eps; x' = mean + sigma2*z
        return __fadd_rn(__fadd_rn(__fmul_rn(k.c0, __fsub_rn(x, __fmul_rn(k.c1, e))), __fmul_rn(k.d, e)),
                         __fmul_rn(k.sg, z));
    // (c1*out + c0*x) + sigma*z   -- predict_original (sampler.py:69-72) / predict_previous (c0=0, c1=1)
    return __fadd_rn(__fadd_rn(__fmul_rn(k.c1, e), __fmul_rn(k.c0, x)), __fmul_rn(k.sg, z));
}
__device__ __forceinline__ float4 ddpm_update4(int mode, const StepCoef& k, float4 x, float4 e, float4 z) {
    return make_float4(ddpm_update1(mode, k, x.x, e.x, z.x), ddpm_update1(mode, k, x.y, e.y, z.y),
                       ddpm_update1(mode, k, x.z, e.z, z.z), ddpm_update1(mode, k, x.w, e.w, z.w));
}
// DPM-Solver++(2M), mode 3 (ddpm.dpm_solver_coefficients): row {a, b, rho, phi | w0, w1, order, 0}.  No noise term.
//   D_t = a*x + b*out;  D = w0*D_t + w1*D_prev (order 2) or D_t (order 1);  x' = rho*x + phi*D;  D_prev <- D_t
// Every operation rounded on its own (no FMA contraction), so torch elementwise ops give the same bits.  An order-1
// step never reads D_prev: a stale or uninitialised buffer cannot reach x.
struct MsCoef {
    float a, b, rho, phi, w0, w1;
};
__device__ __forceinline__ float ms_update1(const MsCoef& k, bool second, float x, float e, float dp, float& dt) {
    dt = __fadd_rn(__fmul_rn(k.a, x), __fmul_rn(k.b, e));
    const float d = second ? __fadd_rn(__fmul_rn(k.w0, dt), __fmul_rn(k.w1, dp)) : dt;
    return __fadd_rn(__fmul_rn(k.rho, x), __fmul_rn(k.phi, d));
}
__device__ __forceinline__ float4 ms_update4(const MsCoef& k, bool second, float4 x, float4 e, float4 dp, float4& dt) {
    return make_float4(ms_update1(k, second, x.x, e.x, dp.x, dt.x), ms_update1(k, second, x.y, e.y, dp.y, dt.y),
                       ms_update1(k, second, x.z, e.z, dp.z, dt.z), ms_update1(k, second, x.w, e.w, dp.w, dt.w));
}
// SDE-DPM-Solver++(2M), mode 5 (ddpm.sde_dpm_solver_coefficients): row {a, b, rho, phi | w0, w1, order, vs}.  The
// update of mode 3 with rho = (sigma_s/sigma_t) exp(-h), phi = alpha_s (-expm1(-2h)), then the noise term:
//   x' = (rho*x + phi*D) + vs*z      (vs = sigma_s sqrt(-expm1(-2h)); 0 on the final step, which adds nothing)
// z is the DDPM tail's draw at t (Philox at (seed, t, global float4 index), or the injected z_all[t]).
__device__ __forceinline__ float4 add_noise4(float4 o, float vs, float4 z) {
    return make_float4(__fadd_rn(o.x, __fmul_rn(vs, z.x)), __fadd_rn(o.y, __fmul_rn(vs, z.y)),
                       __fadd_rn(o.z, __fmul_rn(vs, z.z)), __fadd_rn(o.w, __fmul_rn(vs, z.w)));
}
// UniPC (bh2, data prediction), mode 4 (ddpm.unipc_coefficients): row {a, b, cx, c0 | c1, c2, px, p0 | p1, corr,
// pred, 0}.  No noise term.  With the history of the sampler (xb = corrected x of the previous step, D1 / D2 = the
// data predictions of the previous two steps):
//   D  = a*x + b*out
//   corrector  xc = x (corr 0);  ((cx*xb + c0*D) + c1*D1) (corr 1);  (((cx*xb + c0*D) + c1*D1) + c2*D2) (corr 2)
//   predictor  x' = px*xc + p0*D (pred 1);  (px*xc + p0*D) + p1*D1 (pred 2)
// then xb <- xc, D2 <- D1, D1 <- D.  Every operation rounded on its own.  The order columns decide what is read: a
// corrector-0 row reads no history and a corrector-1 row does not read D2 (NaN * 0 would still be NaN).
struct UniCoef {
    float a, b, cx, c0, c1, c2, px, p0, p1;
};
__device__ __forceinline__ float unipc_update1(const UniCoef& k, int corr, int pred, float x, float e, float xb,
                                               float d1, float d2, float& d, float& xc) {
    d = __fadd_rn(__fmul_rn(k.a, x), __fmul_rn(k.b, e));
    xc = x;
    if (corr >= 1) {
        xc = __fadd_rn(__fadd_rn(__fmul_rn(k.cx, xb), __fmul_rn(k.c0, d)), __fmul_rn(k.c1, d1));
        if (corr == 2) xc = __fadd_rn(xc, __fmul_rn(k.c2, d2));
    }
    const float o = __fadd_rn(__fmul_rn(k.px, xc), __fmul_rn(k.p0, d));
    return pred == 2 ? __fadd_rn(o, __fmul_rn(k.p1, d1)) : o;
}

// seed_dev (graph replay / sampler): {Philox key, float4 index of this shard's first element in the global batch}
__global__ void __launch_bounds__(256) ddpm_step_kernel(float* __restrict__ x, const float* __restrict__ model_out,
                                                        const float* __restrict__ z_all, size_t n, size_t z_stride,
                                                        const float* __restrict__ coef, const int* __restrict__ t_dev,
                                                        int t_host, int mode, unsigned long long seed,
                                                        const unsigned long long* __restrict__ seed_dev,
                                                        float* __restrict__ x_save) {
    pdl_launch_dependents();
    pdl_wait();
    const int t = t_dev ? ld_state(t_dev) : t_host;
    unsigned long long off4 = 0;
    if (seed_dev) seed = ld_state(seed_dev), off4 = ld_state(seed_dev + 1);
    const StepCoef k{coef[t * 4 + 0], coef[t * 4 + 1], coef[t * 4 + 2], coef[t * 4 + 3]};
    const size_t i4 = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i4 * 4 >= n) return;
    const float4 xv = reinterpret_cast<const float4*>(x)[i4];
    const float4 ev = reinterpret_cast<const float4*>(model_out)[i4];
    float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t > 0) zv = z_all ? reinterpret_cast<const float4*>(z_all + (size_t)t * z_stride)[i4] : philox_normal4(i4 + off4, t, seed);
    const float4 o = ddpm_update4(mode, k, xv, ev, zv);
    reinterpret_cast<float4*>(x)[i4] = o;
    if (x_save) reinterpret_cast<float4*>(x_save)[i4] = o;
}

// =====================================================================================================
// Fused tail of one sampling step (plain U-ViT path): final_layer 3x3 conv (models/uvit.py:382) -> eps, the DDPM
// update of x (sampler.py:47-79), and the HEAD of the next step: the bf16 hi|lo patch matrix of the updated x
// (patch_gather_kernel's output), the next step's time / label token rows (token_extras_kernel's output) and the
// step counter t <- next_t[t].  Replaces conv3x3 + ddpm_step + next_t + fill_t + patch_gather + token_extras (six
// launches) by one; every arithmetic expression is shared with those kernels, so the fused and the unfused step give
// the same bits.  One CTA per (sample, 16-row band), 256 threads, one work item = 4 pixels of one output channel.
// The next step may run on the other backbone (DuoDiff hand-off, sampler.py:135-136): next_late[t] selects which
// model's buffers receive the prepared head.
// =====================================================================================================
struct TailTarget {
    __nv_bfloat16* a_patch;  // [B * 256, 128] bf16: patch vectors hi | lo
    __nv_bfloat16* tokens;   // x0 [B * L, D]
    float2* stats_p;         // [B * L, D / 64]
    const float* pos;        // [L, D]
    const float* label_emb;  // [num_classes, D] or null
    const float* time_tab;   // [1000, D] time tokens after their MLP (mlp_time_embed = True) or null
    int P, D, L, extras, normalize_t, num_classes;
};
struct TailArgs {
    const float* img_pre;  // [B,C,H,W] un-patchified decoder output (input of the 3x3 conv)
    const float* conv_w;
    const float* conv_b;
    float* x;              // [B,C,H,W] in place
    const float* z_all;    // injected noise [1000, n] or null (Philox)
    const float* coef;     // [1000,4]; modes 3 and 5 (DPM-Solver++, SDE): [1000,8]; mode 4 (UniPC): [1000,12]
    int* t_dev;            // step counter (read by every CTA, advanced by the last one to finish)
    const int* next_t;     // [1000] successor table; [1000, 2000): 1 = the step after t runs on the late backbone
    const unsigned long long* seed_dev;  // {Philox key, float4 offset of the shard in the global batch}
    const long long* y;    // labels or null
    float* eps_out;        // optional [B,C,H,W]: the model output of this step (parity traces)
    float* x_save;         // optional copy of the updated x
    unsigned* ticket;      // CTA completion counter (self-resetting)
    size_t n;              // B*C*H*W
    int H, W, mode;
    // early-exit compaction (eesampler.py:62-68): image b went through the output head of layer layer_idx[b]; its conv
    // weights come from the stacked arrays grp_w [depth][C*C*9] / grp_b [depth][C] (layer_idx[b] >= depth: the full
    // model's final_layer, conv_w / conv_b)
    const int* layer_idx;
    const float* grp_w;
    const float* grp_b;
    int depth;
    TailTarget tgt[2];     // [0] early backbone, [1] late backbone
    // classifier-free guidance: the forward ran on 2B rows (row b conditional, row b + B unconditional); the tail
    // combines them into eps = c + scale * (c - u) per guided sample b < B and prepares the head of both rows
    int guide;             // 0 / 1; selects the G = true instantiation on the host
    float scale;
    int B;                 // guided samples (x, noise and traces have B rows)
    // DPM-Solver++(2M) (mode 3, K = TAIL_DPM2M) and its SDE form (mode 5, K = TAIL_SDE2M): the previous step's data
    // prediction D_prev [B,C,H,W], sampler-owned
    float* d_prev;
    // UniPC (mode 4, K = TAIL_UNIPC): d_prev is D1; the data prediction of the step before it, D2, and the corrected
    // x of the previous step, xb [B,C,H,W] each, sampler-owned
    float* d_prev2;
    float* x_base;
};
// the update a step_tail_kernel instantiation applies: DDPM / DDIM (modes 0-2), DPM-Solver++(2M) (mode 3), UniPC (4),
// SDE-DPM-Solver++(2M) (5)
enum TailKind { TAIL_DDPM = 0, TAIL_DPM2M = 1, TAIL_UNIPC = 2, TAIL_SDE2M = 3 };
// G = true: the guided tail (one CTA per guided sample b and band).  It stages two bands, rows b and b + B of img_pre,
// one after the other so that the staging needs the registers of one band; shared memory doubles (C = 4, W = 64:
// 43008 B per CTA by -Xptxas -v, so 4 CTAs still fit an SM).  G = false compiles to the same SASS as before.
// K = TAIL_DPM2M: the multistep update of mode 3 (ms_update4) replaces the DDPM / DDIM one; it reads the 8-float row
// as two float4 and D_prev (order-2 rows only) at the element the thread owns, and writes D_t there.
// K = TAIL_UNIPC: the predictor-corrector update of mode 4 (unipc_update1); it reads the 12-float row as three float4,
// and xb, D1 (corrector order >= 1) and D2 (order 2) at the element the thread owns, and writes xb, D1 and D2 there:
// 24 B per element more than the DDIM tail.  Both skip the noise.  K = TAIL_DDPM compiles to the same SASS as before.
// K = TAIL_SDE2M: the update of TAIL_DPM2M plus vs*z (mode 5).  It branches on vs, so the final step (vs = 0) neither
// reads z_all nor runs Philox; the draw and the injected-noise index are the DDPM branch's, so sharding stays exact.
template <int C, int W, bool G = false, int K = TAIL_DDPM>
__global__ void __launch_bounds__(256, 4) step_tail_kernel(const __grid_constant__ TailArgs a) {
    constexpr bool SDE = K == TAIL_SDE2M, MS = K == TAIL_DPM2M || SDE, UP = K == TAIL_UNIPC;
    constexpr int SW = W + 8, SH = CONV_BAND + 2, w4 = W / 4;
    constexpr int N_ITEMS = C * CONV_BAND * w4;          // (output channel, row, 4-pixel group) work items
    constexpr int BAND = C * SH * SW;                    // floats of one staged band
    __shared__ __align__(16) float conv_smem[(G ? 2 : 1) * BAND];
    __shared__ float sw[C * C * 9 + C];
    const int H = a.H;
    const int bands = H / CONV_BAND;
    const int b = blockIdx.x / bands, y0 = (blockIdx.x % bands) * CONV_BAND;
    pdl_launch_dependents();
    if (!a.layer_idx)
        for (int i = threadIdx.x; i < C * C * 9 + C; i += blockDim.x)
            sw[i] = (i < C * C * 9) ? a.conv_w[i] : a.conv_b[i - C * C * 9];
    pdl_wait();
    if (a.layer_idx) {  // which head the sample left through is this step's own result
        const int layer = ld_state(a.layer_idx + b);
        const float* cw = layer < a.depth ? a.grp_w + (size_t)layer * C * C * 9 : a.conv_w;
        const float* cb = layer < a.depth ? a.grp_b + layer * C : a.conv_b;
        for (int i = threadIdx.x; i < C * C * 9 + C; i += blockDim.x) sw[i] = (i < C * C * 9) ? cw[i] : cb[i - C * C * 9];
    }
    const int t = ld_state(a.t_dev);
    // everything that depends on t is requested at once (one further round trip, not three)
    const int t_next = a.next_t[t], late_next = a.next_t[1000 + t];
    constexpr int ROW = UP ? 12 : (MS ? 8 : 4);
    const float4 kc = *reinterpret_cast<const float4*>(a.coef + t * ROW);
    float4 kc2, kc3;
    if constexpr (MS || UP) kc2 = *reinterpret_cast<const float4*>(a.coef + t * ROW + 4);
    if constexpr (UP) kc3 = *reinterpret_cast<const float4*>(a.coef + t * ROW + 8);
    const unsigned long long seed = ld_state(a.seed_dev), off4 = ld_state(a.seed_dev + 1);
    // band of the decoder image (guided: row b, then row b + B): all loads of a thread are in flight before its first
    // shared-memory store
#pragma unroll 1
    for (int h = 0; h < (G ? 2 : 1); ++h) {
        const int src = h ? b + a.B : b;
        float* band = conv_smem + h * BAND;
        constexpr int N_STAGE = C * SH * (w4 + 2);  // float4 slots of the staged band (halo columns included)
        constexpr int PER = (N_STAGE + 255) / 256;
        float4 v[PER];
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int i = threadIdx.x + j * 256;
            const int q = i % (w4 + 2), r = (i / (w4 + 2)) % SH, c = i / ((w4 + 2) * SH);
            const int yy = y0 - 1 + r;
            v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (i < N_STAGE && q >= 1 && q <= w4 && yy >= 0 && yy < H)
                v[j] = __ldg(reinterpret_cast<const float4*>(a.img_pre + (((size_t)src * C + c) * H + yy) * W) + (q - 1));
        }
#pragma unroll
        for (int j = 0; j < PER; ++j) {
            const int i = threadIdx.x + j * 256;
            const int q = i % (w4 + 2), r = (i / (w4 + 2)) % SH, c = i / ((w4 + 2) * SH);
            if (i < N_STAGE) *reinterpret_cast<float4*>(band + (c * SH + r) * SW + q * 4) = v[j];
        }
    }
    const StepCoef k{kc.x, kc.y, kc.z, kc.w};
    const TailTarget& tg = a.tgt[late_next ? 1 : 0];
    const int P = tg.P, Hp = H / P, Wp = W / P;
    __syncthreads();
#pragma unroll 1
    for (int i = threadIdx.x; i < N_ITEMS; i += 256) {
        const int xq = i % w4, yy = (i / w4) % CONV_BAND, co = i / (w4 * CONV_BAND);
        const size_t e4 = ((((size_t)b * C + co) * H + y0 + yy) * W) / 4 + xq;  // float4 index inside the shard
        // x (and the injected noise) do not depend on the conv: their loads are in flight while it is computed
        const float4 xv = reinterpret_cast<const float4*>(a.x)[e4];
        float4 zv = make_float4(0.f, 0.f, 0.f, 0.f);  // MS: D_prev; UP: D1
        float4 xb = zv, d2 = zv;                       // UP
        float4 nz = zv;                                // SDE: this step's noise
        if constexpr (MS) {
            if (kc2.z == 2.f) zv = reinterpret_cast<const float4*>(a.d_prev)[e4];
            if constexpr (SDE)
                if (kc2.w != 0.f && a.z_all) nz = reinterpret_cast<const float4*>(a.z_all + (size_t)t * a.n)[e4];
        } else if constexpr (UP) {
            if (kc3.y != 0.f) {
                zv = reinterpret_cast<const float4*>(a.d_prev)[e4];
                xb = reinterpret_cast<const float4*>(a.x_base)[e4];
            }
            if (kc3.y == 2.f) d2 = reinterpret_cast<const float4*>(a.d_prev2)[e4];
        } else if (t > 0 && a.z_all) {
            zv = reinterpret_cast<const float4*>(a.z_all + (size_t)t * a.n)[e4];
        }
        float acc[4];
        conv_pixels4_one<C>(conv_smem, sw, co, yy, xq, W, acc);
        if constexpr (G) {
            // eps = c + s * (c - u), each operation rounded on its own (no FMA contraction): three torch ops give
            // the same bits
            float u[4];
            conv_pixels4_one<C>(conv_smem + BAND, sw, co, yy, xq, W, u);
#pragma unroll
            for (int p = 0; p < 4; ++p) acc[p] = __fadd_rn(acc[p], __fmul_rn(a.scale, __fsub_rn(acc[p], u[p])));
        }
        const float4 ev = make_float4(acc[0], acc[1], acc[2], acc[3]);
        float4 o;
        if constexpr (MS) {
            float4 dt;
            o = ms_update4(MsCoef{kc.x, kc.y, kc.z, kc.w, kc2.x, kc2.y}, kc2.z == 2.f, xv, ev, zv, dt);
            if constexpr (SDE) {
                if (kc2.w != 0.f) {
                    if (!a.z_all) nz = philox_normal4(e4 + off4, t, seed);
                    o = add_noise4(o, kc2.w, nz);
                }
            }
            reinterpret_cast<float4*>(a.d_prev)[e4] = dt;
        } else if constexpr (UP) {
            const UniCoef u{kc.x, kc.y, kc.z, kc.w, kc2.x, kc2.y, kc2.z, kc2.w, kc3.x};
            const int corr = (int)kc3.y, pred = (int)kc3.z;
            float4 d, xc;
            o.x = unipc_update1(u, corr, pred, xv.x, ev.x, xb.x, zv.x, d2.x, d.x, xc.x);
            o.y = unipc_update1(u, corr, pred, xv.y, ev.y, xb.y, zv.y, d2.y, d.y, xc.y);
            o.z = unipc_update1(u, corr, pred, xv.z, ev.z, xb.z, zv.z, d2.z, d.z, xc.z);
            o.w = unipc_update1(u, corr, pred, xv.w, ev.w, xb.w, zv.w, d2.w, d.w, xc.w);
            reinterpret_cast<float4*>(a.x_base)[e4] = xc;
            if (corr != 0) reinterpret_cast<float4*>(a.d_prev2)[e4] = zv;
            reinterpret_cast<float4*>(a.d_prev)[e4] = d;
        } else {
            if (t > 0 && !a.z_all) zv = philox_normal4(e4 + off4, t, seed);
            o = ddpm_update4(a.mode, k, xv, ev, zv);
        }
        reinterpret_cast<float4*>(a.x)[e4] = o;
        if (a.eps_out) reinterpret_cast<float4*>(a.eps_out)[e4] = ev;
        if (a.x_save) reinterpret_cast<float4*>(a.x_save)[e4] = o;
        // head of the next step: the updated pixels as bf16 hi | lo patch-vector entries (P = 2: two patches)
        patch_store_pair(patch_elem(tg.a_patch, b, co, y0 + yy, 4 * xq, P, Hp, Wp), o.x, o.y);
        patch_store_pair(patch_elem(tg.a_patch, b, co, y0 + yy, 4 * xq + 2, P, Hp, Wp), o.z, o.w);
        if constexpr (G) {  // the unconditional row sees the same x
            patch_store_pair(patch_elem(tg.a_patch, b + a.B, co, y0 + yy, 4 * xq, P, Hp, Wp), o.x, o.y);
            patch_store_pair(patch_elem(tg.a_patch, b + a.B, co, y0 + yy, 4 * xq + 2, P, Hp, Wp), o.z, o.w);
        }
    }
    if (y0 == 0) {  // one CTA per sample also writes the next step's time / label token rows
        write_token_extras(b, (float)t_next, a.y, tg.pos, tg.label_emb, tg.tokens, tg.stats_p, tg.D, tg.L, tg.extras,
                           tg.normalize_t, tg.num_classes,
                           tg.time_tab ? tg.time_tab + (size_t)min(max(t_next, 0), 999) * tg.D : nullptr);
        if constexpr (G)  // row b + B: a.y holds [y ; null label] (2B entries)
            write_token_extras(b + a.B, (float)t_next, a.y, tg.pos, tg.label_emb, tg.tokens, tg.stats_p, tg.D, tg.L,
                               tg.extras, tg.normalize_t, tg.num_classes,
                               tg.time_tab ? tg.time_tab + (size_t)min(max(t_next, 0), 999) * tg.D : nullptr);
    }
    // every CTA has read t above; the last one to get here advances the step counter
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(a.ticket, 1u) == gridDim.x - 1) {
            *a.t_dev = t_next;
            *a.ticket = 0u;
        }
    }
}

// step bookkeeping for graph replay: t_vec[b] = float(*t_dev) for the next forward; (*t_dev) -= 1 after a step
__global__ void fill_t_kernel(const int* __restrict__ t_dev, float* __restrict__ t_vec, int B) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B) t_vec[i] = (float)ld_state(t_dev);
}
__global__ void set_u64_kernel(unsigned long long* p, unsigned long long v) { *p = v; }
// t <- next_t[t]: the timestep sequence of the run (t-1 for DDPM, the strided DDIM schedule, ...) lives in a table
__global__ void next_t_kernel(int* t_dev, const int* __restrict__ next_t) {
    if (threadIdx.x == 0 && blockIdx.x == 0) *t_dev = next_t[ld_state(t_dev)];
}

// samples = (x + 1) / 2, NCHW -> NHWC (sampler.py:145-146)
__global__ void finalize_nhwc_kernel(const float* __restrict__ x, float* __restrict__ out, int B, int C, int H,
                                     int W) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t n = (size_t)B * C * H * W;
    if (i >= n) return;
    const int c = i % C;
    size_t r = i / C;
    const int w = r % W;
    r /= W;
    const int h = r % H;
    const int b = r / H;
    out[i] = (x[(((size_t)b * C + c) * H + h) * W + w] + 1.f) / 2.f;
}

// =====================================================================================================
// Early exit (eesampler.py:62-72): probe score per (layer, sample) = mean over tokens of the per-token sigmoid.
// =====================================================================================================
// timestep-indexed probe types (models/early_exit.py:199-202, 228-239): layer i of a forward at timestep t uses
// matrix["t"] (kind 2) or matrix["i, t"] (kind 3, row t * depth + i of the table).  grid = depth, any block size.
__global__ void probe_select_kernel(const float* __restrict__ tab_w, const float* __restrict__ tab_b,
                                    float* __restrict__ work_w, float* __restrict__ work_b, int depth, int D, int kind,
                                    const float* __restrict__ tsteps, const int* __restrict__ t_dev) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = blockIdx.x;
    int t = t_dev ? ld_state(t_dev) : (int)tsteps[0];  // int(timesteps[0]) (early_exit.py:269)
    t = min(max(t, 0), 999);
    const size_t r = kind == 2 ? (size_t)t : (size_t)t * depth + i;
    for (int k = threadIdx.x; k < D; k += blockDim.x) work_w[(size_t)i * D + k] = tab_w[r * D + k];
    if (threadIdx.x == 0) work_b[i] = tab_b[r];
}

// =====================================================================================================
// AttentionProbe (models/early_exit.py:40-80): one learned query attends over the tokens 1.. of the block input (the
// first token is dropped, :73), the pooled value goes through Linear(D,D) -> SiLU -> Linear(D,1); no sigmoid.
// Restated without the [B, L, 2D] key / value GEMM (the reference's own TODO asks for a cheaper classifier):
//   logit_l = q.(Wk x_l + bk) / sqrt(D) = u.x_l + const     u = Wk^T q / sqrt(D): the constant cancels in the softmax
//   pooled  = sum_l a_l (Wv x_l + bv) = Wv (sum_l a_l x_l) + bv                    (the weights a_l sum to one)
//   score   = w2 . SiLU(W1 pooled + b1) + b2 = w2 . SiLU(Wc xbar + bc) + b2        Wc = W1 Wv, bc = W1 bv + b1
// u sits in the probe working set, so the per-token logits arrive as the same partial dot products the MLP probes use
// (fc2 epilogue / ln_stats_kernel); u, Wc, bc are computed once at model creation by attn_probe_pack_kernel.
// =====================================================================================================
// grid = (D, 2): y == 0: row j of Wc (and bc[j]); y == 1, block 0..: u.  Parameter layouts are the state_dict's.
__global__ void __launch_bounds__(256) attn_probe_pack_kernel(const float* __restrict__ q /*[D]*/,
                                                              const float* __restrict__ wkv /*[2D, D]*/,
                                                              const float* __restrict__ bkv /*[2D]*/,
                                                              const float* __restrict__ w1 /*[D, D]*/,
                                                              const float* __restrict__ b1 /*[D]*/, int D,
                                                              float* __restrict__ u, float* __restrict__ wc,
                                                              float* __restrict__ bc) {
    const int j = blockIdx.x;
    if (blockIdx.y == 1) {  // u[j] = sum_e q[e] Wk[e][j] / sqrt(D)
        if (threadIdx.x == 0) {
            float s = 0.f;
            for (int e = 0; e < D; ++e) s = fmaf(q[e], wkv[(size_t)e * D + j], s);
            u[j] = s * rsqrtf((float)D);
        }
        return;
    }
    const float* wv = wkv + (size_t)D * D;
    for (int d = threadIdx.x; d < D; d += blockDim.x) {
        float s = 0.f;
        for (int e = 0; e < D; ++e) s = fmaf(w1[(size_t)j * D + e], wv[(size_t)e * D + d], s);
        wc[(size_t)j * D + d] = s;
    }
    if (threadIdx.x == 0) {
        float s = b1[j];
        for (int e = 0; e < D; ++e) s = fmaf(w1[(size_t)j * D + e], bkv[D + e], s);
        bc[j] = s;
    }
}
// grid = B (live samples), 256 threads, dynamic smem (L + D + 8) floats.  Fixed summation order: a sample's score does
// not depend on its position in the batch (compact == simulate bit for bit).
__global__ void __launch_bounds__(256) attn_probe_score_kernel(
    const __nv_bfloat16* __restrict__ x /*[M, D] block input*/, const float* __restrict__ pp /*[M, np] u.x partials*/,
    int np, const float* __restrict__ wc, const float* __restrict__ bc, const float* __restrict__ w2,
    const float* __restrict__ b2, int L, int D, const int* __restrict__ n_dev, float* __restrict__ score /*[B]*/) {
    extern __shared__ float ap_smem[];
    float* s_a = ap_smem;          // [L] logits -> softmax weights
    float* s_x = ap_smem + L;      // [D] pooled input row
    float* s_red = s_x + D;        // [8]
    pdl_launch_dependents();
    pdl_wait();
    const int b = blockIdx.x;
    if (n_dev && b >= ld_state(n_dev)) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    auto block_reduce = [&](float v, bool is_max) -> float {
        for (int o = 16; o > 0; o >>= 1) {
            const float w = __shfl_xor_sync(0xffffffffu, v, o);
            v = is_max ? fmaxf(v, w) : v + w;
        }
        __syncthreads();  // s_red is reused
        if (lane == 0) s_red[warp] = v;
        __syncthreads();
        float r = s_red[0];
        for (int w = 1; w < 8; ++w) r = is_max ? fmaxf(r, s_red[w]) : r + s_red[w];
        return r;
    };
    // logits of tokens 1 .. L-1 (token 0 is dropped: x[:, 1:, :], early_exit.py:73)
    float mx = -INFINITY;
    for (int l = 1 + tid; l < L; l += 256) {
        float d = 0.f;
        for (int c = 0; c < np; ++c) d += pp[((size_t)b * L + l) * np + c];
        s_a[l] = d;
        mx = fmaxf(mx, d);
    }
    mx = block_reduce(mx, true);
    float sum = 0.f;
    for (int l = 1 + tid; l < L; l += 256) {
        const float e = expf(s_a[l] - mx);
        s_a[l] = e;
        sum += e;
    }
    sum = block_reduce(sum, false);
    const float inv = 1.f / sum;
    // xbar = sum_l a_l x_l: a thread owns column pairs, rows in increasing order
    for (int c2 = tid; c2 < D / 2; c2 += 256) {
        float a0 = 0.f, a1 = 0.f;
        const uint32_t* col = reinterpret_cast<const uint32_t*>(x + (size_t)b * L * D) + c2;
        for (int l = 1; l < L; ++l) {
            const uint32_t v = col[(size_t)l * (D / 2)];
            const float w = s_a[l];
            a0 = fmaf(w, bf16_lo(v), a0);
            a1 = fmaf(w, bf16_hi(v), a1);
        }
        s_x[2 * c2] = a0 * inv, s_x[2 * c2 + 1] = a1 * inv;
    }
    __syncthreads();
    // h_j = SiLU(Wc[j] . xbar + bc[j]); score = w2 . h + b2: one warp per row j, lanes stride the columns
    float part = 0.f;
    for (int j = warp; j < D; j += 8) {
        float d = 0.f;
        for (int k = lane; k < D; k += 32) d = fmaf(wc[(size_t)j * D + k], s_x[k], d);
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        const float z = d + bc[j];
        part += w2[j] * (z / (1.f + expf(-z)));  // every lane holds the same value
    }
    const float tot = block_reduce(lane == 0 ? part : 0.f, false);
    if (tid == 0) score[b] = tot + b2[0];
}

// per-token probe output sigmoid(w.x + b) from the row's np partial dot products (fixed summation order)
__device__ __forceinline__ float probe_token(const float* __restrict__ pp, size_t row, int np, float bias) {
    float d = 0.f;
    for (int c = 0; c < np; ++c) d += pp[row * np + c];
    return 1.f / (1.f + expf(-(d + bias)));
}
// sum over the tokens l = tid, tid + stride, ... of one sample of the per-token probe outputs, in that order.  For the
// usual np (a multiple of 4, <= 16) the partials of four tokens are requested at once with 16-byte loads -- one memory
// round trip per four tokens instead of np dependent ones per token (7.5 -> 5.2 us per layer in the compaction chain);
// the additions are those of probe_token, in the same order.
__device__ __forceinline__ float probe_tokens_sum(const float* __restrict__ pp, size_t row0, int L, int np, float bias,
                                                  int tid, int stride) {
    float s = 0.f;
    if ((np & 3) == 0 && np <= 16) {
        const int n4 = np >> 2;
        for (int l0 = tid; l0 < L; l0 += 4 * stride) {
            float4 v[4][4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int l = l0 + k * stride;
                const float4* q = reinterpret_cast<const float4*>(pp + (row0 + l) * np);
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    if (l < L && c < n4) v[k][c] = q[c];
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                if (l0 + k * stride < L) {
                    float d = 0.f;
#pragma unroll
                    for (int c = 0; c < 4; ++c)
                        if (c < n4) d += v[k][c].x, d += v[k][c].y, d += v[k][c].z, d += v[k][c].w;
                    s += 1.f / (1.f + expf(-(d + bias)));
                }
            }
        }
    } else {
        for (int l = tid; l < L; l += stride) s += probe_token(pp, row0 + l, np, bias);
    }
    return s;
}
// probe partials [M, np] (one layer) -> score[b] = mean_l sigmoid(w.x_{b,l} + bias); deterministic tree order.
__global__ void __launch_bounds__(128) probe_mean_kernel(const float* __restrict__ pp, int np,
                                                         const float* __restrict__ bias_p, int L,
                                                         float* __restrict__ score /*[B]*/) {
    pdl_launch_dependents();
    pdl_wait();
    const int b = blockIdx.x;
    const float bias = bias_p[0];
    float s = probe_tokens_sum(pp, (size_t)b * L, L, np, bias, threadIdx.x, blockDim.x);
    __shared__ float red[4];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) score[b] = (red[0] + red[1] + red[2] + red[3]) / (float)L;
}

// simulate mode: scores [depth][B], heads [depth+1][B][chw] (last = full model) -> exit index + selected eps
__global__ void __launch_bounds__(256) ee_select_kernel(const float* __restrict__ scores,
                                                        const float* __restrict__ outputs, int depth, int B,
                                                        size_t chw, float threshold, float* __restrict__ eps,
                                                        int* __restrict__ exit_idx, const int* __restrict__ t_dev,
                                                        int* __restrict__ exit_log /*[1000,B] by t, or null*/) {
    const int b = blockIdx.y;
    // eesampler.py:62-67: a row of zeros is appended to the probe outputs, so "no exit" selects index `depth` whenever
    // 0 <= threshold; with a negative threshold the mask is all-false and argmax returns 0 (layer 0's head)
    int idx = (0.f <= threshold) ? depth : 0;
    for (int i = 0; i < depth; ++i) {
        if (scores[(size_t)i * B + b] <= threshold) {
            idx = i;
            break;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        exit_idx[b] = idx;
        if (exit_log) exit_log[(size_t)(t_dev ? ld_state(t_dev) : 0) * B + b] = idx;
    }
    const float4* src = reinterpret_cast<const float4*>(outputs + ((size_t)idx * B + b) * chw);
    float4* dst = reinterpret_cast<float4*>(eps + (size_t)b * chw);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < chw / 4; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src[i];
}

// =====================================================================================================
// Early-exit COMPACTION (ddb_ee_forward mode 1): samples whose probe score drops below the threshold at layer i take
// head_i's output and leave the batch, so every later kernel works on M = n_active * L rows.
// Device-side state ee_n[4] = {n_active, n_active*L, n_exit, n_exit*L}; slot[b] = original index of compact sample b.
// =====================================================================================================
// def_idx: the index of a sample that never triggers -- `depth` (the full model), or 0 when the threshold is negative
// (eesampler.py:62-67: the appended zero row only matches for 0 <= threshold; argmax over an all-false mask is 0).
__global__ void ee_reset_kernel(int* __restrict__ ee_n, int* __restrict__ slot, int B, int L,
                                float* __restrict__ scores, int depth, int def_idx, int* __restrict__ exit_idx,
                                const int* __restrict__ t_dev, int* __restrict__ exit_log) {
    pdl_launch_dependents();
    pdl_wait();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) ee_n[0] = B, ee_n[1] = B * L, ee_n[2] = 0, ee_n[3] = 0;
    if (i < B) {
        slot[i] = i;
        exit_idx[i] = def_idx;
        if (exit_log) exit_log[(size_t)(t_dev ? ld_state(t_dev) : 0) * B + i] = def_idx;
    }
    if (i < depth * B) scores[i] = __int_as_float(0x7fc00000);  // NaN: "not produced" (sample had already left)
}

// grid = B CTAs of 128 threads.  CTA b scores live sample b (mean over tokens of the probe's sigmoid, with exactly the
// summation order of probe_mean_kernel, so the exit decisions of the two modes can never differ by rounding); the LAST
// CTA to finish (atomic ticket) decides who leaves at `layer` and plans the row move.  (Round 1 scored all samples in
// one CTA: with the probe's partial dot products coming from the fc2 epilogue that is 1 MB through a single SM, 11 us
// per layer.)
// The batch is kept dense by SWAPPING, not by shifting: with n_keep samples staying, every leaver at a position
// < n_keep is a hole, and the stayers at positions >= n_keep fill the holes in order.  Only n_exit rows per buffer move
// (an order-preserving squeeze re-wrote every row behind the first leaver: all live buffers, ~0.5 GB per event at
// B = 128); the order of the samples inside the batch carries no meaning -- slot[] maps a position to the sample.
//   ee_n[0..4] = {n_active, n_active*L, n_exit, n_exit*L, n_active BEFORE this layer}
//   leaver j (in position order): ex_pos[j] = its position, exit_slot[j] = its sample index (the scratch batch is indexed
//   by sample), ex_fill[j] = position of the stayer that takes its place, or -1 (the leaver sat behind the new end)
constexpr int EE_MAX_BATCH = 1024;
__global__ void __launch_bounds__(128) ee_decide_kernel(
    const float* __restrict__ pp, int np, const float* __restrict__ bias_p, int L, float thr, int layer, int B,
    int depth, int* __restrict__ ee_n, int* __restrict__ slot, int* __restrict__ ex_pos, int* __restrict__ ex_fill,
    int* __restrict__ exit_slot, float* __restrict__ scores, int* __restrict__ exit_idx,
    const int* __restrict__ t_dev, int* __restrict__ exit_log, float* __restrict__ score_mean_log,
    float* __restrict__ sc_tmp, unsigned* __restrict__ ticket, int prescored) {
    pdl_launch_dependents();
    pdl_wait();
    __shared__ float red[4];
    __shared__ int s_pos[EE_MAX_BATCH];
    __shared__ int wtot[3][4];
    __shared__ float wsum[4];
    __shared__ int is_last;
    const int n = ld_state(ee_n);  // rewritten by the last CTA only after every CTA has passed the ticket below
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (!prescored) {  // (attention probes are scored by attn_probe_score_kernel: sc_tmp is already filled)
        const int b = blockIdx.x;
        if (b < n) {
            const float bias = bias_p[0];
            float s = probe_tokens_sum(pp, (size_t)b * L, L, np, bias, tid, 128);
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) red[warp] = s;
            __syncthreads();
            if (tid == 0) sc_tmp[b] = (red[0] + red[1] + red[2] + red[3]) / (float)L;
        }
    }
    if (tid == 0) {
        __threadfence();
        is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    // ---- decision: thread i owns positions 8i .. 8i+7 (B <= 1024)
    constexpr int PER = EE_MAX_BATCH / 128;
    float sc[PER];
    int ex[PER], myslot[PER];
    int ce = 0, ck = 0;
    float fs = 0.f;
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int b = tid * PER + u;
        const bool live = b < n;
        sc[u] = live ? __ldcg(sc_tmp + b) : 0.f;
        myslot[u] = live ? ld_state(slot + b) : 0;
        // threshold < 0 with sigmoid probes (scores in (0, 1)): nothing ever matches, argmax over the all-false mask
        // selects layer 0 for every sample (see ee_select_kernel) -- everybody leaves at once.  (Attention probes are
        // real-valued: a negative threshold is an ordinary one; the forward saves every sample's layer-0 rows and
        // makes 0 the default index instead.)
        ex[u] = (live && (sc[u] <= thr || (thr < 0.f && layer == 0 && !prescored))) ? 1 : 0;
        ce += ex[u];
        ck += (live && !ex[u]) ? 1 : 0;
        fs += sc[u];
    }
    // block-wide exclusive scan of the leavers, totals of leavers / stayers, and the sum of the live scores
    int ie = ce, tk = ck;
    for (int o = 1; o < 32; o <<= 1) {
        const int te = __shfl_up_sync(0xffffffffu, ie, o);
        if (lane >= o) ie += te;
    }
    for (int o = 16; o > 0; o >>= 1) {
        tk += __shfl_xor_sync(0xffffffffu, tk, o);
        fs += __shfl_xor_sync(0xffffffffu, fs, o);
    }
    if (lane == 31) wtot[0][warp] = ie;
    if (lane == 0) wtot[1][warp] = tk, wsum[warp] = fs;
    __syncthreads();
    int base_e = ie - ce;  // exclusive inside the warp
    for (int w = 0; w < warp; ++w) base_e += wtot[0][w];
    const int n_exit = wtot[0][0] + wtot[0][1] + wtot[0][2] + wtot[0][3];
    const int n_keep = wtot[1][0] + wtot[1][1] + wtot[1][2] + wtot[1][3];
    // movers: stayers behind the new end of the batch; second scan
    int cm = 0;
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int b = tid * PER + u;
        cm += (b < n && !ex[u] && b >= n_keep) ? 1 : 0;
    }
    int im = cm;
    for (int o = 1; o < 32; o <<= 1) {
        const int tm = __shfl_up_sync(0xffffffffu, im, o);
        if (lane >= o) im += tm;
    }
    if (lane == 31) wtot[2][warp] = im;
    const int t_now = t_dev ? ld_state(t_dev) : 0;
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int b = tid * PER + u;
        if (b >= n) break;
        scores[(size_t)layer * B + myslot[u]] = sc[u];
        if (ex[u]) {
            const int j = base_e++;
            s_pos[j] = b;
            ex_pos[j] = b;
            if (b >= n_keep) ex_fill[j] = -1;  // (the holes' entries are written by the movers below)
            exit_slot[j] = myslot[u];
            exit_idx[myslot[u]] = layer;
            if (exit_log) exit_log[(size_t)t_now * B + myslot[u]] = layer;
        }
    }
    __syncthreads();
    int base_m = im - cm;
    for (int w = 0; w < warp; ++w) base_m += wtot[2][w];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
        const int b = tid * PER + u;
        if (b < n && !ex[u] && b >= n_keep) {
            const int q = base_m++;  // the q-th mover takes the q-th hole (holes = the leavers at positions < n_keep)
            ex_fill[q] = b;
            slot[s_pos[q]] = myslot[u];
        }
    }
    if (tid == 0) {
        ee_n[0] = n_keep, ee_n[1] = n_keep * L, ee_n[2] = n_exit, ee_n[3] = n_exit * L, ee_n[4] = n;
        // eesampler.py:71 logs the batch mean of every probe; here: the mean over the samples still in the batch
        if (score_mean_log)
            score_mean_log[(size_t)t_now * depth + layer] =
                n > 0 ? (wsum[0] + wsum[1] + wsum[2] + wsum[3]) / (float)n : __int_as_float(0x7fc00000);
        *ticket = 0u;
    }
}

// One kernel moves the rows after a decision, in every live activation buffer (the block input bufs.p[0] and the
// pending long skips): per leaver, its row of the block input goes to the scratch batch xe for its exit head (indexed by
// the sample, so the leavers of all layers collect there and one grouped decode serves them at the end of the forward),
// and the stayer ex_fill[j] -- if any -- is copied into its place.  blockIdx.y == nbuf does the same for the rows'
// LayerNorm statistics (np float2 each).  grid = (EE_MOVE_GRID, nbuf + 1): a CTA walks the tokens l = blockIdx.x,
// + gridDim.x, ... of every moved row (a small grid: at most layers nobody leaves and the launch is a no-op whose cost
// is draining its CTAs); a work item is one 16-byte chunk.  Sources (positions >= n_keep) and destinations (< n_keep) are disjoint, and the thread that
// overwrites a hole is the one that saved its old content first.  256 threads x 8 work items per round keep enough
// loads in flight for the big events (most of a 128-sample batch leaving at one layer: 67 MB through one launch).
constexpr int EE_MAX_LIVE = 16;
constexpr int EE_MOVE_GRID = 64;
struct EeBufList {
    __nv_bfloat16* p[EE_MAX_LIVE];
};
// s_pos / s_fill / s_slot: the CTA's shared-memory copy of the plan (one L2 round trip per CTA instead of three
// dependent ones per work item)
template <typename T>
__device__ __forceinline__ void ee_move_rows(T* buf, T* scratch, int chunks, const int* s_pos, const int* s_fill,
                                             const int* s_slot, int n_exit, int L, int l) {
    constexpr int NB = 8;  // work items per thread and round: up to 16 loads in flight, then the stores
    const int total = n_exit * chunks;
    for (int i0 = threadIdx.x; i0 < total; i0 += NB * blockDim.x) {
        T hv[NB], fv[NB];
        int pos[NB], fill[NB], cc[NB], jj[NB];
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            const int i = i0 + u * blockDim.x;
            fill[u] = -1, pos[u] = -1;
            if (i < total) {
                jj[u] = i / chunks, cc[u] = i - jj[u] * chunks;
                pos[u] = s_pos[jj[u]], fill[u] = s_fill[jj[u]];
                if (scratch) hv[u] = buf[((size_t)pos[u] * L + l) * chunks + cc[u]];
                if (fill[u] >= 0) fv[u] = buf[((size_t)fill[u] * L + l) * chunks + cc[u]];
            }
        }
#pragma unroll
        for (int u = 0; u < NB; ++u) {
            if (pos[u] < 0) continue;
            if (scratch) scratch[((size_t)s_slot[jj[u]] * L + l) * chunks + cc[u]] = hv[u];
            if (fill[u] >= 0) buf[((size_t)pos[u] * L + l) * chunks + cc[u]] = fv[u];
        }
    }
}
__global__ void __launch_bounds__(256) ee_move_kernel(const __grid_constant__ EeBufList bufs, int nbuf,
                                                      __nv_bfloat16* __restrict__ xe, float2* __restrict__ stats,
                                                      float2* __restrict__ stats_e, int np,
                                                      const int* __restrict__ ee_n, const int* __restrict__ ex_pos,
                                                      const int* __restrict__ ex_fill,
                                                      const int* __restrict__ exit_slot, int L, int D) {
    __shared__ int s_pos[EE_MAX_BATCH], s_fill[EE_MAX_BATCH], s_slot[EE_MAX_BATCH];
    pdl_launch_dependents();
    pdl_wait();
    const int n_exit = ld_state(ee_n + 2);
    if (n_exit == 0) return;  // nobody left at this layer
    const bool is_stats = (int)blockIdx.y == nbuf;
    const bool to_scratch = is_stats || blockIdx.y == 0;
    bool any_fill = false;
    for (int j = threadIdx.x; j < n_exit; j += blockDim.x) {
        s_pos[j] = ld_state(ex_pos + j), s_slot[j] = ld_state(exit_slot + j);
        const int f = ld_state(ex_fill + j);
        s_fill[j] = f;
        any_fill |= f >= 0;
    }
    // a skip buffer with no hole to fill has nothing to do (e.g. the whole batch left)
    if (!__syncthreads_or(any_fill) && !to_scratch) return;
    for (int l = blockIdx.x; l < L; l += gridDim.x) {
        if (is_stats)
            ee_move_rows<float2>(stats, stats_e, np, s_pos, s_fill, s_slot, n_exit, L, l);
        else
            ee_move_rows<uint4>(reinterpret_cast<uint4*>(bufs.p[blockIdx.y]),
                                blockIdx.y == 0 ? reinterpret_cast<uint4*>(xe) : nullptr, D / 8, s_pos, s_fill, s_slot,
                                n_exit, L, l);
    }
}

}  // namespace ddb
