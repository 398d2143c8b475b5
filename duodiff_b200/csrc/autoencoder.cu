// KL-autoencoder decoder (FrozenAutoencoderKL.decode, models/utils/autoencoder.py:486-490 -> Decoder.forward :416-449)
// and encoder (FrozenAutoencoderKL.encode_moments / sample / encode -> Encoder.forward): host side of the ddb_ae_*
// entry points.  Each direction is compiled once into a flat list of kernel launches ("ops") over a handful of NHWC
// bf16 buffers; ddb_ae_decode / ddb_ae_encode_moments replay the list per chunk of max_batch samples.  The encoder
// plan is optional (ddb_ae_create_encoder) and reuses the decoder's activation, GroupNorm and AttnBlock workspace.
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "conv_gemm.cuh"
#include "host_common.h"

using namespace ddb;
using ddb_host::failf;

#define CUDA_TRY(expr)                                                                                              \
    do {                                                                                                            \
        cudaError_t _e = (expr);                                                                                    \
        if (_e != cudaSuccess)                                                                                      \
            return failf(DDB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    } while (0)
#define DDB_TRY(expr)                \
    do {                             \
        int _r = (expr);             \
        if (_r != DDB_OK) return _r; \
    } while (0)
#define LAUNCH_CHECK()                                                                                            \
    do {                                                                                                          \
        ddb_host::count_launch();                                                                                 \
        cudaError_t _e = cudaGetLastError();                                                                      \
        if (_e != cudaSuccess)                                                                                    \
            return failf(DDB_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__,      \
                         __LINE__);                                                                               \
    } while (0)

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    ~DevBuf() {
        if (p) cudaFree(p);
    }
};
typedef std::unique_ptr<DevBuf> Buf;

int new_buf(Buf& b, size_t bytes, bool zero = false) {
    b.reset(new DevBuf);
    if (bytes == 0) bytes = 16;
    CUDA_TRY(cudaMalloc(&b->p, bytes));
    b->bytes = bytes;
    if (zero) CUDA_TRY(cudaMemset(b->p, 0, bytes));
    return DDB_OK;
}

// Workspace both plans use (AttnBlock buffers): allocated by the first plan, reused by the second -- its address is
// baked into the first plan's tensor maps, so it must never be reallocated.
int shared_buf(Buf& b, size_t bytes, bool zero = false) {
    if (!b) return new_buf(b, bytes, zero);
    if (b->bytes < bytes)
        return failf(DDB_ERR_INVALID, "autoencoder: encoder needs %zu bytes of attention workspace, the decoder has %zu",
                     bytes, b->bytes);
    return DDB_OK;
}

typedef std::map<std::string, const ddb_tensor*> TensorMap;
int get_tensor(const TensorMap& tm, const std::string& name, int64_t numel, const float** out) {
    auto it = tm.find(name);
    if (it == tm.end()) return failf(DDB_ERR_MISSING_KEY, "state_dict key '%s' missing", name.c_str());
    if (numel >= 0 && it->second->numel != numel)
        return failf(DDB_ERR_SHAPE, "state_dict key '%s' has %lld elements, expected %lld", name.c_str(),
                     (long long)it->second->numel, (long long)numel);
    *out = it->second->data_dev;
    return DDB_OK;
}

enum OpKind { OP_PREP, OP_CONV, OP_GN_FINALIZE, OP_GN_APPLY, OP_TRANSPOSE_V, OP_SOFTMAX, OP_IM2COL };
enum AeCat { AC_CONV3 = 0, AC_CONV_UP, AC_CONV1, AC_ATTN_MM, AC_GN, AC_OTHER, AC_COUNT };

struct Op {
    OpKind kind;
    int cat = AC_OTHER;
    std::string name;
    // what the op leaves behind (debug dumps / parity of intermediates)
    const void* out = nullptr;
    int out_C = 0, out_H = 0, out_W = 0, out_f32 = 0;  // per-sample [H, W, C] (NHWC) unless noted by the name
    // OP_CONV
    ConvArgs conv;
    int BN = 0, epi = 0;
    double flops_per_sample = 0;
    // OP_GN_FINALIZE
    const float2* part = nullptr;
    int slots = 0, C = 0, cpg = 0;
    float count = 0;
    const float *gamma = nullptr, *beta = nullptr;
    // OP_GN_APPLY
    const __nv_bfloat16* x = nullptr;
    __nv_bfloat16* y = nullptr;
    int HW = 0, swish = 0;
    // OP_TRANSPOSE_V / OP_SOFTMAX
    int T = 0, pitch = 0, v_off = 0;
    const float* S = nullptr;
};

struct ConvW {
    Buf w, bias;
    int N = 0, N_pad = 0, ktot = 0, nw = 1;
};

}  // namespace

struct ddb_ae {
    ddb_ae_config cfg;
    int num_sms = 0;
    int zres = 0, maxB = 0;
    std::vector<Buf> keep;
    std::vector<std::unique_ptr<ConvW>> convs;
    Buf pq_w, pq_b;
    Buf zin;                // [maxB, zres, zres, 64] bf16
    Buf act[4];             // activation ring
    Buf part[3];            // GroupNorm partials ring
    Buf affine;             // [maxB, Cmax] float2
    Buf qkv, vT, S, P, O;   // AttnBlock workspace
    Buf zero_bias;          // bias of the plain matrix products (the conv epilogue always adds one)
    std::vector<Op> ops;
    std::vector<Op> enc_ops;  // encoder plan (empty until ddb_ae_create_encoder)
    int enc_in_ch = 0;        // encoder in_channels (from encoder.conv_in.weight)
    float2* affine_p() const { return reinterpret_cast<float2*>(affine->p); }
};

namespace {

int tmap_act(CUtensorMap* tm, const void* base, int C, int pitch, int W, int H, int B, int BW, int BH) {
    const unsigned long long dims[4] = {(unsigned long long)C, (unsigned long long)W, (unsigned long long)H,
                                        (unsigned long long)B};
    const unsigned long long str[3] = {(unsigned long long)pitch * 2, (unsigned long long)W * pitch * 2,
                                       (unsigned long long)H * W * pitch * 2};
    const unsigned box[4] = {64, (unsigned)BW, (unsigned)BH, 1};
    return ddb_host::encode_bf16_sw128(tm, base, 4, dims, str, box);
}
int tmap_w(CUtensorMap* tm, const void* base, int K, int pitch, int N, int nw, size_t set_stride_elems, int BN) {
    const unsigned long long dims[3] = {(unsigned long long)K, (unsigned long long)N, (unsigned long long)nw};
    const unsigned long long str[2] = {(unsigned long long)pitch * 2, (unsigned long long)set_stride_elems * 2};
    const unsigned box[3] = {64, (unsigned)BN, 1};
    return ddb_host::encode_bf16_sw128(tm, base, 3, dims, str, box);
}
int tmap_2d(CUtensorMap* tm, const void* base, size_t rows, int cols) {
    const unsigned long long dims[2] = {(unsigned long long)cols, (unsigned long long)rows};
    const unsigned long long str[1] = {(unsigned long long)cols * 2};
    const unsigned box[2] = {64, 128};
    return ddb_host::encode_bf16_sw128(tm, base, 2, dims, str, box);
}
// high-resolution output of the fused upsample convolution: {N, px, x, py, b*H + y}
int tmap_subpixel(CUtensorMap* tm, const void* base, int N, int W, int H, int B, int BW, int BH) {
    const unsigned long long dims[5] = {(unsigned long long)N, 2ull, (unsigned long long)W, 2ull,
                                        (unsigned long long)B * H};
    const unsigned long long str[4] = {(unsigned long long)N * 2, (unsigned long long)N * 4,
                                       (unsigned long long)W * N * 4, (unsigned long long)W * N * 8};
    const unsigned box[5] = {64, 1, (unsigned)BW, 1, (unsigned)BH};
    return ddb_host::encode_bf16_sw128(tm, base, 5, dims, str, box);
}

// stride-2 source of the Downsample conv, NHWC [B, 2H, 2W, C] viewed as {(q, c), x, p, y, b} with source pixel
// (2y + p, 2x + q); H, W: the output grid
int tmap_stride2(CUtensorMap* tm, const void* base, int C, int W, int H, int B, int BW, int BH) {
    const unsigned long long dims[5] = {2ull * C, (unsigned long long)W, 2ull, (unsigned long long)H,
                                        (unsigned long long)B};
    const unsigned long long str[4] = {4ull * C, 4ull * W * C, 8ull * W * C, 8ull * H * W * C};
    const unsigned box[5] = {64, (unsigned)BW, 1, (unsigned)BH, 1};
    return ddb_host::encode_bf16_sw128(tm, base, 5, dims, str, box);
}

int pick_bn(int N) { return (N % 256 == 0) ? 256 : (N % 128 == 0 ? 128 : 64); }

int tile_shape(int H, int W, int* BW, int* BH) {
    if (W < 16 || (W & (W - 1))) return failf(DDB_ERR_INVALID, "autoencoder: feature-map width %d must be a power of two >= 16", W);
    *BW = W < 128 ? W : 128;
    *BH = 128 / *BW;
    if (H % *BH) return failf(DDB_ERR_INVALID, "autoencoder: feature-map height %d not a multiple of %d", H, *BH);
    return DDB_OK;
}

template <int BN, int EPI, int MT = 1>
int launch_conv_t(const ConvArgs& a, int num_sms, cudaStream_t st) {
    static ddb_host::DeviceOnce configured;
    auto kfn = conv_igemm_kernel<BN, EPI, MT>;
    if (!configured.done()) {
        CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, ConvCfg<BN, MT>::SMEM_BYTES));
        configured.mark();
    }
    const long long units = (long long)a.B * ((a.H * a.W) >> 7) * (a.subpixel ? 4 : 1) / MT * (a.N / BN);
    const int grid = units < num_sms ? (int)units : num_sms;
    if (grid <= 0) return DDB_OK;
    CUDA_TRY(ddb_host::launch_pdl(kfn, dim3(grid), dim3(384), (size_t)ConvCfg<BN, MT>::SMEM_BYTES, st, a));
    LAUNCH_CHECK();
    return DDB_OK;
}

int g_conv_mt2 = 1;  // two pixel tiles per work unit for the N = 128 layers (conv_gemm.cuh, MT)

int launch_conv(const ConvArgs& a, int BN, int epi, int num_sms, cudaStream_t st) {
    // N = 128: two pixel tiles share each weight tile (less shared-memory fill per MMA); needs an even tile count
    if (g_conv_mt2 && BN == 128 && !a.subpixel && ((a.B * ((a.H * a.W) >> 7)) % 2 == 0)) {
        if (epi == CEPI_BIAS) return launch_conv_t<128, CEPI_BIAS, 2>(a, num_sms, st);
        if (epi == CEPI_RES) return launch_conv_t<128, CEPI_RES, 2>(a, num_sms, st);
    }
#define CONV_CASE(bn, e) \
    if (BN == bn && epi == e) return launch_conv_t<bn, e>(a, num_sms, st);
    CONV_CASE(256, CEPI_BIAS) CONV_CASE(256, CEPI_RES) CONV_CASE(256, CEPI_F32)
    CONV_CASE(128, CEPI_BIAS) CONV_CASE(128, CEPI_RES) CONV_CASE(128, CEPI_F32)
    CONV_CASE(64, CEPI_BIAS) CONV_CASE(64, CEPI_RES) CONV_CASE(64, CEPI_F32) CONV_CASE(64, CEPI_IMG)
#undef CONV_CASE
    return failf(DDB_ERR_INVALID, "no conv kernel for BN=%d epilogue=%d", BN, epi);
}

// --------------------------------------------------------------------------------------------------- plan builder
struct Builder {
    ddb_ae* ae;
    const TensorMap& tm;
    int B;                 // max chunk
    std::vector<Op>& ops;  // the plan being built (decoder or encoder)
    int part_next = 0;

    float2* next_part() {
        float2* p = reinterpret_cast<float2*>(ae->part[part_next]->p);
        part_next = (part_next + 1) % 3;
        return p;
    }

    // pack a Conv2d (plus an optional 1x1 K-extension) into the kernel's weight layout
    int pack(const std::string& key, int N, int C, int k, int C_pad, const std::string& ext_key, int C1, bool subpixel,
             ConvW** out) {
        std::unique_ptr<ConvW> cw(new ConvW);
        const float *w, *b, *w1 = nullptr, *b1 = nullptr;
        DDB_TRY(get_tensor(tm, key + ".weight", (int64_t)N * C * k * k, &w));
        DDB_TRY(get_tensor(tm, key + ".bias", N, &b));
        if (C1 > 0) {
            DDB_TRY(get_tensor(tm, ext_key + ".weight", (int64_t)N * C1, &w1));
            DDB_TRY(get_tensor(tm, ext_key + ".bias", N, &b1));
        }
        const int taps = subpixel ? 4 : k * k;
        cw->N = N, cw->N_pad = (N + 63) / 64 * 64, cw->ktot = taps * C_pad + C1, cw->nw = subpixel ? 4 : 1;
        DDB_TRY(new_buf(cw->w, (size_t)cw->nw * cw->N_pad * cw->ktot * 2, true));
        DDB_TRY(new_buf(cw->bias, (size_t)cw->N_pad * 4, true));
        for (int s = 0; s < cw->nw; ++s) {
            __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(cw->w->p) + (size_t)s * cw->N_pad * cw->ktot;
            pack_conv_kernel<<<cw->N_pad, 256>>>(w, N, C, k, k, cw->N_pad, C_pad, cw->ktot, 0, subpixel ? s + 1 : 0, dst);
            LAUNCH_CHECK();
            if (C1 > 0) {
                pack_conv_kernel<<<cw->N_pad, 256>>>(w1, N, C1, 1, 1, cw->N_pad, C1, cw->ktot, taps * C_pad, 0, dst);
                LAUNCH_CHECK();
            }
        }
        add_bias_kernel<<<(cw->N_pad + 255) / 256, 256>>>(b, b1, N, cw->N_pad, reinterpret_cast<float*>(cw->bias->p));
        LAUNCH_CHECK();
        *out = cw.get();
        ae->convs.push_back(std::move(cw));
        return DDB_OK;
    }

    int gn_params(const std::string& key, int C, const float** g, const float** b) {
        const float *gs, *bs;
        DDB_TRY(get_tensor(tm, key + ".weight", C, &gs));
        DDB_TRY(get_tensor(tm, key + ".bias", C, &bs));
        Buf gb, bb;
        DDB_TRY(new_buf(gb, (size_t)C * 4));
        DDB_TRY(new_buf(bb, (size_t)C * 4));
        CUDA_TRY(cudaMemcpy(gb->p, gs, (size_t)C * 4, cudaMemcpyDeviceToDevice));
        CUDA_TRY(cudaMemcpy(bb->p, bs, (size_t)C * 4, cudaMemcpyDeviceToDevice));
        *g = reinterpret_cast<const float*>(gb->p), *b = reinterpret_cast<const float*>(bb->p);
        ae->keep.push_back(std::move(gb));
        ae->keep.push_back(std::move(bb));
        return DDB_OK;
    }

    // GroupNorm(32, C) [+ swish]: partials -> per-(sample, channel) affine -> elementwise pass
    int add_gn(const std::string& name, const std::string& key, const float2* part, int slots, const void* x, void* y,
               int C, int H, int W, bool swish) {
        if (C % 64) return failf(DDB_ERR_INVALID, "autoencoder: channel count %d must be a multiple of 64", C);
        Op f;
        f.kind = OP_GN_FINALIZE, f.cat = AC_GN, f.name = name + ".stats";
        f.part = part, f.slots = slots, f.C = C, f.cpg = C / 32, f.count = (float)((double)H * W * (C / 32));
        DDB_TRY(gn_params(key, C, &f.gamma, &f.beta));
        ops.push_back(f);
        Op a;
        a.kind = OP_GN_APPLY, a.cat = AC_GN, a.name = name;
        a.x = reinterpret_cast<const __nv_bfloat16*>(x), a.y = reinterpret_cast<__nv_bfloat16*>(y);
        a.HW = H * W, a.C = C, a.swish = swish;
        a.out = y, a.out_C = C, a.out_H = H, a.out_W = W;
        ops.push_back(a);
        return DDB_OK;
    }

    // generic convolution / matmul op.  src1/C1: 1x1 K-extension; res: residual [M, N]; gn_part: partials of the output
    int add_conv(const std::string& name, int cat, const ConvW* cw, const void* src0, int C0, int pitch0, int H, int W,
                 int k, bool subpixel, const void* src1, int C1, const void* res, void* out, float2* gn_part) {
        Op o;
        o.kind = OP_CONV, o.cat = cat, o.name = name;
        ConvArgs& a = o.conv;
        memset(&a, 0, sizeof(a));
        a.B = B, a.H = H, a.W = W, a.C0 = C0, a.C1 = C1, a.N = cw->N_pad;
        DDB_TRY(tile_shape(H, W, &a.BW, &a.BH));
        if (C0 % 64 || C1 % 64) return failf(DDB_ERR_INVALID, "autoencoder: %s has %d/%d input channels (need multiples of 64)", name.c_str(), C0, C1);
        a.subpixel = subpixel ? 1 : 0;
        a.wmode = subpixel ? 2 : 0;
        if (subpixel) a.tw = 2, a.taps = 4;
        else a.tw = k, a.taps = k * k, a.dy0 = a.dx0 = -(k / 2);
        a.bias = reinterpret_cast<const float*>(cw->bias->p);
        a.gn_part = gn_part, a.cpg = cw->N_pad / 32;
        if (gn_part && (cw->N_pad % 64 || cw->N_pad / 32 > 64)) return failf(DDB_ERR_INVALID, "autoencoder: GroupNorm over %d channels unsupported", cw->N_pad);
        o.BN = pick_bn(cw->N_pad);
        o.epi = res ? CEPI_RES : CEPI_BIAS;
        DDB_TRY(tmap_act(&a.tmA0, src0, C0, pitch0, W, H, B, a.BW, a.BH));
        if (C1 > 0) DDB_TRY(tmap_act(&a.tmA1, src1, C1, C1, W, H, B, a.BW, a.BH));
        DDB_TRY(tmap_w(&a.tmB, cw->w->p, cw->ktot, cw->ktot, cw->N_pad, cw->nw, (size_t)cw->N_pad * cw->ktot, o.BN));
        const int oh = subpixel ? 2 * H : H, ow = subpixel ? 2 * W : W;
        if (out && subpixel) DDB_TRY(tmap_subpixel(&a.tmOut, out, cw->N_pad, W, H, B, a.BW, a.BH));
        else if (out) DDB_TRY(tmap_2d(&a.tmOut, out, (size_t)B * H * W, cw->N_pad));
        if (res) DDB_TRY(tmap_2d(&a.tmRes, res, (size_t)B * H * W, cw->N_pad));
        o.out = out, o.out_C = cw->N_pad, o.out_H = oh, o.out_W = ow;
        o.flops_per_sample = 2.0 * (double)oh * ow * cw->N * ((subpixel ? 9.0 : (double)k * k) * C0 + C1);
        ops.push_back(o);
        return DDB_OK;
    }

    // ResnetBlock.forward (autoencoder.py:116-137, temb = None): x in `X` with its partials `px`; result in `Y`
    int add_resblock(const std::string& name, const std::string& key, int Cin, int Cout, int H, int W, void* X,
                     const float2* px, int px_slots, void* T1, void* T2, void* Y, float2** py) {
        DDB_TRY(add_gn(name + ".norm1", key + ".norm1", px, px_slots, X, T1, Cin, H, W, true));
        ConvW *c1, *c2;
        DDB_TRY(pack(key + ".conv1", Cout, Cin, 3, Cin, "", 0, false, &c1));
        float2* p2 = next_part();
        const int slots = (H * W) >> 7;
        DDB_TRY(add_conv(name + ".conv1", AC_CONV3, c1, T1, Cin, Cin, H, W, 3, false, nullptr, 0, nullptr, T2, p2));
        DDB_TRY(add_gn(name + ".norm2", key + ".norm2", p2, slots, T2, T1, Cout, H, W, true));
        *py = next_part();
        if (Cin != Cout) {
            if (tm.count(key + ".conv_shortcut.weight")) return failf(DDB_ERR_INVALID, "autoencoder: conv_shortcut ResnetBlocks are not supported (%s)", key.c_str());
            DDB_TRY(pack(key + ".conv2", Cout, Cout, 3, Cout, key + ".nin_shortcut", Cin, false, &c2));
            DDB_TRY(add_conv(name + ".conv2+nin", AC_CONV3, c2, T1, Cout, Cout, H, W, 3, false, X, Cin, nullptr, Y, *py));
        } else {
            DDB_TRY(pack(key + ".conv2", Cout, Cout, 3, Cout, "", 0, false, &c2));
            DDB_TRY(add_conv(name + ".conv2+res", AC_CONV3, c2, T1, Cout, Cout, H, W, 3, false, nullptr, 0, X, Y, *py));
        }
        return DDB_OK;
    }

    // AttnBlock.forward (autoencoder.py:165-189): single head over T = H*W tokens of dimension C
    int add_attn(const std::string& name, const std::string& key, int C, int H, int W, void* X, const float2* px,
                 int px_slots, void* T1, void* Y, float2** py) {
        const int T = H * W;
        if (T % 128 || C % 64) return failf(DDB_ERR_INVALID, "autoencoder: AttnBlock over %d tokens x %d channels unsupported", T, C);
        DDB_TRY(add_gn(name + ".norm", key + ".norm", px, px_slots, X, T1, C, H, W, false));
        // q, k, v as one 1x1 convolution with N = 3C
        std::unique_ptr<ConvW> cw(new ConvW);
        cw->N = 3 * C, cw->N_pad = 3 * C, cw->ktot = C, cw->nw = 1;
        DDB_TRY(new_buf(cw->w, (size_t)3 * C * C * 2));
        DDB_TRY(new_buf(cw->bias, (size_t)3 * C * 4));
        const char* names[3] = {".q", ".k", ".v"};
        for (int i = 0; i < 3; ++i) {
            const float *w, *b;
            DDB_TRY(get_tensor(tm, key + names[i] + ".weight", (int64_t)C * C, &w));
            DDB_TRY(get_tensor(tm, key + names[i] + ".bias", C, &b));
            pack_conv_kernel<<<C, 256>>>(w, C, C, 1, 1, C, C, C, 0, 0, reinterpret_cast<__nv_bfloat16*>(cw->w->p) + (size_t)i * C * C);
            LAUNCH_CHECK();
            CUDA_TRY(cudaMemcpy(reinterpret_cast<float*>(cw->bias->p) + i * C, b, (size_t)C * 4, cudaMemcpyDeviceToDevice));
        }
        ConvW* qkv_w = cw.get();
        ae->convs.push_back(std::move(cw));
        DDB_TRY(shared_buf(ae->qkv, (size_t)B * T * 3 * C * 2));
        DDB_TRY(shared_buf(ae->vT, (size_t)B * C * T * 2));
        DDB_TRY(shared_buf(ae->S, (size_t)B * T * T * 4));
        DDB_TRY(shared_buf(ae->P, (size_t)B * T * T * 2));
        DDB_TRY(shared_buf(ae->O, (size_t)B * T * C * 2));
        DDB_TRY(add_conv(name + ".qkv", AC_CONV1, qkv_w, T1, C, C, H, W, 1, false, nullptr, 0, nullptr, ae->qkv->p, nullptr));
        {
            Op t;
            t.kind = OP_TRANSPOSE_V, t.cat = AC_OTHER, t.name = name + ".vT";
            t.T = T, t.C = C, t.pitch = 3 * C, t.v_off = 2 * C;
            t.out = ae->vT->p, t.out_C = T, t.out_H = 1, t.out_W = C;
            ops.push_back(t);
        }
        {   // S[b] = q[b] k[b]^T / sqrt(C)   (autoencoder.py:174-181)
            Op o;
            o.kind = OP_CONV, o.cat = AC_ATTN_MM, o.name = name + ".scores";
            ConvArgs& a = o.conv;
            memset(&a, 0, sizeof(a));
            a.B = B, a.H = H, a.W = W, a.C0 = C, a.N = T;
            DDB_TRY(tile_shape(H, W, &a.BW, &a.BH));
            a.tw = 1, a.taps = 1, a.wmode = 1;
            a.out_f32 = reinterpret_cast<float*>(ae->S->p), a.scale = 1.0f / sqrtf((float)C);
            o.BN = pick_bn(T), o.epi = CEPI_F32;
            DDB_TRY(tmap_act(&a.tmA0, ae->qkv->p, C, 3 * C, W, H, B, a.BW, a.BH));
            DDB_TRY(tmap_w(&a.tmB, reinterpret_cast<__nv_bfloat16*>(ae->qkv->p) + C, C, 3 * C, T, B, (size_t)T * 3 * C, o.BN));
            o.out = ae->S->p, o.out_C = T, o.out_H = H, o.out_W = W, o.out_f32 = 1;
            o.flops_per_sample = 2.0 * T * T * C;
            ops.push_back(o);
        }
        {
            Op s;
            s.kind = OP_SOFTMAX, s.cat = AC_OTHER, s.name = name + ".softmax";
            s.S = reinterpret_cast<const float*>(ae->S->p), s.T = T;
            s.out = ae->P->p, s.out_C = T, s.out_H = H, s.out_W = W;
            ops.push_back(s);
        }
        {   // O[b] = P[b] v[b]   (autoencoder.py:183-187)
            Op o;
            o.kind = OP_CONV, o.cat = AC_ATTN_MM, o.name = name + ".pv";
            ConvArgs& a = o.conv;
            memset(&a, 0, sizeof(a));
            a.B = B, a.H = H, a.W = W, a.C0 = T, a.N = C;
            DDB_TRY(tile_shape(H, W, &a.BW, &a.BH));
            a.tw = 1, a.taps = 1, a.wmode = 1;
            o.BN = pick_bn(C), o.epi = CEPI_BIAS;
            DDB_TRY(shared_buf(ae->zero_bias, (size_t)C * 4, true));
            a.bias = reinterpret_cast<const float*>(ae->zero_bias->p);
            DDB_TRY(tmap_act(&a.tmA0, ae->P->p, T, T, W, H, B, a.BW, a.BH));
            DDB_TRY(tmap_w(&a.tmB, ae->vT->p, T, T, C, B, (size_t)C * T, o.BN));
            DDB_TRY(tmap_2d(&a.tmOut, ae->O->p, (size_t)B * T, C));
            o.out = ae->O->p, o.out_C = C, o.out_H = H, o.out_W = W;
            o.flops_per_sample = 2.0 * T * T * C;
            ops.push_back(o);
        }
        ConvW* proj;
        DDB_TRY(pack(key + ".proj_out", C, C, 1, C, "", 0, false, &proj));
        *py = next_part();
        DDB_TRY(add_conv(name + ".proj_out+res", AC_CONV1, proj, ae->O->p, C, C, H, W, 1, false, nullptr, 0, X, Y, *py));
        return DDB_OK;
    }
};

int ae_create_impl(const ddb_ae_config* cfg, const ddb_tensor* tensors, int n_tensors, ddb_ae* ae) {
    ae->cfg = *cfg;
    DDB_TRY(ddb_host::sm100_device(&ae->num_sms));
    const int L = cfg->n_levels;
    if (L < 1 || L > 8) return failf(DDB_ERR_INVALID, "autoencoder: n_levels must be 1..8");
    if (cfg->z_channels < 1 || cfg->z_channels > 8) return failf(DDB_ERR_INVALID, "autoencoder: z_channels must be 1..8");
    if (cfg->out_ch < 1 || cfg->out_ch > 8) return failf(DDB_ERR_INVALID, "autoencoder: out_ch must be 1..8");
    if (cfg->embed_dim != cfg->z_channels) return failf(DDB_ERR_INVALID, "autoencoder: embed_dim != z_channels unsupported");
    if (cfg->max_batch < 1) return failf(DDB_ERR_INVALID, "autoencoder: max_batch must be >= 1");
    if (cfg->resolution % (1 << (L - 1))) return failf(DDB_ERR_INVALID, "autoencoder: resolution not divisible by 2^(levels-1)");
    const int B = ae->maxB = cfg->max_batch;
    const int zres = ae->zres = cfg->resolution >> (L - 1);
    TensorMap tm;
    for (int i = 0; i < n_tensors; ++i) tm[tensors[i].name] = &tensors[i];

    // buffer sizes: walk the resolutions once
    size_t max_elems = 0;
    int cmax = 64;
    {
        int res = zres, c = cfg->ch * cfg->ch_mult[L - 1];
        for (int lvl = L - 1; lvl >= 0; --lvl) {
            const int co = cfg->ch * cfg->ch_mult[lvl];
            const int cm = c > co ? c : co;
            if ((size_t)res * res * cm > max_elems) max_elems = (size_t)res * res * cm;
            if (cm > cmax) cmax = cm;
            c = co;
            if (lvl != 0) {
                res *= 2;
                if ((size_t)res * res * c > max_elems) max_elems = (size_t)res * res * c;
            }
        }
    }
    for (auto& b : ae->act) DDB_TRY(new_buf(b, (size_t)B * max_elems * 2, true));
    const int max_slots = (cfg->resolution * cfg->resolution) >> 7;
    for (auto& p : ae->part) DDB_TRY(new_buf(p, (size_t)B * (max_slots > 1 ? max_slots : 1) * 32 * sizeof(float2), true));
    DDB_TRY(new_buf(ae->affine, (size_t)B * cmax * sizeof(float2), true));
    DDB_TRY(new_buf(ae->zin, (size_t)B * zres * zres * 64 * 2, true));

    // post_quant_conv (1x1, embed_dim -> z_channels), fused with the 1/scale_factor into the prep kernel
    const float *pw, *pb;
    const int Cz = cfg->z_channels;
    DDB_TRY(get_tensor(tm, "post_quant_conv.weight", (int64_t)Cz * Cz, &pw));
    DDB_TRY(get_tensor(tm, "post_quant_conv.bias", Cz, &pb));
    DDB_TRY(new_buf(ae->pq_w, (size_t)Cz * Cz * 4));
    DDB_TRY(new_buf(ae->pq_b, (size_t)Cz * 4));
    CUDA_TRY(cudaMemcpy(ae->pq_w->p, pw, (size_t)Cz * Cz * 4, cudaMemcpyDeviceToDevice));
    CUDA_TRY(cudaMemcpy(ae->pq_b->p, pb, (size_t)Cz * 4, cudaMemcpyDeviceToDevice));

    Builder bld{ae, tm, B, ae->ops};
    void *X = ae->act[0]->p, *Y = ae->act[1]->p, *T1 = ae->act[2]->p, *T2 = ae->act[3]->p;
    {
        Op p;
        p.kind = OP_PREP, p.cat = AC_OTHER, p.name = "post_quant_conv";
        p.out = ae->zin->p, p.out_C = 64, p.out_H = zres, p.out_W = zres;
        ae->ops.push_back(p);
    }
    int res = zres;
    int c = cfg->ch * cfg->ch_mult[L - 1];
    ConvW* cin;
    DDB_TRY(bld.pack("decoder.conv_in", c, Cz, 3, 64, "", 0, false, &cin));
    float2* px = bld.next_part();
    int px_slots = (res * res) >> 7;
    DDB_TRY(bld.add_conv("conv_in", AC_CONV3, cin, ae->zin->p, 64, 64, res, res, 3, false, nullptr, 0, nullptr, X, px));
    ae->ops.back().flops_per_sample = 2.0 * res * res * c * 9.0 * Cz;  // algorithmic (unpadded) work

    float2* py;
    DDB_TRY(bld.add_resblock("mid.block_1", "decoder.mid.block_1", c, c, res, res, X, px, px_slots, T1, T2, Y, &py));
    std::swap(X, Y), px = py;
    DDB_TRY(bld.add_attn("mid.attn_1", "decoder.mid.attn_1", c, res, res, X, px, px_slots, T1, Y, &py));
    std::swap(X, Y), px = py;
    DDB_TRY(bld.add_resblock("mid.block_2", "decoder.mid.block_2", c, c, res, res, X, px, px_slots, T1, T2, Y, &py));
    std::swap(X, Y), px = py;

    for (int lvl = L - 1; lvl >= 0; --lvl) {
        const int co = cfg->ch * cfg->ch_mult[lvl];
        for (int j = 0; j < cfg->num_res_blocks + 1; ++j) {
            char nm[64], key[96];
            snprintf(nm, sizeof(nm), "up.%d.block.%d", lvl, j);
            snprintf(key, sizeof(key), "decoder.up.%d.block.%d", lvl, j);
            DDB_TRY(bld.add_resblock(nm, key, c, co, res, res, X, px, px_slots, T1, T2, Y, &py));
            std::swap(X, Y), px = py;
            c = co;
        }
        if (lvl != 0) {
            char nm[64], key[96];
            snprintf(nm, sizeof(nm), "up.%d.upsample", lvl);
            snprintf(key, sizeof(key), "decoder.up.%d.upsample.conv", lvl);
            ConvW* up;
            DDB_TRY(bld.pack(key, c, c, 3, c, "", 0, true, &up));
            py = bld.next_part();
            DDB_TRY(bld.add_conv(nm, AC_CONV_UP, up, X, c, c, res, res, 3, true, nullptr, 0, nullptr, Y, py));
            std::swap(X, Y), px = py;
            res *= 2;
            px_slots = (res * res) >> 7;
        }
    }
    DDB_TRY(bld.add_gn("norm_out", "decoder.norm_out", px, px_slots, X, T1, c, res, res, true));
    ConvW* cout;
    DDB_TRY(bld.pack("decoder.conv_out", cfg->out_ch, c, 3, c, "", 0, false, &cout));
    DDB_TRY(bld.add_conv("conv_out", AC_CONV3, cout, T1, c, c, res, res, 3, false, nullptr, 0, nullptr, nullptr, nullptr));
    {
        Op& o = ae->ops.back();
        o.epi = CEPI_IMG, o.BN = 64;
        o.conv.img_C = cfg->out_ch;
        o.out = nullptr, o.out_C = cfg->out_ch, o.out_f32 = 1;
    }
    CUDA_TRY(cudaDeviceSynchronize());
    return DDB_OK;
}

// Encoder.forward + quant_conv (FrozenAutoencoderKL.encode_moments): image [B, in_ch, R, R] fp32 -> moments
// [B, 2*embed_dim, R/2^(L-1), R/2^(L-1)] fp32.  Built on a handle whose decoder plan exists; every encoder tensor lives
// in the decoder's activation / GroupNorm / AttnBlock workspace (checked here, true for get_autoencoder's ddconfig).
int encoder_build(ddb_ae* ae, TensorMap& tm) {
    const ddb_ae_config* cfg = &ae->cfg;
    const int L = cfg->n_levels, B = ae->maxB, R = cfg->resolution, ch = cfg->ch;
    auto it = tm.find("encoder.conv_in.weight");
    if (it == tm.end()) return failf(DDB_ERR_MISSING_KEY, "state_dict key 'encoder.conv_in.weight' missing");
    if (ch < 1 || it->second->numel % (9LL * ch))
        return failf(DDB_ERR_SHAPE, "state_dict key 'encoder.conv_in.weight' has %lld elements, not ch * in_channels * 9",
                     (long long)it->second->numel);
    const int Cin = (int)(it->second->numel / (9LL * ch));
    if (Cin < 1 || Cin > 7)
        return failf(DDB_ERR_INVALID, "autoencoder: encoder in_channels %d unsupported (conv_in packs 9 * in_channels <= 64 "
                     "im2col columns, so in_channels <= 7)", Cin);
    if (2 * cfg->embed_dim > 8)  // the CEPI_IMG epilogue writes at most 8 fp32 channel planes
        return failf(DDB_ERR_INVALID, "autoencoder: encoder needs 2 * embed_dim <= 8 (got embed_dim %d)", cfg->embed_dim);
    ae->enc_in_ch = Cin;

    // fit into the decoder's workspace: activations (incl. the 64-column im2col rows), affine, GroupNorm partials
    {
        size_t need = (size_t)R * R * 64;
        int cmax = ch, res = R, c = ch;
        for (int lvl = 0; lvl < L; ++lvl) {
            const int co = ch * cfg->ch_mult[lvl], cm = c > co ? c : co;
            if ((size_t)res * res * cm > need) need = (size_t)res * res * cm;
            if (cm > cmax) cmax = cm;
            c = co;
            if (lvl != L - 1) res /= 2;
        }
        const size_t have = ae->act[0]->bytes / ((size_t)B * 2);
        if (need > have)
            return failf(DDB_ERR_INVALID, "autoencoder: encoder activations (%zu elements per sample) exceed the decoder's "
                         "workspace (%zu)", need, have);
        if ((size_t)B * cmax * sizeof(float2) > ae->affine->bytes)
            return failf(DDB_ERR_INVALID, "autoencoder: encoder width %d exceeds the decoder's GroupNorm workspace", cmax);
        const size_t slots = ((size_t)R * R) >> 7;
        if ((size_t)B * slots * 32 * sizeof(float2) > ae->part[0]->bytes)
            return failf(DDB_ERR_INVALID, "autoencoder: encoder GroupNorm partials exceed the decoder's workspace");
    }

    Builder bld{ae, tm, B, ae->enc_ops};
    void *X = ae->act[0]->p, *Y = ae->act[1]->p, *T1 = ae->act[2]->p, *T2 = ae->act[3]->p;
    {
        Op p;
        p.kind = OP_IM2COL, p.cat = AC_OTHER, p.name = "im2col", p.C = Cin;
        p.out = T1, p.out_C = 64, p.out_H = R, p.out_W = R;
        ae->enc_ops.push_back(p);
    }
    // conv_in as one tap over the 64 im2col columns: weight rows k = (ky*3 + kx)*Cin + c, zero-padded to K = 64
    ConvW* cin;
    {
        const float *w, *b;
        DDB_TRY(get_tensor(tm, "encoder.conv_in.weight", (int64_t)ch * Cin * 9, &w));
        DDB_TRY(get_tensor(tm, "encoder.conv_in.bias", ch, &b));
        std::unique_ptr<ConvW> cw(new ConvW);
        cw->N = ch, cw->N_pad = (ch + 63) / 64 * 64, cw->ktot = 64, cw->nw = 1;
        DDB_TRY(new_buf(cw->w, (size_t)cw->N_pad * 64 * 2, true));
        DDB_TRY(new_buf(cw->bias, (size_t)cw->N_pad * 4, true));
        pack_conv_kernel<<<cw->N_pad, 256>>>(w, ch, Cin, 3, 3, cw->N_pad, Cin, 64, 0, 0,
                                             reinterpret_cast<__nv_bfloat16*>(cw->w->p));
        LAUNCH_CHECK();
        add_bias_kernel<<<(cw->N_pad + 255) / 256, 256>>>(b, nullptr, ch, cw->N_pad, reinterpret_cast<float*>(cw->bias->p));
        LAUNCH_CHECK();
        cin = cw.get();
        ae->convs.push_back(std::move(cw));
    }
    int res = R, c = ch;
    float2* px = bld.next_part();
    int px_slots = (res * res) >> 7;
    DDB_TRY(bld.add_conv("conv_in", AC_CONV3, cin, T1, 64, 64, res, res, 1, false, nullptr, 0, nullptr, X, px));
    ae->enc_ops.back().flops_per_sample = 2.0 * res * res * ch * 9.0 * Cin;  // algorithmic (unpadded) work

    float2* py;
    for (int lvl = 0; lvl < L; ++lvl) {
        const int co = ch * cfg->ch_mult[lvl];
        for (int j = 0; j < cfg->num_res_blocks; ++j) {
            char nm[64], key[96];
            snprintf(nm, sizeof(nm), "down.%d.block.%d", lvl, j);
            snprintf(key, sizeof(key), "encoder.down.%d.block.%d", lvl, j);
            DDB_TRY(bld.add_resblock(nm, key, c, co, res, res, X, px, px_slots, T1, T2, Y, &py));
            std::swap(X, Y), px = py;
            c = co;
        }
        if (lvl != L - 1) {  // Downsample: F.pad(h, (0, 1, 0, 1)), Conv2d(c, c, 3, stride=2, padding=0)
            char nm[64], key[96];
            snprintf(nm, sizeof(nm), "down.%d.downsample", lvl);
            snprintf(key, sizeof(key), "encoder.down.%d.downsample.conv", lvl);
            ConvW* dn;
            DDB_TRY(bld.pack(key, c, c, 3, c, "", 0, false, &dn));
            py = bld.next_part();
            const int ro = res / 2;
            DDB_TRY(bld.add_conv(nm, AC_CONV3, dn, X, c, c, ro, ro, 3, false, nullptr, 0, nullptr, Y, py));
            ConvArgs& a = ae->enc_ops.back().conv;
            a.stride2 = 1, a.dy0 = a.dx0 = 0;
            DDB_TRY(tmap_stride2(&a.tmA0, X, c, ro, ro, B, a.BW, a.BH));
            std::swap(X, Y), px = py;
            res = ro;
            px_slots = (res * res) >> 7;
        }
    }
    DDB_TRY(bld.add_resblock("mid.block_1", "encoder.mid.block_1", c, c, res, res, X, px, px_slots, T1, T2, Y, &py));
    std::swap(X, Y), px = py;
    DDB_TRY(bld.add_attn("mid.attn_1", "encoder.mid.attn_1", c, res, res, X, px, px_slots, T1, Y, &py));
    std::swap(X, Y), px = py;
    DDB_TRY(bld.add_resblock("mid.block_2", "encoder.mid.block_2", c, c, res, res, X, px, px_slots, T1, T2, Y, &py));
    std::swap(X, Y), px = py;
    DDB_TRY(bld.add_gn("norm_out", "encoder.norm_out", px, px_slots, X, T1, c, res, res, true));

    // conv_out (c -> 2*z_channels) with quant_conv (1x1, 2*z_channels -> 2*embed_dim) folded into its weights and bias
    // in fp32, before the bf16 rounding; the CEPI_IMG epilogue writes the moments straight into the caller's NCHW buffer
    const int Nz = 2 * cfg->z_channels, Nm = 2 * cfg->embed_dim, K = c * 9;
    const float *ow, *ob, *qw, *qb;
    DDB_TRY(get_tensor(tm, "encoder.conv_out.weight", (int64_t)Nz * K, &ow));
    DDB_TRY(get_tensor(tm, "encoder.conv_out.bias", Nz, &ob));
    DDB_TRY(get_tensor(tm, "quant_conv.weight", (int64_t)Nm * Nz, &qw));
    DDB_TRY(get_tensor(tm, "quant_conv.bias", Nm, &qb));
    Buf fw, fb;
    DDB_TRY(new_buf(fw, (size_t)Nm * K * 4));
    DDB_TRY(new_buf(fb, (size_t)Nm * 4));
    fold_1x1_kernel<<<Nm, 256>>>(qw, qb, ow, ob, Nm, Nz, K, reinterpret_cast<float*>(fw->p),
                                 reinterpret_cast<float*>(fb->p));
    LAUNCH_CHECK();
    const ddb_tensor folded[2] = {{"moments.weight", reinterpret_cast<const float*>(fw->p), (int64_t)Nm * K},
                                  {"moments.bias", reinterpret_cast<const float*>(fb->p), Nm}};
    tm["moments.weight"] = &folded[0], tm["moments.bias"] = &folded[1];
    ConvW* mo;
    DDB_TRY(bld.pack("moments", Nm, c, 3, c, "", 0, false, &mo));
    DDB_TRY(bld.add_conv("moments", AC_CONV3, mo, T1, c, c, res, res, 3, false, nullptr, 0, nullptr, nullptr, nullptr));
    {
        Op& o = ae->enc_ops.back();
        o.epi = CEPI_IMG, o.BN = 64;
        o.conv.img_C = Nm;
        o.out = nullptr, o.out_C = Nm, o.out_f32 = 1;
    }
    CUDA_TRY(cudaDeviceSynchronize());  // the folded fp32 weights are freed on return
    return DDB_OK;
}

// in: the plan's fp32 input (latents / image) of this chunk; out: its fp32 output (image / moments)
int run_op(const ddb_ae* ae, const Op& op, int B, const float* in, float* out, cudaStream_t st) {
    switch (op.kind) {
        case OP_PREP: {
            const int HW = ae->zres * ae->zres, n = B * HW;
            CUDA_TRY(ddb_host::launch_pdl(ae_prep_kernel, dim3((n + 127) / 128), dim3(128), 0, st, in,
                                          reinterpret_cast<const float*>(ae->pq_w->p),
                                          reinterpret_cast<const float*>(ae->pq_b->p), 1.0f / ae->cfg.scale_factor, B,
                                          ae->cfg.z_channels, HW, reinterpret_cast<__nv_bfloat16*>(ae->zin->p)));
            LAUNCH_CHECK();
            return DDB_OK;
        }
        case OP_CONV: {
            ConvArgs a = op.conv;
            a.B = B;
            if (op.epi == CEPI_IMG) a.img = out;
            return launch_conv(a, op.BN, op.epi, ae->num_sms, st);
        }
        case OP_GN_FINALIZE:
            CUDA_TRY(ddb_host::launch_pdl(gn_finalize_kernel, dim3(B), dim3(256), 0, st, op.part, op.slots, op.C, op.cpg,
                                          op.count, 1e-6f, op.gamma, op.beta, ae->affine_p()));
            LAUNCH_CHECK();
            return DDB_OK;
        case OP_GN_APPLY: {
            const int units = op.C >> 3;
            int rows = 4096 / units;  // ~4096 16-byte units (64 KB) per CTA
            if (rows < 1) rows = 1;
            if (rows > op.HW) rows = op.HW;
            const dim3 grid((op.HW + rows - 1) / rows, B);
            if (256 % units == 0)
                CUDA_TRY(ddb_host::launch_pdl(gn_apply_kernel<true>, grid, dim3(256), 0, st, op.x,
                                              (const float2*)ae->affine_p(), op.HW, op.C, rows, op.swish, op.y));
            else
                CUDA_TRY(ddb_host::launch_pdl(gn_apply_kernel<false>, grid, dim3(256), (size_t)op.C * sizeof(float2),
                                              st, op.x, (const float2*)ae->affine_p(), op.HW, op.C, rows, op.swish,
                                              op.y));
            LAUNCH_CHECK();
            return DDB_OK;
        }
        case OP_TRANSPOSE_V:
            CUDA_TRY(ddb_host::launch_pdl(transpose_v_kernel, dim3(op.T / 32, op.C / 32, B), dim3(32, 8), 0, st,
                                          reinterpret_cast<const __nv_bfloat16*>(ae->qkv->p), op.T, op.C, op.pitch,
                                          op.v_off, reinterpret_cast<__nv_bfloat16*>(ae->vT->p)));
            LAUNCH_CHECK();
            return DDB_OK;
        case OP_SOFTMAX: {
            const int rows = B * op.T;
            CUDA_TRY(ddb_host::launch_pdl(softmax_rows_kernel, dim3((rows + 7) / 8), dim3(256), 0, st, op.S, rows, op.T,
                                          reinterpret_cast<__nv_bfloat16*>(ae->P->p)));
            LAUNCH_CHECK();
            return DDB_OK;
        }
        case OP_IM2COL: {
            const int R = ae->cfg.resolution, n = B * R * R;
            CUDA_TRY(ddb_host::launch_pdl(ae_im2col_kernel, dim3((n + 127) / 128), dim3(128), 0, st, in, B, op.C, R, R,
                                          reinterpret_cast<__nv_bfloat16*>(const_cast<void*>(op.out))));
            LAUNCH_CHECK();
            return DDB_OK;
        }
    }
    return failf(DDB_ERR_INVALID, "bad op");
}

// replay one plan per chunk of max_batch samples; in_s / out_s: fp32 elements per sample of its input / output
int run_plan(const ddb_ae* ae, const std::vector<Op>& ops, const float* in, size_t in_s, int B, float* out,
             size_t out_s, cudaStream_t st, int dump_op, void* dump_dev, float* ms_host, double* flops_host) {
    std::vector<cudaEvent_t> ev;
    if (ms_host) {
        ev.resize(ops.size() + 1);
        for (auto& e : ev) CUDA_TRY(cudaEventCreate(&e));
        for (int i = 0; i < AC_COUNT; ++i) ms_host[i] = 0.f;
        if (flops_host) for (int i = 0; i < AC_COUNT; ++i) flops_host[i] = 0.0;
    }
    for (int b0 = 0; b0 < B; b0 += ae->maxB) {
        const int nb = (B - b0 < ae->maxB) ? B - b0 : ae->maxB;
        if (ms_host) CUDA_TRY(cudaEventRecord(ev[0], st));
        for (size_t i = 0; i < ops.size(); ++i) {
            const Op& op = ops[i];
            DDB_TRY(run_op(ae, op, nb, in + (size_t)b0 * in_s, out + (size_t)b0 * out_s, st));
            if (ms_host) CUDA_TRY(cudaEventRecord(ev[i + 1], st));
            if ((int)i == dump_op && dump_dev && op.out && b0 == 0) {
                const size_t bytes = (size_t)nb * op.out_C * op.out_H * op.out_W * (op.out_f32 ? 4 : 2);
                CUDA_TRY(cudaMemcpyAsync(dump_dev, op.out, bytes, cudaMemcpyDeviceToDevice, st));
            }
        }
        if (ms_host) {
            CUDA_TRY(cudaStreamSynchronize(st));
            for (size_t i = 0; i < ops.size(); ++i) {
                float ms = 0.f;
                CUDA_TRY(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
                ms_host[ops[i].cat] += ms;
                if (flops_host) flops_host[ops[i].cat] += ops[i].flops_per_sample * nb;
            }
        }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    return DDB_OK;
}

int decode_impl(ddb_ae* ae, const float* z, int B, float* img, cudaStream_t st, int dump_op, void* dump_dev,
                float* ms_host, double* flops_host) {
    const size_t zs = (size_t)ae->cfg.z_channels * ae->zres * ae->zres;
    const size_t is = (size_t)ae->cfg.out_ch * ae->cfg.resolution * ae->cfg.resolution;
    return run_plan(ae, ae->ops, z, zs, B, img, is, st, dump_op, dump_dev, ms_host, flops_host);
}

int encode_impl(ddb_ae* ae, const float* img, int B, float* moments, cudaStream_t st, int dump_op, void* dump_dev,
                float* ms_host, double* flops_host) {
    if (ae->enc_ops.empty())
        return failf(DDB_ERR_INVALID, "autoencoder: no encoder on this handle (ddb_ae_create_encoder)");
    const size_t is = (size_t)ae->enc_in_ch * ae->cfg.resolution * ae->cfg.resolution;
    const size_t ms = (size_t)2 * ae->cfg.embed_dim * ae->zres * ae->zres;
    return run_plan(ae, ae->enc_ops, img, is, B, moments, ms, st, dump_op, dump_dev, ms_host, flops_host);
}

}  // namespace

namespace ddb_host {
bool ae_set_option(const char* name, int value) {
    if (!strcmp(name, "conv_mt2")) {
        g_conv_mt2 = value != 0;
        return true;
    }
    return false;
}
}  // namespace ddb_host

namespace {
int op_info(const Op& op, char* name_out, int32_t name_cap, int32_t* chw_f32_out) {
    snprintf(name_out, name_cap, "%s", op.name.c_str());
    chw_f32_out[0] = op.out ? op.out_C : 0, chw_f32_out[1] = op.out_H, chw_f32_out[2] = op.out_W,
    chw_f32_out[3] = op.out_f32;
    return DDB_OK;
}
}  // namespace

extern "C" {

int ddb_ae_create(const ddb_ae_config* cfg, const ddb_tensor* tensors, int32_t n_tensors, ddb_ae** out) {
    if (!cfg || !tensors || !out) return failf(DDB_ERR_INVALID, "null argument");
    std::unique_ptr<ddb_ae> ae(new ddb_ae);
    DDB_TRY(ae_create_impl(cfg, tensors, n_tensors, ae.get()));
    *out = ae.release();
    return DDB_OK;
}

void ddb_ae_destroy(ddb_ae* ae) {
    if (!ae) return;
    cudaDeviceSynchronize();
    delete ae;
}

int ddb_ae_decode(ddb_ae* ae, const float* z_dev, int32_t B, float* img_dev, void* stream) {
    if (!ae || !z_dev || !img_dev || B < 0) return failf(DDB_ERR_INVALID, "ddb_ae_decode: bad argument");
    return decode_impl(ae, z_dev, B, img_dev, reinterpret_cast<cudaStream_t>(stream), -1, nullptr, nullptr, nullptr);
}

int ddb_ae_profile_decode(ddb_ae* ae, const float* z_dev, int32_t B, float* img_dev, float* ms_host,
                          double* flops_host, void* stream) {
    if (!ae || !z_dev || !img_dev || !ms_host || B < 0) return failf(DDB_ERR_INVALID, "ddb_ae_profile_decode: bad argument");
    return decode_impl(ae, z_dev, B, img_dev, reinterpret_cast<cudaStream_t>(stream), -1, nullptr, ms_host, flops_host);
}

int32_t ddb_ae_num_ops(const ddb_ae* ae) { return ae ? (int32_t)ae->ops.size() : 0; }

int ddb_ae_op_info(const ddb_ae* ae, int32_t i, char* name_out, int32_t name_cap, int32_t* chw_f32_out) {
    if (!ae || i < 0 || i >= (int32_t)ae->ops.size() || !name_out || !chw_f32_out)
        return failf(DDB_ERR_INVALID, "ddb_ae_op_info: bad argument");
    return op_info(ae->ops[i], name_out, name_cap, chw_f32_out);
}

int ddb_ae_decode_debug(ddb_ae* ae, const float* z_dev, int32_t B, float* img_dev, int32_t op_index, void* dump_dev,
                        void* stream) {
    if (!ae || !z_dev || !img_dev || B < 0 || B > ae->maxB)
        return failf(DDB_ERR_INVALID, "ddb_ae_decode_debug: bad argument (B must be <= max_batch)");
    return decode_impl(ae, z_dev, B, img_dev, reinterpret_cast<cudaStream_t>(stream), op_index, dump_dev, nullptr,
                       nullptr);
}

int ddb_ae_create_encoder(ddb_ae* ae, const ddb_tensor* tensors, int32_t n_tensors) {
    if (!ae || n_tensors < 0 || (n_tensors > 0 && !tensors)) return failf(DDB_ERR_INVALID, "ddb_ae_create_encoder: bad argument");
    if (!ae->enc_ops.empty()) return failf(DDB_ERR_INVALID, "ddb_ae_create_encoder: the handle already has an encoder");
    TensorMap tm;
    for (int i = 0; i < n_tensors; ++i) tm[tensors[i].name] = &tensors[i];
    const int r = encoder_build(ae, tm);
    if (r != DDB_OK) ae->enc_ops.clear();  // no half-built plan: encode keeps failing with "no encoder"
    return r;
}

int ddb_ae_encode_moments(ddb_ae* ae, const float* img_dev, int32_t B, float* moments_dev, void* stream) {
    if (!ae || !img_dev || !moments_dev || B < 0) return failf(DDB_ERR_INVALID, "ddb_ae_encode_moments: bad argument");
    return encode_impl(ae, img_dev, B, moments_dev, reinterpret_cast<cudaStream_t>(stream), -1, nullptr, nullptr,
                       nullptr);
}

int ddb_ae_sample(ddb_ae* ae, const float* moments_dev, const float* noise_dev, int32_t B, float* z_dev, void* stream) {
    if (!ae || !moments_dev || !noise_dev || !z_dev || B < 0) return failf(DDB_ERR_INVALID, "ddb_ae_sample: bad argument");
    const int E = ae->cfg.embed_dim, HW = ae->zres * ae->zres;
    const size_t n = (size_t)B * E * HW;
    if (n == 0) return DDB_OK;
    ae_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
        moments_dev, noise_dev, B, E, HW, ae->cfg.scale_factor, z_dev);
    LAUNCH_CHECK();
    return DDB_OK;
}

int ddb_ae_profile_encode(ddb_ae* ae, const float* img_dev, int32_t B, float* moments_dev, float* ms_host,
                          double* flops_host, void* stream) {
    if (!ae || !img_dev || !moments_dev || !ms_host || B < 0)
        return failf(DDB_ERR_INVALID, "ddb_ae_profile_encode: bad argument");
    return encode_impl(ae, img_dev, B, moments_dev, reinterpret_cast<cudaStream_t>(stream), -1, nullptr, ms_host,
                       flops_host);
}

int32_t ddb_ae_encoder_num_ops(const ddb_ae* ae) { return ae ? (int32_t)ae->enc_ops.size() : 0; }

int ddb_ae_encoder_op_info(const ddb_ae* ae, int32_t i, char* name_out, int32_t name_cap, int32_t* chw_f32_out) {
    if (!ae || i < 0 || i >= (int32_t)ae->enc_ops.size() || !name_out || !chw_f32_out)
        return failf(DDB_ERR_INVALID, "ddb_ae_encoder_op_info: bad argument");
    return op_info(ae->enc_ops[i], name_out, name_cap, chw_f32_out);
}

int ddb_ae_encode_debug(ddb_ae* ae, const float* img_dev, int32_t B, float* moments_dev, int32_t op_index,
                        void* dump_dev, void* stream) {
    if (!ae || !img_dev || !moments_dev || B < 0 || B > ae->maxB)
        return failf(DDB_ERR_INVALID, "ddb_ae_encode_debug: bad argument (B must be <= max_batch)");
    return encode_impl(ae, img_dev, B, moments_dev, reinterpret_cast<cudaStream_t>(stream), op_index, dump_dev,
                       nullptr, nullptr);
}

}  // extern "C"
