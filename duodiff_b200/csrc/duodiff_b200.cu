// Host side of libduodiff_b200.so: weight re-packing, workspace, TMA descriptors, the U-ViT launch sequence,
// the DDPM sampler loop with CUDA-graph replay, and the extern "C" boundary declared in include/duodiff_b200.h.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <utility>
#include <vector>

#include "../../include/duodiff_b200.h"
#include "attention.cuh"
#include "elementwise.cuh"
#include "gemm.cuh"
#include "gemm2.cuh"
#include "host_common.h"
// Measured-and-rejected kernel variants (A-in-TMEM GEMM, two-threads-per-row attention, generic mma.sync attention,
// fp32-FMA token assembly, single-CTA GEMM for the block linears) are only part of -DDDB_EXPERIMENTAL builds; the
// product library contains the path that runs.
#ifdef DDB_EXPERIMENTAL
#include "experimental/attention2.cuh"
#include "experimental/attention_mma.cuh"
#include "experimental/embed_tokens.cuh"
#include "experimental/gemm3.cuh"
#define DDB_NEEDS_EXPERIMENTAL(what) ((void)0)
#else
#define DDB_NEEDS_EXPERIMENTAL(what) \
    return fail(DDB_ERR_INVALID, "%s is an experimental variant: rebuild with DDB_EXPERIMENTAL=1", what)
#endif

using namespace ddb;

// ------------------------------------------------------------------------------------------------ errors
static thread_local char g_err[1024] = "";
static std::atomic<long long> g_launches{0};

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_TRY(expr)                                                                                  \
    do {                                                                                                \
        cudaError_t _e = (expr);                                                                        \
        if (_e != cudaSuccess)                                                                          \
            return fail(DDB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                        __LINE__);                                                                      \
    } while (0)
#define DDB_TRY(expr)            \
    do {                         \
        int _r = (expr);         \
        if (_r != DDB_OK) return _r; \
    } while (0)
#define LAUNCH_CHECK()                                                                                      \
    do {                                                                                                    \
        g_launches.fetch_add(1, std::memory_order_relaxed);                                                 \
        cudaError_t _e = cudaGetLastError();                                                                \
        if (_e != cudaSuccess)                                                                              \
            return fail(DDB_ERR_CUDA, "kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, \
                        __LINE__);                                                                          \
    } while (0)

// ------------------------------------------------------------------------------------------------ profiling
// Optional per-launch CUDA-event timing of one forward (ddb_profile_forward): events are recorded on the launching
// stream around every kernel and accumulated per category.
enum ProfCat : int {
    PC_EMBED = 0, PC_LN_STATS, PC_GEMM_QKV, PC_ATTENTION, PC_GEMM_PROJ, PC_GEMM_FC1, PC_GEMM_FC2, PC_GEMM_SKIP,
    PC_GEMM_DECODE, PC_CONV, PC_EE_OTHER, PC_DDPM, PC_TAIL, PC_COUNT
};
static_assert(PC_COUNT == DDB_PROF_CATEGORIES, "include/duodiff_b200.h lists the categories");
struct Profiler {
    bool active = false;
    cudaStream_t st = nullptr;
    std::vector<cudaEvent_t> pool;
    std::vector<int> cats;
    size_t used = 0;
    cudaEvent_t next() {
        if (used == pool.size()) {
            cudaEvent_t e;
            cudaEventCreate(&e);
            pool.push_back(e);
        }
        return pool[used++];
    }
    void begin(int cat) {
        if (!active) return;
        cats.push_back(cat);
        cudaEventRecord(next(), st);
    }
    void end() {
        if (active) cudaEventRecord(next(), st);
    }
};
static thread_local Profiler g_prof;  // per calling thread: ddb_profile_forward() of distinct handles may run concurrently
struct ProfScope {
    explicit ProfScope(int cat) { g_prof.begin(cat); }
    ~ProfScope() { g_prof.end(); }
};

// ------------------------------------------------------------------------------------------------ device info
struct DeviceInfo {
    int num_sms = 0;
    int cc_major = 0;
    bool ok = false;
};
static int device_info(DeviceInfo& d) {
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&d.num_sms, cudaDevAttrMultiProcessorCount, dev));
    CUDA_TRY(cudaDeviceGetAttribute(&d.cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    if (d.cc_major != 10)
        return fail(DDB_ERR_CUDA, "duodiff_b200 needs an sm_100 (B200) device; found compute capability %d.x",
                    d.cc_major);
    d.ok = true;
    return DDB_OK;
}

// ------------------------------------------------------------------------------------------------ TMA descriptors
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static int load_encode() {
    if (g_encode) return DDB_OK;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (!fn || qres != cudaDriverEntryPointSuccess)
        return fail(DDB_ERR_CUDA, "cuTensorMapEncodeTiled not available from the driver");
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    return DDB_OK;
}
// bf16 row-major [rows, cols] with row pitch `pitch_elems`; box = 64 columns (128 B, SWIZZLE_128B) x box_rows
static int make_tmap_bf16(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                          uint32_t box_rows) {
    DDB_TRY(load_encode());
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {pitch_elems * 2};
    cuuint32_t box[2] = {64, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS)
        return fail(DDB_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu pitch=%llu box_rows=%u",
                    (int)r, (unsigned long long)rows, (unsigned long long)cols, (unsigned long long)pitch_elems,
                    box_rows);
    return DDB_OK;
}

// bf16 row-major [rows, cols]; box = 32 columns (64 B, SWIZZLE_64B) x box_rows: the CTA-pair GEMM's output sub-chunks
static int make_tmap_bf16_sw64(CUtensorMap* tm, const void* base, uint64_t rows, uint64_t cols, uint64_t pitch_elems,
                               uint32_t box_rows) {
    DDB_TRY(load_encode());
    cuuint64_t gdim[2] = {cols, rows};
    cuuint64_t gstr[1] = {pitch_elems * 2};
    cuuint32_t box[2] = {32, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(DDB_ERR_CUDA, "cuTensorMapEncodeTiled(sw64) failed (%d)", (int)r);
    return DDB_OK;
}

// bf16 [d2, d1, d0] (d0 contiguous) with byte strides; box {64, box1, 1}, SWIZZLE_128B
static int make_tmap_bf16_3d(CUtensorMap* tm, const void* base, uint64_t d0, uint64_t d1, uint64_t d2,
                             uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t box1) {
    DDB_TRY(load_encode());
    cuuint64_t gdim[3] = {d0, d1, d2};
    cuuint64_t gstr[2] = {stride1_bytes, stride2_bytes};
    cuuint32_t box[3] = {64, box1, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return fail(DDB_ERR_CUDA, "cuTensorMapEncodeTiled(3d) failed (%d)", (int)r);
    return DDB_OK;
}

// helpers shared with the other translation units (csrc/host_common.h)
namespace ddb_host {
int fail_msg(int code, const char* msg) { return fail(code, "%s", msg); }
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
int sm100_device(int* num_sms) {
    DeviceInfo d;
    DDB_TRY(device_info(d));
    *num_sms = d.num_sms;
    return DDB_OK;
}
int encode_bf16_sw128(CUtensorMap* tm, const void* base, int rank, const unsigned long long* dims,
                      const unsigned long long* strides, const unsigned* box) {
    DDB_TRY(load_encode());
    cuuint64_t gdim[5], gstr[4];
    cuuint32_t bx[5], estr[5];
    for (int i = 0; i < rank; ++i) gdim[i] = dims[i], bx[i] = box[i], estr[i] = 1;
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides[i];
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(base), gdim, gstr, bx, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        char msg[256];
        snprintf(msg, sizeof(msg), "cuTensorMapEncodeTiled(rank %d) failed (%d): dims %llu %llu %llu box %u %u %u", rank,
                 (int)r, dims[0], dims[1], rank > 2 ? dims[2] : 0ull, box[0], box[1], rank > 2 ? box[2] : 0u);
        return fail(DDB_ERR_CUDA, "%s", msg);
    }
    return DDB_OK;
}
}  // namespace ddb_host

// ------------------------------------------------------------------------------------------------ launches
// ---- process-wide runtime options (ddb_set_option).  They are A/B switches for measurements, read when a kernel is
// launched or a step graph is captured; g_option_epoch invalidates captured graphs when one of them changes.
static std::atomic<int> g_option_epoch{0};
static std::atomic<int> g_use_pdl{1};
namespace ddb_host {
int use_pdl() { return g_use_pdl; }
}  // ddb_set_option "pdl": programmatic dependent launch between the kernels of a step
// Launch with programmaticStreamSerialization: the kernel may become resident while its predecessor drains; every
// kernel launched this way calls pdl_wait() before it touches global memory (csrc/ptx.cuh).
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kfn)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
    if (!g_use_pdl) {
        kfn<<<grid, block, smem, st>>>(std::forward<Args>(args)...);
        return cudaGetLastError();
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at, cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kfn, std::forward<Args>(args)...);
}

// ------------------------------------------------------------------------------------------------ GEMM launch
template <int BN, int EPI>
static int launch_gemm_t(const GemmArgs& a, int num_sms, cudaStream_t st) {
    static ddb_host::DeviceOnce configured;
    auto kfn = gemm_tcgen05_kernel<BN, EPI>;
    if (!configured.done()) {
        CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<BN>::SMEM_BYTES));
        configured.mark();
    }
    const int tiles = a.grp_layer ? a.grp_B * ((a.L + 127) / 128) : ((a.M + 127) / 128) * (a.N / BN);
    const int grid = tiles < num_sms ? tiles : num_sms;
    if (grid <= 0) return DDB_OK;
    CUDA_TRY(launch_pdl(kfn, dim3(grid), dim3(384), GemmCfg<BN>::SMEM_BYTES, st, a));
    LAUNCH_CHECK();
    return DDB_OK;
}
// runtime options (ddb_set_option): gemm_variant 2 = CTA-pair kernel (default), 1 = single-CTA kernel
static std::atomic<int> g_gemm_variant{2};
static std::atomic<int> g_gemm_debug{0};
// bench-only (tools/ee_overhead.py): price the early-exit bookkeeping of a NEVER-EXIT step by leaving parts of it out --
// 1 no row move, 2 no decision, 4 no probe partials in the fc2 epilogue, 8 no probe pass over the first block input
static std::atomic<int> g_ee_debug{0};
// ddb_set_option "ee_fuse": the early-exit step in compaction mode ends in the fused step tail (per-sample conv weights)
static std::atomic<int> g_ee_fuse{1};
static std::atomic<long long*> g_gemm_trace{nullptr};  // bench-only (ddb_debug_set_ptr "gemm_trace")

static std::atomic<int> g_attn_discard{1};  // ddb_set_option "attn_discard": discard consumed q|k|v lines from L2 (attention.cuh)
static std::atomic<int> g_mlp_split{0};  // ddb_set_option "mlp_split": fc1 -> fc2 in two half batches (hidden stays in L2).  Parity-green but
                             // measured SLOWER at CelebA B = 128 (42.8 -> 41.7 images/s): two partial GEMM rounds and two more
                             // kernel boundaries per block cost more than the ~3 GB of HBM traffic per step it removes.
static std::atomic<int> g_l2_hints{0};  // ddb_set_option "l2_hints": bit 0 fc2 A evict_first, bit 1 fc1 out evict_last, bit 2 qkv out evict_last
static std::atomic<int> g_gemm_ln_cfg{0};  // ddb_set_option "gemm_ln_cfg": 1 = 5 operand stages + 1 staging buffer per warpgroup for qkv / fc1
static std::atomic<int> g_alt_dir{1};  // ddb_set_option "alt_dir": alternate the row direction of consecutive kernels (L2 reuse)
static std::atomic<int> g_gemm_bn128{0};  // ddb_set_option "gemm_bn128": 256x128 tiles for the N = 512 GEMMs. Measured SLOWER (fc2 63 -> 81 us):
                              // a 256x128x16 MMA takes ~0.75x the time of a 256x256x16 one, not 0.5x (shared-memory operand reads)
template <int EPI, bool STATS, int STAGES, int NBUF, int BN = 256, bool PROBE = false>
static int launch_gemm2_t(const GemmArgs& a, int num_sms, cudaStream_t st) {
    static ddb_host::DeviceOnce configured;
    constexpr bool kLN = (EPI == EPI_LN || EPI == EPI_LN_GELU);
    constexpr int kSmem = Gemm2Cfg<STAGES, NBUF, kLN, BN, PROBE>::SMEM_BYTES;
    auto kfn = gemm2_tcgen05_kernel<EPI, STATS, STAGES, NBUF, BN, PROBE>;
    if (!configured.done()) {
        CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
        configured.mark();
    }
    const int tiles = ((a.M + 255) / 256) * (a.N / BN);
    if (g_gemm_debug) const_cast<GemmArgs&>(a).debug = g_gemm_debug;
    const_cast<GemmArgs&>(a).trace = g_gemm_trace;
    int clusters = num_sms / 2;
    if (tiles < clusters) clusters = tiles;
    if (clusters <= 0) return DDB_OK;
    CUDA_TRY(launch_pdl(kfn, dim3(2 * clusters), dim3(384), kSmem, st, a));
    LAUNCH_CHECK();
    return DDB_OK;
}
// CTA-pair GEMM with the A panel resident in TMEM (experimental/gemm3.cuh): K <= 512, one K source, 32-column SWIZZLE_64B output maps
static std::atomic<int> g_gemm_ts{0};
#ifdef DDB_EXPERIMENTAL  // ddb_set_option "gemm_ts": measured no faster than gemm2 (the MMA takes ~165 clk in SS and TS form alike)
template <int EPI, bool STATS>
static int launch_gemm3_t(const GemmArgs& a, int num_sms, cudaStream_t st) {
    static ddb_host::DeviceOnce configured;
    constexpr bool kLN = (EPI == EPI_LN || EPI == EPI_LN_GELU);
    constexpr int kSmem = Gemm3Cfg<8, kLN>::SMEM_BYTES;
    auto kfn = gemm3_tcgen05_kernel<EPI, STATS, 8>;
    if (!configured.done()) {
        CUDA_TRY(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem));
        configured.mark();
    }
    const int tiles = ((a.M + 255) / 256) * (a.N / 256);
    if (g_gemm_debug) const_cast<GemmArgs&>(a).debug = g_gemm_debug;
    const_cast<GemmArgs&>(a).trace = g_gemm_trace;
    int clusters = num_sms / 2;
    if (tiles < clusters) clusters = tiles;
    if (clusters <= 0) return DDB_OK;
    CUDA_TRY(launch_pdl(kfn, dim3(2 * clusters), dim3(G3_THREADS), kSmem, st, a));
    LAUNCH_CHECK();
    return DDB_OK;
}
#endif

// CTA-pair GEMM: a.tmB2 must have been encoded with a 128-row box.  Pipeline shape per epilogue:
//   LN / LN+GELU (K = embed_dim, epilogue-heavy): 4 operand stages, aux-staged row statistics + bias + colsum
//   residual, K <= 512 (proj: epilogue-latency-bound): 4 stages, 3 staging buffers (residual prefetched 2 chunks ahead)
//   residual / bias, K > 512 (fc2, skip: mainloop-bound): 5 stages, 2 staging buffers
static int launch_gemm2(const GemmArgs& a, int epi, int num_sms, cudaStream_t st) {
    const bool stats = a.stats_out != nullptr;
    const bool short_k = (a.K0 + a.K1) <= 512;
#ifdef DDB_EXPERIMENTAL
    if (g_gemm_ts && short_k && a.K1 == 0 && !a.embed_mode) {
        switch (epi) {
            case EPI_LN: return launch_gemm3_t<EPI_LN, false>(a, num_sms, st);
            case EPI_LN_GELU: return launch_gemm3_t<EPI_LN_GELU, false>(a, num_sms, st);
            case EPI_RES:
                return stats ? launch_gemm3_t<EPI_RES, true>(a, num_sms, st)
                             : launch_gemm3_t<EPI_RES, false>(a, num_sms, st);
            default: break;
        }
    }
#endif
    // Wave quantisation: with 256x256 tiles an N = 512 GEMM at M = 32 896 has 258 tiles for 74 CTA pairs (3.49 -> 4
    // rounds); 256x128 tiles give 516 (6.97 -> 7 half-size rounds).  Used whenever it removes at least 5 % of the
    // rounds' work.
    {
        const int clusters = num_sms / 2, mb = (a.M + 255) / 256;
        const int t256 = mb * (a.N / 256), t128 = mb * (a.N / 128);
        const double r256 = (double)((t256 + clusters - 1) / clusters), r128 = 0.5 * ((t128 + clusters - 1) / clusters);
#ifdef DDB_EXPERIMENTAL
        if (g_gemm_bn128 && a.N % 128 == 0 && r128 < 0.95 * r256 && (epi == EPI_BIAS || epi == EPI_RES)) {
            if (epi == EPI_BIAS)
                return stats ? launch_gemm2_t<EPI_BIAS, true, 6, 2, 128>(a, num_sms, st)
                             : launch_gemm2_t<EPI_BIAS, false, 6, 2, 128>(a, num_sms, st);
            return stats ? launch_gemm2_t<EPI_RES, true, 6, 2, 128>(a, num_sms, st)
                         : launch_gemm2_t<EPI_RES, false, 6, 2, 128>(a, num_sms, st);
        }
#else
        (void)r256, (void)r128;
#endif
    }
    switch (epi) {
        case EPI_BIAS:
            return stats ? launch_gemm2_t<EPI_BIAS, true, 5, 2>(a, num_sms, st)
                         : launch_gemm2_t<EPI_BIAS, false, 5, 2>(a, num_sms, st);
        case EPI_LN:
#ifdef DDB_EXPERIMENTAL
            if (g_gemm_ln_cfg == 1) return launch_gemm2_t<EPI_LN, false, 5, 1>(a, num_sms, st);
#endif
            return launch_gemm2_t<EPI_LN, false, 4, 2>(a, num_sms, st);
        case EPI_LN_GELU:
#ifdef DDB_EXPERIMENTAL
            if (g_gemm_ln_cfg == 1) return launch_gemm2_t<EPI_LN_GELU, false, 5, 1>(a, num_sms, st);
#endif
            return launch_gemm2_t<EPI_LN_GELU, false, 4, 2>(a, num_sms, st);
        case EPI_RES:
            if (short_k)
                return stats ? launch_gemm2_t<EPI_RES, true, 4, 3>(a, num_sms, st)
                             : launch_gemm2_t<EPI_RES, false, 4, 3>(a, num_sms, st);
            if (a.probe_w) {  // fc2 of an early-exit model: + the next layer's probe partial dot products
                if (!stats || !a.probe_out) return fail(DDB_ERR_INVALID, "the probe epilogue needs stats_out and probe_out");
                return launch_gemm2_t<EPI_RES, true, 5, 2, 256, true>(a, num_sms, st);
            }
            return stats ? launch_gemm2_t<EPI_RES, true, 5, 2>(a, num_sms, st)
                         : launch_gemm2_t<EPI_RES, false, 5, 2>(a, num_sms, st);
    }
    return fail(DDB_ERR_INVALID, "unknown CTA-pair GEMM epilogue %d", epi);
}

// single-CTA kernel (gemm.cuh): the narrow-N decode head of the model path; the 128x256 variants for the block linears
// (gemm_variant = 1) only exist in experimental builds
static int launch_gemm(const GemmArgs& a, int epi, int num_sms, cudaStream_t st) {
    switch (epi) {
#ifdef DDB_EXPERIMENTAL
        case EPI_BIAS: return launch_gemm_t<256, EPI_BIAS>(a, num_sms, st);
        case EPI_LN: return launch_gemm_t<256, EPI_LN>(a, num_sms, st);
        case EPI_LN_GELU: return launch_gemm_t<256, EPI_LN_GELU>(a, num_sms, st);
        case EPI_RES: return launch_gemm_t<256, EPI_RES>(a, num_sms, st);
#endif
        case EPI_DECODE: return launch_gemm_t<64, EPI_DECODE>(a, num_sms, st);
    }
    return fail(DDB_ERR_INVALID, "single-CTA GEMM epilogue %d is not part of this build", epi);
}

static int launch_ln_stats(const __nv_bfloat16* x, int M, int D, const int* m_dev, float2* stats, const float* pw,
                           float* pp, cudaStream_t st) {
    const int grid = (M + 7) / 8;
    if (grid <= 0) return DDB_OK;
    ProfScope ps(PC_LN_STATS);
    switch (D) {
        case 256: CUDA_TRY(launch_pdl(ln_stats_kernel<256>, dim3(grid), dim3(256), 0, st, x, M, m_dev, stats, pw, pp)); break;
        case 512: CUDA_TRY(launch_pdl(ln_stats_kernel<512>, dim3(grid), dim3(256), 0, st, x, M, m_dev, stats, pw, pp)); break;
        case 768: CUDA_TRY(launch_pdl(ln_stats_kernel<768>, dim3(grid), dim3(256), 0, st, x, M, m_dev, stats, pw, pp)); break;
        case 1024: CUDA_TRY(launch_pdl(ln_stats_kernel<1024>, dim3(grid), dim3(256), 0, st, x, M, m_dev, stats, pw, pp)); break;
        case 2048: CUDA_TRY(launch_pdl(ln_stats_kernel<2048>, dim3(grid), dim3(256), 0, st, x, M, m_dev, stats, pw, pp)); break;
        default: return fail(DDB_ERR_INVALID, "embed_dim %d unsupported (need 256/512/768/1024/2048)", D);
    }
    LAUNCH_CHECK();
    return DDB_OK;
}

// tcgen05 attention: needs exactly 256 patch tokens (L = 256 + extras)
static int plan_attention(AttnArgs& a, const __nv_bfloat16* qkv, __nv_bfloat16* out, int Bcap, int L, int H) {
    memset(&a, 0, sizeof(a));
    const uint64_t D = (uint64_t)H * 64;
    a.qkv = qkv, a.out = out, a.L = L, a.H = H, a.extras = L - 256, a.B = Bcap;
    a.scale_log2e = 0.125f * 1.4426950408889634f;
    DDB_TRY(make_tmap_bf16_3d(&a.tmQKV, qkv, 3 * D, L, Bcap, 3 * D * 2, (uint64_t)L * 3 * D * 2, 128));
    DDB_TRY(make_tmap_bf16_3d(&a.tmKV, qkv, 3 * D, L, Bcap, 3 * D * 2, (uint64_t)L * 3 * D * 2, 256));
    DDB_TRY(make_tmap_bf16_3d(&a.tmX, qkv, 3 * D, L, Bcap, 3 * D * 2, (uint64_t)L * 3 * D * 2, 16));
    DDB_TRY(make_tmap_bf16_3d(&a.tmOut, out, D, L, Bcap, D * 2, (uint64_t)L * D * 2, 128));
    DDB_TRY(make_tmap_bf16_3d(&a.tmOut32, out, D, L, Bcap, D * 2, (uint64_t)L * D * 2, 32));
    return DDB_OK;
}
static std::atomic<long long*> g_attn_trace{nullptr};  // bench-only (ddb_debug_set_ptr "attn_trace")
// persistent tcgen05 attention: one CTA per SM, (sample, head) work items; covers the extras rows too
static std::atomic<int> g_attn_x2{0};
static std::atomic<int> g_attn_direct{0};  // ddb_set_option "attn_direct": attention epilogue stores its rows straight from registers
                                           // (eight 16-byte global stores per thread) instead of staging + TMA store.  Measured
                                           // SLOWER: 42.0 vs 37.9 us per launch (ImageNet-64 shape 117.4 vs 96.6 us)
static std::atomic<int> g_attn_token{1};  // ddb_set_option "attn_token": the two query tiles alternate in the exp pass  // ddb_set_option "attn_x2": two softmax threads per query row (attention2.cuh)
static int launch_attention_tc(AttnArgs a, int B, int num_sms, cudaStream_t st, int force_x2 = -1) {
    static ddb_host::DeviceOnce configured;
    if (!configured.done()) {
        CUDA_TRY(cudaFuncSetAttribute(attention_tcgen05_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      ATT3_SMEM));
#ifdef DDB_EXPERIMENTAL
        CUDA_TRY(cudaFuncSetAttribute(attention_tcgen05_x2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      ATT4_SMEM));
#endif
        configured.mark();
    }
    if (B <= 0) return DDB_OK;
    a.B = B;
    a.trace = g_attn_trace;
    a.token = g_attn_token;
    a.direct_store = g_attn_direct;
    const int items = B * a.H;
    const dim3 grid(items < num_sms ? items : num_sms);
    if (force_x2 >= 0 ? force_x2 != 0 : g_attn_x2 != 0) {
#ifdef DDB_EXPERIMENTAL
        CUDA_TRY(launch_pdl(attention_tcgen05_x2_kernel, grid, dim3(ATT4_THREADS), ATT4_SMEM, st, a));
#else
        DDB_NEEDS_EXPERIMENTAL("attn_x2 (two softmax threads per query row)");
#endif
    } else {
        CUDA_TRY(launch_pdl(attention_tcgen05_kernel, grid, dim3(ATT3_THREADS), ATT3_SMEM, st, a));
    }
    LAUNCH_CHECK();
    return DDB_OK;
}

// generic-L mma.sync attention (experimental builds only: no reference config has L != 256 + extras)
static int launch_attention(const __nv_bfloat16* qkv, __nv_bfloat16* out, int B, int L, int H, cudaStream_t st) {
#ifdef DDB_EXPERIMENTAL
    const int Lp = (L + 15) & ~15;
    const int smem = 2 * Lp * 128;
    if (smem > 227 * 1024) return fail(DDB_ERR_INVALID, "sequence length %d too long for the resident-KV kernel", L);
    CUDA_TRY(cudaFuncSetAttribute(attention_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    if (B <= 0) return DDB_OK;
    attention_mma_kernel<<<B * H, ATT_THREADS, smem, st>>>(qkv, out, L, H, 0.125f * 1.4426950408889634f);
    LAUNCH_CHECK();
    return DDB_OK;
#else
    (void)qkv, (void)out, (void)B, (void)H, (void)st;
    return fail(DDB_ERR_INVALID, "attention with L = %d needs the generic mma.sync kernel: rebuild with DDB_EXPERIMENTAL=1 "
                                 "(the model path needs L = 256 + {1, 2})", L);
#endif
}

// ------------------------------------------------------------------------------------------------ model
struct DevMem {
    void* p = nullptr;
    ~DevMem() {
        if (p) cudaFree(p);
    }
    int alloc(size_t bytes) {
        if (bytes == 0) bytes = 16;
        CUDA_TRY(cudaMalloc(&p, bytes));
        return DDB_OK;
    }
    template <typename T>
    T* as() const {
        return reinterpret_cast<T*>(p);
    }
};
typedef std::unique_ptr<DevMem> Buf;

struct Linear {
    Buf w, bias, colsum;
    int N = 0, N_src = 0, K = 0;
};
struct BlockW {
    Linear qkv, proj, fc1, fc2, skip;
    bool has_skip = false;
};
struct HeadW {
    Linear dec;  // LN folded, N padded to 64
    Buf conv_w, conv_b;
};
struct BlockOps {
    GemmArgs skip, qkv, proj, fc1, fc2;
};

struct ddb_model {
    ddb_uvit_config cfg;
    DeviceInfo dev;
    int L = 0, Np = 0, extras = 0, pd = 0, D = 0, Hh = 0, Mmax = 0, Mpad = 0;
    size_t chw = 0;
    Buf pe_wt, pe_bias, pos, label_emb;
    Buf pe_w2, pos_patch, a_patch;  // tensor-core patch embed: [D,128] bf16 weight, bf16 pos rows, gathered patches
    GemmArgs embed_gemm;
    std::vector<BlockW> blocks;
    HeadW final_head;
    std::vector<HeadW> ee_heads;
    // MLP probes (models/early_exit.py:31-37, 194-204).  The kernels read the probe of layer i from the working set
    // probe_w [depth][D] / probe_b [depth].  probe_kind 1 (mlp_probe_per_layer): the working set IS the parameters.
    // 2 (mlp_probe_per_timestep: matrix["t"]) and 3 (mlp_probe_per_layer_per_timestep: matrix["i, t"]): the parameters
    // live in probe_tab_w [1000 (x depth)][D] / probe_tab_b and probe_select_kernel copies the depth rows of the current
    // timestep into the working set at the start of every forward (t from device memory: graph-replay safe).
    // 4 (attention_probe, early_exit.py:40-80): the working set holds u = Wk^T q / sqrt(D) per layer (the per-token
    // logits then come from the same partial dot products); ap_wc [depth][D][D] = W1 Wv, ap_bc = W1 bv + b1, ap_w2, ap_b2
    // feed attn_probe_score_kernel (elementwise.cuh).
    int probe_kind = 0;
    Buf probe_w, probe_b, probe_tab_w, probe_tab_b, ap_wc, ap_bc, ap_w2, ap_b2;
    float* pw(int i) const { return probe_w->as<float>() + (size_t)i * D; }
    float* pb(int i) const { return probe_b->as<float>() + i; }
    // mlp_time_embed = True (models/uvit.py:264-272): the MLP's weights, the table of the 1000 integer timesteps' time
    // tokens (what the sampler's steps use) and a [max_batch, D] scratch for a caller's arbitrary timesteps
    Buf te_w1, te_b1, te_w2, te_b2, time_tab, time_tok;
    // workspace
    Buf x0, xs, xm, qkv, ao, hbuf, stats, stats_p, img_pre, probe_p, scores, outputs, exit_idx;
    // early-exit compaction (mode 1): device-side live counts, slot maps, gather lists, scratch batch of leavers
    Buf ee_n, ee_slot, ee_dest, ee_exit_slot, ee_sc, ee_ticket, xe, stats_e;
    GemmArgs head_grp;                      // all leavers in one launch, head selected per sample (grouped decode)
    Buf hg_w, hg_bias, hg_colsum, hg_conv_w, hg_conv_b;  // the depth exit heads stacked for it
    std::vector<EeBufList> ee_live;         // buffers that must be compacted when samples leave before block i
    std::vector<int> ee_live_n;
    std::vector<Buf> xo;
    // plan
    std::vector<BlockOps> ops;
    GemmArgs final_dec;
    std::vector<GemmArgs> head_dec;
    AttnArgs attn;
    std::vector<Buf> keep;  // misc allocations
    // MLP in two half batches (see forward_impl): per batch size, the fc1 / fc2 descriptors of both halves of every block
    struct HalfOps {
        GemmArgs fc1[2], fc2[2];
    };
    std::map<int, std::vector<HalfOps>> mlp_split;
};

typedef std::map<std::string, const ddb_tensor*> TensorMap;

static int get_tensor(const TensorMap& tm, const std::string& name, int64_t numel, const float** out,
                      bool optional = false) {
    auto it = tm.find(name);
    if (it == tm.end()) {
        *out = nullptr;
        if (optional) return DDB_OK;
        return fail(DDB_ERR_MISSING_KEY, "state_dict key '%s' missing", name.c_str());
    }
    if (numel >= 0 && it->second->numel != numel)
        return fail(DDB_ERR_SHAPE, "state_dict key '%s' has %lld elements, expected %lld", name.c_str(),
                    (long long)it->second->numel, (long long)numel);
    *out = it->second->data_dev;
    return DDB_OK;
}

static int pack_linear(Linear& lin, const float* W, const float* bias, const float* gamma, const float* beta,
                       int N_src, int N_pad, int K, bool want_colsum) {
    lin.N = N_pad, lin.N_src = N_src, lin.K = K;
    lin.w.reset(new DevMem), lin.bias.reset(new DevMem), lin.colsum.reset(new DevMem);
    DDB_TRY(lin.w->alloc((size_t)N_pad * K * 2));
    DDB_TRY(lin.bias->alloc((size_t)N_pad * 4));
    DDB_TRY(lin.colsum->alloc((size_t)N_pad * 4));
    pack_linear_kernel<<<N_pad, 256>>>(W, bias, gamma, beta, N_src, K, lin.w->as<__nv_bfloat16>(),
                                       want_colsum ? lin.colsum->as<float>() : nullptr, lin.bias->as<float>());
    LAUNCH_CHECK();
    return DDB_OK;
}

static int load_block(ddb_model* m, const TensorMap& tm, const std::string& pfx, bool skip, BlockW& bw) {
    const int D = m->D, Hd = m->cfg.mlp_hidden;
    const float *g1, *b1, *g2, *b2, *w, *b;
    DDB_TRY(get_tensor(tm, pfx + "norm1.weight", D, &g1));
    DDB_TRY(get_tensor(tm, pfx + "norm1.bias", D, &b1));
    DDB_TRY(get_tensor(tm, pfx + "norm2.weight", D, &g2));
    DDB_TRY(get_tensor(tm, pfx + "norm2.bias", D, &b2));
    DDB_TRY(get_tensor(tm, pfx + "attn.qkv.weight", (int64_t)3 * D * D, &w));
    DDB_TRY(get_tensor(tm, pfx + "attn.qkv.bias", 3 * D, &b, true));
    DDB_TRY(pack_linear(bw.qkv, w, b, g1, b1, 3 * D, 3 * D, D, true));
    DDB_TRY(get_tensor(tm, pfx + "attn.proj.weight", (int64_t)D * D, &w));
    DDB_TRY(get_tensor(tm, pfx + "attn.proj.bias", D, &b));
    DDB_TRY(pack_linear(bw.proj, w, b, nullptr, nullptr, D, D, D, false));
    DDB_TRY(get_tensor(tm, pfx + "mlp.fc1.weight", (int64_t)Hd * D, &w));
    DDB_TRY(get_tensor(tm, pfx + "mlp.fc1.bias", Hd, &b));
    DDB_TRY(pack_linear(bw.fc1, w, b, g2, b2, Hd, Hd, D, true));
    DDB_TRY(get_tensor(tm, pfx + "mlp.fc2.weight", (int64_t)D * Hd, &w));
    DDB_TRY(get_tensor(tm, pfx + "mlp.fc2.bias", D, &b));
    DDB_TRY(pack_linear(bw.fc2, w, b, nullptr, nullptr, D, D, Hd, false));
    // UViT(skip=False) (models/uvit.py:200-204): the out-blocks have no skip_linear and ignore the popped skip
    if (skip) DDB_TRY(get_tensor(tm, pfx + "skip_linear.weight", (int64_t)2 * D * D, &w, true));
    bw.has_skip = skip && w != nullptr;
    if (bw.has_skip) {
        DDB_TRY(get_tensor(tm, pfx + "skip_linear.weight", (int64_t)2 * D * D, &w));
        DDB_TRY(get_tensor(tm, pfx + "skip_linear.bias", D, &b));
        DDB_TRY(pack_linear(bw.skip, w, b, nullptr, nullptr, D, D, 2 * D, false));
    }
    return DDB_OK;
}

static int load_head(ddb_model* m, const TensorMap& tm, const std::string& pfx, HeadW& hw) {
    const int D = m->D, C = m->cfg.in_chans;
    const float *g, *b, *w, *wb, *cw, *cb;
    DDB_TRY(get_tensor(tm, pfx + "norm.weight", D, &g));
    DDB_TRY(get_tensor(tm, pfx + "norm.bias", D, &b));
    DDB_TRY(get_tensor(tm, pfx + "decoder_pred.weight", (int64_t)m->pd * D, &w));
    DDB_TRY(get_tensor(tm, pfx + "decoder_pred.bias", m->pd, &wb));
    DDB_TRY(pack_linear(hw.dec, w, wb, g, b, m->pd, 64, D, true));
    DDB_TRY(get_tensor(tm, pfx + "final_layer.weight", (int64_t)C * C * 9, &cw, true));
    hw.conv_w.reset(new DevMem), hw.conv_b.reset(new DevMem);
    DDB_TRY(hw.conv_w->alloc((size_t)C * C * 9 * 4));
    DDB_TRY(hw.conv_b->alloc((size_t)C * 4));
    if (!cw) {
        // conv=False (models/uvit.py:329-333, early_exit.py:17-21): final_layer is nn.Identity().  The conv kernels run
        // with the identity stencil (centre tap 1 on the channel diagonal, zero bias): fma(1, x, 0 + 0*..) == x exactly
        std::vector<float> idw((size_t)C * C * 9, 0.f);
        for (int ch = 0; ch < C; ++ch) idw[((size_t)ch * C + ch) * 9 + 4] = 1.f;
        CUDA_TRY(cudaMemcpy(hw.conv_w->p, idw.data(), idw.size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemset(hw.conv_b->p, 0, (size_t)C * 4));
        return DDB_OK;
    }
    DDB_TRY(get_tensor(tm, pfx + "final_layer.bias", C, &cb));
    CUDA_TRY(cudaMemcpy(hw.conv_w->p, cw, (size_t)C * C * 9 * 4, cudaMemcpyDeviceToDevice));
    CUDA_TRY(cudaMemcpy(hw.conv_b->p, cb, (size_t)C * 4, cudaMemcpyDeviceToDevice));
    return DDB_OK;
}

static int new_buf(Buf& b, size_t bytes, bool zero = true) {
    b.reset(new DevMem);
    DDB_TRY(b->alloc(bytes));
    if (zero) CUDA_TRY(cudaMemset(b->p, 0, bytes));
    return DDB_OK;
}

// Fill the shape/pointer fields + descriptors of one GEMM of the plan.
static int plan_gemm(GemmArgs& g, const ddb_model* m, const void* A0, int K0, const void* A1, int K1, const Linear& W,
                     int BN, const void* out, const void* res, const float2* stats) {
    memset(&g, 0, sizeof(g));
    g.M = m->Mmax, g.N = W.N, g.K0 = K0, g.K1 = K1;
    g.bias = W.bias->as<float>();
    g.colsum = W.colsum->as<float>();
    g.stats = stats;
    g.nparts = 1, g.ln_dim = m->D, g.ln_eps = m->cfg.ln_eps;
    DDB_TRY(make_tmap_bf16(&g.tmA0, A0, m->Mpad, K0, K0, 128));
    if (K1 > 0) DDB_TRY(make_tmap_bf16(&g.tmA1, A1, m->Mpad, K1, K1, 128));
    DDB_TRY(make_tmap_bf16(&g.tmB, W.w->p, W.N, K0 + K1, K0 + K1, BN));
    if (BN == 256) DDB_TRY(make_tmap_bf16(&g.tmB2, W.w->p, W.N, K0 + K1, K0 + K1, 128));
    if (BN == 256) DDB_TRY(make_tmap_bf16(&g.tmB3, W.w->p, W.N, K0 + K1, K0 + K1, 64));
    if (out) DDB_TRY(make_tmap_bf16(&g.tmOut, out, m->Mpad, W.N, W.N, 128));
    if (res) DDB_TRY(make_tmap_bf16(&g.tmRes, res, m->Mpad, W.N, W.N, 128));
    if (out && BN == 256) DDB_TRY(make_tmap_bf16_sw64(&g.tmOut2, out, m->Mpad, W.N, W.N, 128));
    if (res && BN == 256) DDB_TRY(make_tmap_bf16_sw64(&g.tmRes2, res, m->Mpad, W.N, W.N, 128));
    return DDB_OK;
}
// Copy of a planned GEMM restricted to `rows` rows starting at row `row0` of its A / out / residual tensors.  The maps
// cover exactly those rows, so the partial last tile is clipped by TMA (it must not touch the other half's rows).
static int retarget_rows(GemmArgs& g, const GemmArgs& src, const void* A0, const void* out, const void* res, int row0,
                         int rows) {
    g = src;
    g.M = rows;
    const char* a = reinterpret_cast<const char*>(A0) + (size_t)row0 * src.K0 * 2;
    DDB_TRY(make_tmap_bf16(&g.tmA0, a, rows, src.K0, src.K0, 128));
    if (out) {
        char* o = reinterpret_cast<char*>(const_cast<void*>(out)) + (size_t)row0 * src.N * 2;
        DDB_TRY(make_tmap_bf16(&g.tmOut, o, rows, src.N, src.N, 128));
        DDB_TRY(make_tmap_bf16_sw64(&g.tmOut2, o, rows, src.N, src.N, 128));
    }
    if (res) {
        const char* r = reinterpret_cast<const char*>(res) + (size_t)row0 * src.N * 2;
        DDB_TRY(make_tmap_bf16(&g.tmRes, r, rows, src.N, src.N, 128));
        DDB_TRY(make_tmap_bf16_sw64(&g.tmRes2, r, rows, src.N, src.N, 128));
    }
    return DDB_OK;
}

static void plan_decode_geometry(GemmArgs& g, const ddb_model* m, float* img) {
    g.img = img;
    g.L = m->L, g.extras = m->extras, g.C = m->cfg.in_chans, g.P = m->cfg.patch_size;
    g.Wp = m->cfg.img_size / m->cfg.patch_size, g.H = m->cfg.img_size, g.W = m->cfg.img_size;
    g.patch_dim = m->pd;
}

static int model_create_impl(const ddb_uvit_config* cfg, const ddb_tensor* tensors, int n_tensors, ddb_model* m) {
    m->cfg = *cfg;
    DDB_TRY(device_info(m->dev));
    const int D = cfg->embed_dim, P = cfg->patch_size, C = cfg->in_chans;
    if (cfg->img_size % P) return fail(DDB_ERR_INVALID, "img_size %% patch_size != 0");
    if (cfg->img_size / P != EMB_TOK)
        return fail(DDB_ERR_INVALID, "img_size/patch_size must be 16 (every reference config), got %d",
                    cfg->img_size / P);
    if (cfg->img_size % CONV_BAND) return fail(DDB_ERR_INVALID, "img_size must be a multiple of 16");
    if (D % 256 || D / cfg->num_heads != 64 || D % cfg->num_heads)
        return fail(DDB_ERR_INVALID, "embed_dim must be a multiple of 256 with head_dim 64 (got %d / %d heads)", D,
                    cfg->num_heads);
    if (cfg->mlp_hidden % 256) return fail(DDB_ERR_INVALID, "mlp_hidden must be a multiple of 256");
    if (cfg->depth < 1 || cfg->depth % 2 == 0) return fail(DDB_ERR_INVALID, "depth must be odd");
    if (cfg->max_batch < 1) return fail(DDB_ERR_INVALID, "max_batch must be >= 1");
    m->D = D, m->Hh = cfg->num_heads;
    m->Np = (cfg->img_size / P) * (cfg->img_size / P);
    m->extras = cfg->num_classes > 0 ? 2 : 1;
    m->L = m->Np + m->extras;
    m->pd = P * P * C;
    if (m->pd > 64) return fail(DDB_ERR_INVALID, "patch_dim %d > 64 unsupported", m->pd);
    m->chw = (size_t)C * cfg->img_size * cfg->img_size;
    if (m->chw % 4) return fail(DDB_ERR_INVALID, "C*H*W must be a multiple of 4");
    m->Mmax = cfg->max_batch * m->L;
    m->Mpad = (m->Mmax + 127) / 128 * 128;

    TensorMap tm;
    const std::string up = cfg->early_exit ? "uvit." : "";
    for (int i = 0; i < n_tensors; ++i) tm[tensors[i].name] = &tensors[i];

    // ---- embeddings
    const float *pw, *pb, *pos, *lab;
    DDB_TRY(get_tensor(tm, up + "patch_embed.proj.weight", (int64_t)D * m->pd, &pw));
    DDB_TRY(get_tensor(tm, up + "patch_embed.proj.bias", D, &pb));
    DDB_TRY(get_tensor(tm, up + "pos_embed", (int64_t)m->L * D, &pos));
    DDB_TRY(new_buf(m->pe_wt, (size_t)m->pd * D * 4));
    transpose_pe_kernel<<<(D * m->pd + 255) / 256, 256>>>(pw, D, m->pd, m->pe_wt->as<float>());
    LAUNCH_CHECK();
    DDB_TRY(new_buf(m->pe_bias, (size_t)D * 4));
    CUDA_TRY(cudaMemcpy(m->pe_bias->p, pb, (size_t)D * 4, cudaMemcpyDeviceToDevice));
    DDB_TRY(new_buf(m->pos, (size_t)m->L * D * 4));
    CUDA_TRY(cudaMemcpy(m->pos->p, pos, (size_t)m->L * D * 4, cudaMemcpyDeviceToDevice));
    DDB_TRY(new_buf(m->pe_w2, (size_t)D * 128 * 2));
    pack_patch_embed_kernel<<<(D * 128 + 255) / 256, 256>>>(pw, D, m->pd, m->pe_w2->as<__nv_bfloat16>());
    LAUNCH_CHECK();
    DDB_TRY(new_buf(m->pos_patch, (size_t)m->Np * D * 2));
    cast_bf16_kernel<<<(unsigned)(((size_t)m->Np * D + 255) / 256), 256>>>(pos + (size_t)m->extras * D,
                                                                         m->pos_patch->as<__nv_bfloat16>(),
                                                                         (size_t)m->Np * D);
    LAUNCH_CHECK();
    DDB_TRY(new_buf(m->a_patch, (size_t)cfg->max_batch * m->Np * 128 * 2));  // zero: the K padding stays zero
    if (cfg->num_classes > 0) {
        DDB_TRY(get_tensor(tm, up + "label_emb.weight", (int64_t)cfg->num_classes * D, &lab));
        DDB_TRY(new_buf(m->label_emb, (size_t)cfg->num_classes * D * 4));
        CUDA_TRY(cudaMemcpy(m->label_emb->p, lab, (size_t)cfg->num_classes * D * 4, cudaMemcpyDeviceToDevice));
    }
    {
        const float *w1, *b1, *w2, *b2;
        DDB_TRY(get_tensor(tm, up + "time_embed.0.weight", (int64_t)4 * D * D, &w1, true));
        if (w1) {
            DDB_TRY(get_tensor(tm, up + "time_embed.0.bias", 4 * D, &b1));
            DDB_TRY(get_tensor(tm, up + "time_embed.2.weight", (int64_t)4 * D * D, &w2));
            DDB_TRY(get_tensor(tm, up + "time_embed.2.bias", D, &b2));
            DDB_TRY(new_buf(m->te_w1, (size_t)4 * D * D * 4));
            DDB_TRY(new_buf(m->te_b1, (size_t)4 * D * 4));
            DDB_TRY(new_buf(m->te_w2, (size_t)4 * D * D * 4));
            DDB_TRY(new_buf(m->te_b2, (size_t)D * 4));
            CUDA_TRY(cudaMemcpy(m->te_w1->p, w1, (size_t)4 * D * D * 4, cudaMemcpyDeviceToDevice));
            CUDA_TRY(cudaMemcpy(m->te_b1->p, b1, (size_t)4 * D * 4, cudaMemcpyDeviceToDevice));
            CUDA_TRY(cudaMemcpy(m->te_w2->p, w2, (size_t)4 * D * D * 4, cudaMemcpyDeviceToDevice));
            CUDA_TRY(cudaMemcpy(m->te_b2->p, b2, (size_t)D * 4, cudaMemcpyDeviceToDevice));
            DDB_TRY(new_buf(m->time_tab, (size_t)1000 * D * 4));
            DDB_TRY(new_buf(m->time_tok, (size_t)cfg->max_batch * D * 4));
            time_mlp_kernel<<<1000, 256, (size_t)5 * D * 4>>>(nullptr, (int)cfg->normalize_timesteps, D,
                                                              m->te_w1->as<float>(), m->te_b1->as<float>(),
                                                              m->te_w2->as<float>(), m->te_b2->as<float>(),
                                                              m->time_tab->as<float>());
            LAUNCH_CHECK();
        }
    }
    // ---- blocks
    const int half = cfg->depth / 2;
    m->blocks.resize(cfg->depth);
    for (int i = 0; i < half; ++i)
        DDB_TRY(load_block(m, tm, up + "in_blocks." + std::to_string(i) + ".", false, m->blocks[i]));
    DDB_TRY(load_block(m, tm, up + "mid_block.", false, m->blocks[half]));
    for (int i = 0; i < half; ++i)
        DDB_TRY(load_block(m, tm, up + "out_blocks." + std::to_string(i) + ".", true, m->blocks[half + 1 + i]));
    DDB_TRY(load_head(m, tm, up, m->final_head));
    if (cfg->early_exit) {
        m->ee_heads.resize(cfg->depth);
        m->probe_kind = cfg->early_exit;
        if (m->probe_kind < 1 || m->probe_kind > 4)
            return fail(DDB_ERR_INVALID, "early_exit must be 0 (plain), 1 (mlp_probe_per_layer), 2 (mlp_probe_per_timestep), "
                                         "3 (mlp_probe_per_layer_per_timestep) or 4 (attention_probe)");
        DDB_TRY(new_buf(m->probe_w, (size_t)cfg->depth * D * 4));
        DDB_TRY(new_buf(m->probe_b, (size_t)cfg->depth * 4));
        auto load_probe = [&](const std::string& key, float* w_dst, float* b_dst) -> int {
            const float *w, *b;
            const std::string pp = "matrix." + key + ".classifier.0.";
            DDB_TRY(get_tensor(tm, pp + "weight", D, &w));
            DDB_TRY(get_tensor(tm, pp + "bias", 1, &b));
            CUDA_TRY(cudaMemcpyAsync(w_dst, w, (size_t)D * 4, cudaMemcpyDeviceToDevice, 0));
            CUDA_TRY(cudaMemcpyAsync(b_dst, b, 4, cudaMemcpyDeviceToDevice, 0));
            return DDB_OK;
        };
        if (m->probe_kind == 4) {
            DDB_TRY(new_buf(m->ap_wc, (size_t)cfg->depth * D * D * 4));
            DDB_TRY(new_buf(m->ap_bc, (size_t)cfg->depth * D * 4));
            DDB_TRY(new_buf(m->ap_w2, (size_t)cfg->depth * D * 4));
            DDB_TRY(new_buf(m->ap_b2, (size_t)cfg->depth * 4));
            for (int i = 0; i < cfg->depth; ++i) {
                const std::string pp = "matrix." + std::to_string(i) + ".";
                const float *q, *wkv, *bkv, *w1, *b1, *w2, *b2;
                DDB_TRY(get_tensor(tm, pp + "q", D, &q));  // [1, num_heads = 1, 1, D]
                DDB_TRY(get_tensor(tm, pp + "weight_kv.weight", (int64_t)2 * D * D, &wkv));
                DDB_TRY(get_tensor(tm, pp + "weight_kv.bias", 2 * D, &bkv));
                DDB_TRY(get_tensor(tm, pp + "classification.0.weight", (int64_t)D * D, &w1));
                DDB_TRY(get_tensor(tm, pp + "classification.0.bias", D, &b1));
                DDB_TRY(get_tensor(tm, pp + "classification.2.weight", D, &w2));
                DDB_TRY(get_tensor(tm, pp + "classification.2.bias", 1, &b2));
                attn_probe_pack_kernel<<<dim3(D, 2), 256>>>(q, wkv, bkv, w1, b1, D, m->pw(i),
                                                            m->ap_wc->as<float>() + (size_t)i * D * D,
                                                            m->ap_bc->as<float>() + (size_t)i * D);
                LAUNCH_CHECK();
                CUDA_TRY(cudaMemcpyAsync(m->ap_w2->as<float>() + (size_t)i * D, w2, (size_t)D * 4, cudaMemcpyDeviceToDevice, 0));
                CUDA_TRY(cudaMemcpyAsync(m->ap_b2->as<float>() + i, b2, 4, cudaMemcpyDeviceToDevice, 0));
            }
        } else if (m->probe_kind > 1) {
            const int n = m->probe_kind == 2 ? 1000 : 1000 * cfg->depth;
            DDB_TRY(new_buf(m->probe_tab_w, (size_t)n * D * 4));
            DDB_TRY(new_buf(m->probe_tab_b, (size_t)n * 4));
            for (int t = 0; t < 1000; ++t) {
                if (m->probe_kind == 2) {
                    DDB_TRY(load_probe(std::to_string(t), m->probe_tab_w->as<float>() + (size_t)t * D,
                                       m->probe_tab_b->as<float>() + t));
                } else {
                    for (int i = 0; i < cfg->depth; ++i) {
                        const size_t r = (size_t)t * cfg->depth + i;  // row of matrix["i, t"]
                        DDB_TRY(load_probe(std::to_string(i) + ", " + std::to_string(t),
                                           m->probe_tab_w->as<float>() + r * D, m->probe_tab_b->as<float>() + r));
                    }
                }
            }
        }
        for (int i = 0; i < cfg->depth; ++i) {
            std::string hp = i < half    ? "in_blocks_heads." + std::to_string(i) + "."
                             : i == half ? std::string("mid_block_head.")
                                         : "out_blocks_heads." + std::to_string(i - half - 1) + ".";
            DDB_TRY(load_head(m, tm, hp, m->ee_heads[i]));
            if (m->probe_kind == 1) DDB_TRY(load_probe(std::to_string(i), m->pw(i), m->pb(i)));
        }
        CUDA_TRY(cudaStreamSynchronize(0));
    }
    // ---- workspace
    const size_t act = (size_t)m->Mpad * D * 2;
    DDB_TRY(new_buf(m->x0, act));
    DDB_TRY(new_buf(m->xs, act));
    DDB_TRY(new_buf(m->xm, act));
    DDB_TRY(new_buf(m->ao, act));
    DDB_TRY(new_buf(m->qkv, act * 3));
    DDB_TRY(new_buf(m->hbuf, (size_t)m->Mpad * cfg->mlp_hidden * 2));
    DDB_TRY(new_buf(m->stats, (size_t)m->Mpad * sizeof(float2)));
    DDB_TRY(new_buf(m->stats_p, (size_t)m->Mpad * (D / 64) * sizeof(float2)));
    DDB_TRY(new_buf(m->img_pre, (size_t)cfg->max_batch * m->chw * 4));
    m->xo.resize(cfg->depth);
    for (int i = 0; i < cfg->depth; ++i) DDB_TRY(new_buf(m->xo[i], act));
    if (cfg->early_exit) {
        DDB_TRY(new_buf(m->probe_p, (size_t)m->Mpad * (D / 64) * 4));
        DDB_TRY(new_buf(m->scores, (size_t)cfg->depth * cfg->max_batch * 4));
        DDB_TRY(new_buf(m->outputs, (size_t)(cfg->depth + 1) * cfg->max_batch * m->chw * 4));
        DDB_TRY(new_buf(m->exit_idx, (size_t)cfg->max_batch * 4));
        DDB_TRY(new_buf(m->ee_n, 8 * 4));
        DDB_TRY(new_buf(m->ee_slot, (size_t)cfg->max_batch * 4));
        DDB_TRY(new_buf(m->ee_dest, (size_t)cfg->max_batch * 2 * 4));  // leavers' positions | the stayers that replace them
        DDB_TRY(new_buf(m->ee_sc, (size_t)cfg->max_batch * 4));
        DDB_TRY(new_buf(m->ee_ticket, 4));
        DDB_TRY(new_buf(m->ee_exit_slot, (size_t)cfg->max_batch * 4));
        DDB_TRY(new_buf(m->xe, act));
        DDB_TRY(new_buf(m->stats_e, (size_t)m->Mpad * (D / 64) * sizeof(float2)));
    }
    // ---- plan (buffer routing of models/uvit.py:367-375)
    m->ops.resize(cfg->depth);
    const float2* st = m->stats->as<float2>();
    const void* cur = m->x0->p;
    std::vector<const void*> skips;
    for (int i = 0; i < cfg->depth; ++i) {
        BlockW& bw = m->blocks[i];
        BlockOps& op = m->ops[i];
        if (bw.has_skip) {
            const void* sk = skips.back();
            skips.pop_back();
            DDB_TRY(plan_gemm(op.skip, m, cur, D, sk, D, bw.skip, 256, m->xs->p, nullptr, nullptr));
            cur = m->xs->p;
        }
        DDB_TRY(plan_gemm(op.qkv, m, cur, D, nullptr, 0, bw.qkv, 256, m->qkv->p, nullptr, st));
        DDB_TRY(plan_gemm(op.proj, m, m->ao->p, D, nullptr, 0, bw.proj, 256, m->xm->p, cur, nullptr));
        DDB_TRY(plan_gemm(op.fc1, m, m->xm->p, D, nullptr, 0, bw.fc1, 256, m->hbuf->p, nullptr, st));
        DDB_TRY(plan_gemm(op.fc2, m, m->hbuf->p, cfg->mlp_hidden, nullptr, 0, bw.fc2, 256, m->xo[i]->p, m->xm->p,
                          nullptr));
        cur = m->xo[i]->p;
        if (i < half) skips.push_back(cur);
    }
    DDB_TRY(plan_attention(m->attn, m->qkv->as<__nv_bfloat16>(), m->ao->as<__nv_bfloat16>(), cfg->max_batch, m->L,
                           m->Hh));
    {
        // patch embed as a GEMM: [B*256, 128] x [D, 128]^T, output rows scattered to the token buffer (3-D map)
        GemmArgs& g = m->embed_gemm;
        memset(&g, 0, sizeof(g));
        const uint64_t rowsA = (uint64_t)cfg->max_batch * m->Np;
        g.M = (int)rowsA, g.N = D, g.K0 = 128, g.K1 = 0;
        g.bias = m->pe_bias->as<float>();
        g.nparts = 1, g.ln_dim = D, g.ln_eps = cfg->ln_eps;
        g.embed_mode = 1, g.tok_L = m->L, g.tok_extras = m->extras;
        DDB_TRY(make_tmap_bf16(&g.tmA0, m->a_patch->p, rowsA, 128, 128, 128));
        DDB_TRY(make_tmap_bf16(&g.tmB, m->pe_w2->p, D, 128, 128, 256));
        DDB_TRY(make_tmap_bf16(&g.tmB2, m->pe_w2->p, D, 128, 128, 128));
        DDB_TRY(make_tmap_bf16(&g.tmB3, m->pe_w2->p, D, 128, 128, 64));
        DDB_TRY(make_tmap_bf16_3d(&g.tmOut, m->x0->as<__nv_bfloat16>() + (size_t)m->extras * D, D, m->Np,
                                  cfg->max_batch, (uint64_t)D * 2, (uint64_t)m->L * D * 2, 128));
        DDB_TRY(make_tmap_bf16(&g.tmRes, m->pos_patch->p, m->Np, D, D, 128));
    }
    DDB_TRY(plan_gemm(m->final_dec, m, cur, D, nullptr, 0, m->final_head.dec, 64, nullptr, nullptr, st));
    plan_decode_geometry(m->final_dec, m, m->img_pre->as<float>());
    if (cfg->early_exit) {
        m->head_dec.resize(cfg->depth);
        for (int i = 0; i < cfg->depth; ++i) {
            // head i reads the input of block i (models/early_exit.py:291-313)
            const void* in = (i == 0) ? m->x0->p : m->xo[i - 1]->p;
            DDB_TRY(plan_gemm(m->head_dec[i], m, in, D, nullptr, 0, m->ee_heads[i].dec, 64, nullptr, nullptr, st));
            plan_decode_geometry(m->head_dec[i], m, m->img_pre->as<float>());
        }
        // compaction mode: head i on the scratch batch of leavers; list of live buffers per layer = the block input
        // plus every long skip that is still pending (models/uvit.py:367-375)
        m->ee_live.resize(cfg->depth);
        m->ee_live_n.resize(cfg->depth);
        {
            // the exit heads stacked: decoder weights [depth][64][D] bf16 (LayerNorm folded), bias / colsum [depth][64],
            // conv weights [depth][C*C*9], conv bias [depth][C]
            const int dpt = cfg->depth;
            const size_t wb = (size_t)64 * D * 2, cw = (size_t)C * C * 9 * 4;
            DDB_TRY(new_buf(m->hg_w, wb * dpt));
            DDB_TRY(new_buf(m->hg_bias, (size_t)dpt * 64 * 4));
            DDB_TRY(new_buf(m->hg_colsum, (size_t)dpt * 64 * 4));
            DDB_TRY(new_buf(m->hg_conv_w, cw * dpt));
            DDB_TRY(new_buf(m->hg_conv_b, (size_t)dpt * C * 4));
            for (int i = 0; i < dpt; ++i) {
                const HeadW& hw = m->ee_heads[i];
                CUDA_TRY(cudaMemcpy(m->hg_w->as<char>() + wb * i, hw.dec.w->p, wb, cudaMemcpyDeviceToDevice));
                CUDA_TRY(cudaMemcpy(m->hg_bias->as<float>() + 64 * i, hw.dec.bias->p, 64 * 4, cudaMemcpyDeviceToDevice));
                CUDA_TRY(cudaMemcpy(m->hg_colsum->as<float>() + 64 * i, hw.dec.colsum->p, 64 * 4, cudaMemcpyDeviceToDevice));
                CUDA_TRY(cudaMemcpy(m->hg_conv_w->as<char>() + cw * i, hw.conv_w->p, cw, cudaMemcpyDeviceToDevice));
                CUDA_TRY(cudaMemcpy(m->hg_conv_b->as<float>() + C * i, hw.conv_b->p, C * 4, cudaMemcpyDeviceToDevice));
            }
            GemmArgs& g = m->head_grp;
            memset(&g, 0, sizeof(g));
            g.M = m->Mmax, g.N = 64, g.K0 = D, g.K1 = 0;
            g.bias = m->hg_bias->as<float>(), g.colsum = m->hg_colsum->as<float>();
            g.stats = m->stats_e->as<float2>();
            g.nparts = D / 64, g.ln_dim = D, g.ln_eps = cfg->ln_eps;
            DDB_TRY(make_tmap_bf16_3d(&g.tmA0, m->xe->p, D, m->L, cfg->max_batch, (uint64_t)D * 2,
                                      (uint64_t)m->L * D * 2, 128));
            DDB_TRY(make_tmap_bf16_3d(&g.tmB, m->hg_w->p, D, 64, dpt, (uint64_t)D * 2, (uint64_t)64 * D * 2, 64));
            plan_decode_geometry(g, m, m->img_pre->as<float>());
            g.grp_depth = dpt;
        }
        for (int i = 0; i < cfg->depth; ++i) {
            const int last_skip = (i <= half) ? std::min(i, half) - 1 : half - 1 - (i - half - 1);
            EeBufList& bl = m->ee_live[i];
            memset(&bl, 0, sizeof(bl));
            int n = 0;
            void* cur_in = (i == 0) ? m->x0->p : m->xo[i - 1]->p;
            bl.p[n++] = reinterpret_cast<__nv_bfloat16*>(cur_in);
            for (int k = 0; k <= last_skip; ++k) {
                if (m->xo[k]->p == cur_in) continue;
                if (n >= EE_MAX_LIVE)
                    return fail(DDB_ERR_INVALID, "depth %d needs more than %d live buffers", cfg->depth, EE_MAX_LIVE);
                bl.p[n++] = m->xo[k]->as<__nv_bfloat16>();
            }
            m->ee_live_n[i] = n;
        }
    }
    CUDA_TRY(cudaDeviceSynchronize());
    return DDB_OK;
}

static int run_conv(const ddb_model* m, const HeadW& hw, const float* in, float* out, int B, cudaStream_t st,
                    const int* n_dev = nullptr, const int* slot_map = nullptr, const int* layer_idx = nullptr) {
    const int C = m->cfg.in_chans, H = m->cfg.img_size, W = m->cfg.img_size;
    const size_t smem = (size_t)C * (CONV_BAND + 2) * (W + 8) * 4;
    const dim3 grid(B * (H / CONV_BAND));
    // layer_idx: grouped mode -- image b takes the stacked exit head layer_idx[b] (hw is ignored)
    const float* w = layer_idx ? m->hg_conv_w->as<float>() : hw.conv_w->as<float>();
    const float* bs = layer_idx ? m->hg_conv_b->as<float>() : hw.conv_b->as<float>();
    const int depth = m->cfg.depth;
    ProfScope ps(PC_CONV);
    switch (C) {
        case 3: CUDA_TRY(launch_pdl(conv3x3_kernel<3>, grid, dim3(256), smem, st, in, w, bs, out, H, W, n_dev, slot_map, layer_idx, depth)); break;
        case 4: CUDA_TRY(launch_pdl(conv3x3_kernel<4>, grid, dim3(256), smem, st, in, w, bs, out, H, W, n_dev, slot_map, layer_idx, depth)); break;
        default: return fail(DDB_ERR_INVALID, "in_chans %d unsupported by the final 3x3 conv (3 or 4)", C);
    }
    LAUNCH_CHECK();
    return DDB_OK;
}

// Compaction-mode parameters of a forward (ddb_ee_forward mode 1)
struct EeCompact {
    float threshold;
    int32_t* exit_idx;     // [B]
    const int* t_dev;      // device timestep for the logs (or null)
    int32_t* exit_log;     // [1000,B] by t (or null)
    float* score_mean_log; // [1000,depth] by t (or null)
};

// Inside the sampler (plain U-ViT path) a step is fused at both ends: the previous step's tail kernel has already
// written this forward's patch matrix and time / label token rows, and this forward ends in step_tail_kernel (3x3
// conv + DDPM update + the head of the next step) instead of conv3x3.  `tail` carries that kernel's arguments.
struct StepFuse {
    TailArgs tail;
};
// row0: first row of the patch matrix written (the guided sampler gathers x into rows [0, B) and [B, 2B))
static int launch_patch_gather(const ddb_model* m, const float* x, int B, cudaStream_t st, int row0 = 0) {
    const ddb_uvit_config& c = m->cfg;
    const size_t n_thr = (size_t)B * c.in_chans * c.img_size * (c.img_size / c.patch_size);
    CUDA_TRY(launch_pdl(patch_gather_kernel, dim3((unsigned)((n_thr + 255) / 256)), dim3(256), 0, st, x,
                        m->a_patch->as<__nv_bfloat16>() + (size_t)row0 * m->Np * 128, B, (int)c.in_chans,
                        (int)c.img_size, (int)c.img_size, (int)c.patch_size));
    LAUNCH_CHECK();
    return DDB_OK;
}
static int launch_token_extras(const ddb_model* m, const float* t_vec, const int* t_dev, const int64_t* y, int B,
                               cudaStream_t st) {
    const float *rows = nullptr, *tab = nullptr;
    if (m->time_tab) {  // mlp_time_embed: table row of the step, or the MLP on the caller's timesteps
        tab = m->time_tab->as<float>();
        if (!t_dev) {
            rows = m->time_tok->as<float>();
            CUDA_TRY(launch_pdl(time_mlp_kernel, dim3(B), dim3(256), (size_t)5 * m->D * 4, st, t_vec,
                                (int)m->cfg.normalize_timesteps, m->D, (const float*)m->te_w1->as<float>(),
                                (const float*)m->te_b1->as<float>(), (const float*)m->te_w2->as<float>(),
                                (const float*)m->te_b2->as<float>(), m->time_tok->as<float>()));
            LAUNCH_CHECK();
        }
    }
    CUDA_TRY(launch_pdl(token_extras_kernel, dim3(B), dim3(256), 0, st, t_vec, t_dev,
                        reinterpret_cast<const long long*>(y), (const float*)m->pos->as<float>(),
                        (const float*)(m->label_emb ? m->label_emb->as<float>() : nullptr),
                        m->x0->as<__nv_bfloat16>(), m->stats_p->as<float2>(), m->D, m->L, m->extras,
                        (int)m->cfg.normalize_timesteps, (int)m->cfg.num_classes, rows, tab));
    LAUNCH_CHECK();
    return DDB_OK;
}
template <bool G, int K>
static void (*ms_tail_kernel(int C, int W))(TailArgs) {
    if (C == 3 && W == 64) return step_tail_kernel<3, 64, G, K>;
    if (C == 3 && W == 32) return step_tail_kernel<3, 32, G, K>;
    if (C == 4 && W == 32) return step_tail_kernel<4, 32, G, K>;
    if (C == 4 && W == 64) return step_tail_kernel<4, 64, G, K>;
    return nullptr;
}
// B: rows of the forward; a guided tail runs one CTA per guided sample (ta.B = B / 2) and band
static int launch_step_tail(const ddb_model* m, const TailArgs& ta, int B, cudaStream_t st) {
    const int C = m->cfg.in_chans, H = m->cfg.img_size, W = m->cfg.img_size;
    const dim3 grid((ta.guide ? ta.B : B) * (H / CONV_BAND));
    ProfScope ps(PC_TAIL);
    if (ta.mode == 3) {  // DPM-Solver++(2M): the multistep instantiations, guided or not
        void (*k)(TailArgs) = ta.guide ? ms_tail_kernel<true, TAIL_DPM2M>(C, W) : ms_tail_kernel<false, TAIL_DPM2M>(C, W);
        if (!k) return fail(DDB_ERR_INVALID, "sample shape [%d,%d,%d] unsupported by the multistep step tail", C, H, W);
        CUDA_TRY(launch_pdl(k, grid, dim3(256), 0, st, ta));
    } else if (ta.mode == 4) {  // UniPC: the predictor-corrector instantiations, guided or not
        void (*k)(TailArgs) = ta.guide ? ms_tail_kernel<true, TAIL_UNIPC>(C, W) : ms_tail_kernel<false, TAIL_UNIPC>(C, W);
        if (!k) return fail(DDB_ERR_INVALID, "sample shape [%d,%d,%d] unsupported by the UniPC step tail", C, H, W);
        CUDA_TRY(launch_pdl(k, grid, dim3(256), 0, st, ta));
    } else if (ta.mode == 5) {  // SDE-DPM-Solver++(2M): the stochastic multistep instantiations, guided or not
        void (*k)(TailArgs) = ta.guide ? ms_tail_kernel<true, TAIL_SDE2M>(C, W) : ms_tail_kernel<false, TAIL_SDE2M>(C, W);
        if (!k)
            return fail(DDB_ERR_INVALID, "sample shape [%d,%d,%d] unsupported by the SDE-DPM-Solver++ step tail", C, H, W);
        CUDA_TRY(launch_pdl(k, grid, dim3(256), 0, st, ta));
    } else if (ta.guide) {
        if (C == 3 && W == 64)
            CUDA_TRY(launch_pdl(step_tail_kernel<3, 64, true>, grid, dim3(256), 0, st, ta));
        else if (C == 3 && W == 32)
            CUDA_TRY(launch_pdl(step_tail_kernel<3, 32, true>, grid, dim3(256), 0, st, ta));
        else if (C == 4 && W == 32)
            CUDA_TRY(launch_pdl(step_tail_kernel<4, 32, true>, grid, dim3(256), 0, st, ta));
        else if (C == 4 && W == 64)
            CUDA_TRY(launch_pdl(step_tail_kernel<4, 64, true>, grid, dim3(256), 0, st, ta));
        else
            return fail(DDB_ERR_INVALID, "sample shape [%d,%d,%d] unsupported by the guided step tail", C, H, W);
    } else if (C == 3 && W == 64)
        CUDA_TRY(launch_pdl(step_tail_kernel<3, 64>, grid, dim3(256), 0, st, ta));
    else if (C == 3 && W == 32)
        CUDA_TRY(launch_pdl(step_tail_kernel<3, 32>, grid, dim3(256), 0, st, ta));
    else if (C == 4 && W == 32)
        CUDA_TRY(launch_pdl(step_tail_kernel<4, 32>, grid, dim3(256), 0, st, ta));
    else if (C == 4 && W == 64)
        CUDA_TRY(launch_pdl(step_tail_kernel<4, 64>, grid, dim3(256), 0, st, ta));
    else
        return fail(DDB_ERR_INVALID, "sample shape [%d,%d,%d] unsupported by the fused step tail (C in {3,4}, size in "
                                     "{32,64}: every reference config)", C, H, W);
    LAUNCH_CHECK();
    return DDB_OK;
}

static int forward_impl(ddb_model* m, const float* x, const float* t, const int64_t* y, int B, float* eps, bool ee,
                        cudaStream_t st, const EeCompact* cp = nullptr, const StepFuse* fuse = nullptr) {
    const ddb_uvit_config& c = m->cfg;
    if (B < 1 || B > c.max_batch) return fail(DDB_ERR_INVALID, "batch %d outside [1, max_batch=%d]", B, c.max_batch);
    if (m->extras == 2 && !y) return fail(DDB_ERR_INVALID, "class-conditional model needs y (models/uvit.py:361)");
    if (ee && !c.early_exit) return fail(DDB_ERR_INVALID, "model was not created with early_exit=1");
    if (cp && (!ee || B > 1024)) return fail(DDB_ERR_INVALID, "compaction needs an early-exit model and batch <= 1024");
    if (fuse && ((ee && !cp) || g_gemm_variant != 2 || m->Np != 256))
        return fail(DDB_ERR_INVALID, "the fused step needs the CTA-pair path (plain backbone, or early exit with compaction)");
    const int D = m->D, M = B * m->L, nsm = m->dev.num_sms, half = c.depth / 2;
    // compaction: live sample / row counts are read from device memory by every kernel after the token assembly
    int* een = cp ? m->ee_n->as<int>() : nullptr;
    float2* st2 = m->stats->as<float2>();

    // ---- token assembly
    float2* stp = m->stats_p->as<float2>();
    const bool pair = (g_gemm_variant == 2);
    if (pair && m->Np == 256) {
        // tensor-core path: gather patches (bf16 hi + lo) -> CTA-pair GEMM (+bias +pos_embed, LayerNorm partials,
        // rows scattered into the token buffer) -> time / label token rows
        ProfScope ps(PC_EMBED);
        if (!fuse) DDB_TRY(launch_patch_gather(m, x, B, st));
        GemmArgs g = m->embed_gemm;
        g.M = B * m->Np;
        g.stats_out = stp;
        DDB_TRY(launch_gemm2(g, EPI_RES, nsm, st));
        if (!fuse) DDB_TRY(launch_token_extras(m, t, nullptr, y, B, st));
    } else {
#ifndef DDB_EXPERIMENTAL
        DDB_NEEDS_EXPERIMENTAL("gemm_variant = 1 (fp32-FMA token assembly + single-CTA GEMMs)");
#else
        // fp32 FMA path (single-CTA GEMM variant); writes one (mean, M2) per row
        ProfScope ps(PC_EMBED);
        const int grid = B * (c.img_size / c.patch_size);
        float2* emb_stats = ee ? nullptr : st2;
#define DDB_EMBED(PD)                                                                                              \
    CUDA_TRY(launch_pdl(embed_tokens_kernel<PD>, dim3(grid), dim3(256), 0, st, x, t,                               \
                        reinterpret_cast<const long long*>(y), (const float*)m->pe_wt->as<float>(),                \
                        (const float*)m->pe_bias->as<float>(), (const float*)m->pos->as<float>(),                  \
                        (const float*)(m->label_emb ? m->label_emb->as<float>() : nullptr),                        \
                        m->x0->as<__nv_bfloat16>(), emb_stats, c.in_chans, c.img_size, c.img_size, c.patch_size, D, \
                        m->L, m->extras, (int)c.normalize_timesteps))
        switch (m->pd) {
            case 12: DDB_EMBED(12); break;
            case 16: DDB_EMBED(16); break;
            case 48: DDB_EMBED(48); break;
            case 64: DDB_EMBED(64); break;
            default: return fail(DDB_ERR_INVALID, "patch_dim %d unsupported (12, 16, 48 or 64)", m->pd);
        }
#undef DDB_EMBED
        LAUNCH_CHECK();
#endif
    }

    // LayerNorm statistics travel either as one (mean, M2) per row from ln_stats_kernel (kind 1) or as D/64
    // partials per row written by the producing CTA-pair GEMM's epilogue (kind 2).
    const int np_p = D / 64;
    const int eed = cp ? (int)g_ee_debug : 0;
    int kind = 0;
    // consecutive kernels walk the rows in alternating directions (GemmArgs::reverse): L2 reuse between kernels
    bool rev = false;
    int probe_layer = -1;  // >= 0: this (fc2) GEMM also writes the partial dot products of that layer's probe
    auto run_gemm = [&](GemmArgs g, int epi, int cat, bool ln_in, bool stats_out) -> int {
        g.M = M;
        if (probe_layer >= 0) {
            g.probe_w = m->pw(probe_layer);
            g.probe_out = m->probe_p->as<float>();
        }
        if (g_alt_dir && pair && epi != EPI_DECODE) {
            g.reverse = rev ? 1 : 0;
            rev = !rev;
        }
        if (cat == PC_GEMM_FC2 && (g_l2_hints & 1)) g.l2_hints |= 1;
        if (cat == PC_GEMM_FC1 && (g_l2_hints & 2)) g.l2_hints |= 2;
        if (cat == PC_GEMM_QKV && (g_l2_hints & 4)) g.l2_hints |= 2;
        if (cp && !g.m_dev) g.m_dev = een + 1;
        if (ln_in) {
            g.stats = kind == 2 ? stp : st2;
            g.nparts = kind == 2 ? np_p : 1;
        }
        g.stats_out = (pair && stats_out) ? stp : nullptr;
        ProfScope ps(cat);
        return (pair && epi != EPI_DECODE) ? launch_gemm2(g, epi, nsm, st) : launch_gemm(g, epi, nsm, st);
    };
    kind = (pair && m->Np == 256) ? 2 : (ee ? 0 : 1);  // statistics of x0 were written by the token assembly
    // attention probes: per-sample softmax pooling of the block input + the classification MLP -> score[b]
    auto attn_probe_score = [&](int i, const __nv_bfloat16* xin, const int* n_dev, float* out) -> int {
        ProfScope ps(PC_EE_OTHER);
        const size_t smem = (size_t)(m->L + D + 8) * 4;
        CUDA_TRY(launch_pdl(attn_probe_score_kernel, dim3(B), dim3(256), smem, st, xin,
                            (const float*)m->probe_p->as<float>(), np_p,
                            (const float*)(m->ap_wc->as<float>() + (size_t)i * D * D),
                            (const float*)(m->ap_bc->as<float>() + (size_t)i * D),
                            (const float*)(m->ap_w2->as<float>() + (size_t)i * D),
                            (const float*)(m->ap_b2->as<float>() + i), m->L, D, n_dev, out));
        LAUNCH_CHECK();
        return DDB_OK;
    };
    if (ee && (m->probe_kind == 2 || m->probe_kind == 3)) {
        // timestep-indexed probes: this step's depth probes -> working set (t = int(timesteps[0]), early_exit.py:269)
        ProfScope ps(PC_EE_OTHER);
        CUDA_TRY(launch_pdl(probe_select_kernel, dim3(c.depth), dim3(128), 0, st,
                            (const float*)m->probe_tab_w->as<float>(), (const float*)m->probe_tab_b->as<float>(),
                            m->probe_w->as<float>(), m->probe_b->as<float>(), (int)c.depth, D, m->probe_kind, t,
                            cp ? cp->t_dev : (const int*)nullptr));
        LAUNCH_CHECK();
    }
    // real-valued (attention) probes with a negative threshold: a sample that never triggers takes head 0
    // (eesampler.py:62-67), which is only known after the last layer -- every sample's layer-0 rows are kept
    const bool neg_real = cp && m->probe_kind == 4 && cp->threshold < 0.f;
    if (cp) {
        ProfScope ps(PC_EE_OTHER);
        const int n = std::max(B, c.depth * B);
        CUDA_TRY(launch_pdl(ee_reset_kernel, dim3((n + 255) / 256), dim3(256), 0, st, een, m->ee_slot->as<int>(), B, m->L, m->scores->as<float>(),
                                                        c.depth, neg_real ? 0 : (int)c.depth, cp->exit_idx, cp->t_dev, cp->exit_log));
        LAUNCH_CHECK();
    }
    const std::vector<ddb_model::HalfOps>* split = nullptr;
    const int rows_h0 = (B / 2) * m->L;
    if (g_mlp_split && pair && !ee && B >= 2) {
        auto it = m->mlp_split.find(B);
        if (it == m->mlp_split.end()) {
            std::vector<ddb_model::HalfOps> v(c.depth);
            for (int i = 0; i < c.depth; ++i) {
                const BlockOps& op = m->ops[i];
                for (int hlf = 0; hlf < 2; ++hlf) {
                    const int row0 = hlf ? rows_h0 : 0, rows = hlf ? M - rows_h0 : rows_h0;
                    // fc1: A = xm rows [row0, +rows), out = hidden rows [0, rows);  fc2: A = hidden rows [0, rows),
                    // residual = xm rows [row0, ..), out = xo[i] rows [row0, ..)
                    DDB_TRY(retarget_rows(v[i].fc1[hlf], op.fc1, m->xm->p, nullptr, nullptr, row0, rows));
                    GemmArgs& g1 = v[i].fc1[hlf];
                    DDB_TRY(make_tmap_bf16(&g1.tmOut, m->hbuf->p, rows, g1.N, g1.N, 128));
                    DDB_TRY(make_tmap_bf16_sw64(&g1.tmOut2, m->hbuf->p, rows, g1.N, g1.N, 128));
                    DDB_TRY(retarget_rows(v[i].fc2[hlf], op.fc2, m->hbuf->p, m->xo[i]->p, m->xm->p, row0, rows));
                    GemmArgs& g2 = v[i].fc2[hlf];
                    DDB_TRY(make_tmap_bf16(&g2.tmA0, m->hbuf->p, rows, g2.K0, g2.K0, 128));
                }
            }
            it = m->mlp_split.emplace(B, std::move(v)).first;
        }
        split = &it->second;
    }
    const __nv_bfloat16* cur = m->x0->as<__nv_bfloat16>();
    bool probe_ready = false;  // early exit: the probe partials of the current block input are already in probe_p
    int np_exit = 1;           // compaction: format of the leavers' statistics in the scratch batch
    for (int i = 0; i < c.depth; ++i) {
        const BlockOps& op = m->ops[i];
        const BlockW& bw = m->blocks[i];
        if (ee) {
            // probe i + head i look at the block input (models/early_exit.py:294-296).  Its LayerNorm statistics and the
            // probe's partial dot products were written by the fc2 epilogue that produced it; only the first layer (and the
            // single-CTA GEMM variant) needs a pass of its own over the activations.
            if (!probe_ready && !(eed & 8)) {
                DDB_TRY(launch_ln_stats(cur, M, D, cp ? een + 1 : nullptr, st2, m->pw(i),
                                        m->probe_p->as<float>(), st));
                if (kind != 2) kind = 1;  // the token assembly's partial statistics of x0 stay in force (CTA-pair path)
            }
            probe_ready = false;
        }
        const int np_cur = kind == 2 ? np_p : 1;           // format of the block input's statistics
        float2* st_cur = kind == 2 ? stp : st2;
        if (cp) {
            // leavers take head i's output and are squeezed out of every live buffer
            {
                if (neg_real && i == 0) {  // positions == samples before the first move
                    ProfScope ps(PC_EE_OTHER);
                    CUDA_TRY(cudaMemcpyAsync(m->xe->p, cur, (size_t)M * D * 2, cudaMemcpyDeviceToDevice, st));
                    CUDA_TRY(cudaMemcpyAsync(m->stats_e->p, st_cur, (size_t)M * np_cur * 8, cudaMemcpyDeviceToDevice, st));
                }
                if (m->probe_kind == 4) DDB_TRY(attn_probe_score(i, cur, een, m->ee_sc->as<float>()));
                ProfScope ps(PC_EE_OTHER);
                if (!(eed & 2))
                    CUDA_TRY(launch_pdl(ee_decide_kernel, dim3(B), dim3(128), 0, st, (const float*)m->probe_p->as<float>(),
                                        np_p, (const float*)m->pb(i), m->L, cp->threshold, i, B,
                                        (int)c.depth, een, m->ee_slot->as<int>(), m->ee_dest->as<int>(),
                                        m->ee_dest->as<int>() + c.max_batch, m->ee_exit_slot->as<int>(), m->scores->as<float>(), cp->exit_idx, cp->t_dev,
                                        cp->exit_log, cp->score_mean_log, m->ee_sc->as<float>(),
                                        m->ee_ticket->as<unsigned>(), m->probe_kind == 4 ? 1 : 0));
                LAUNCH_CHECK();
                // the batch stays dense: stayers from its end take the leavers' places (block input, pending long skips,
                // statistics); the leavers' rows and statistics go to the scratch batch at their ORIGINAL slot -- their
                // heads run once, after the last block
                if (!(eed & 1))
                    CUDA_TRY(launch_pdl(ee_move_kernel, dim3(EE_MOVE_GRID, m->ee_live_n[i] + 1), dim3(256), 0, st, m->ee_live[i],
                                        m->ee_live_n[i], m->xe->as<__nv_bfloat16>(), st_cur, m->stats_e->as<float2>(), np_cur,
                                        (const int*)een, (const int*)m->ee_dest->as<int>(),
                                        (const int*)(m->ee_dest->as<int>() + c.max_batch),
                                        (const int*)m->ee_exit_slot->as<int>(), m->L, D));
                LAUNCH_CHECK();
            }
            np_exit = np_cur;
        } else if (ee) {
            if (m->probe_kind == 4) {
                DDB_TRY(attn_probe_score(i, cur, nullptr, m->scores->as<float>() + (size_t)i * B));
            } else {
                ProfScope ps(PC_EE_OTHER);
                CUDA_TRY(launch_pdl(probe_mean_kernel, dim3(B), dim3(128), 0, st, (const float*)m->probe_p->as<float>(),
                                    np_p, (const float*)m->pb(i), m->L,
                                    m->scores->as<float>() + (size_t)i * B));
                LAUNCH_CHECK();
            }
            DDB_TRY(run_gemm(m->head_dec[i], EPI_DECODE, PC_GEMM_DECODE, true, false));
            DDB_TRY(run_conv(m, m->ee_heads[i], m->img_pre->as<float>(),
                             m->outputs->as<float>() + (size_t)i * B * m->chw, B, st));
        }
        if (bw.has_skip) {
            DDB_TRY(run_gemm(op.skip, EPI_BIAS, PC_GEMM_SKIP, false, true));
            cur = m->xs->as<__nv_bfloat16>();
            kind = pair ? 2 : 0;
        }
        if (kind == 0) {
            DDB_TRY(launch_ln_stats(cur, M, D, nullptr, st2, nullptr, nullptr, st));
            kind = 1;
        }
        DDB_TRY(run_gemm(op.qkv, EPI_LN, PC_GEMM_QKV, true, false));
        {
            ProfScope ps(PC_ATTENTION);
            AttnArgs aa = m->attn;
            aa.b_dev = een;  // live sample count (compaction) or null
            if (g_alt_dir) {
                aa.reverse = rev ? 1 : 0;
                rev = !rev;
            }
            aa.discard = g_attn_discard;  // qkv is the library's own scratch: dead once attention has read it
            DDB_TRY(launch_attention_tc(aa, B, nsm, st));
        }
        DDB_TRY(run_gemm(op.proj, EPI_RES, PC_GEMM_PROJ, false, true));
        if (pair) {
            kind = 2;
        } else {
            DDB_TRY(launch_ln_stats(m->xm->as<__nv_bfloat16>(), M, D, nullptr, st2, nullptr, nullptr, st));
            kind = 1;
        }
        if (split) {
            // fc1 -> fc2 on the first half of the samples, then on the second half THROUGH THE SAME hidden rows: a half's
            // hidden (67 MB at CelebA B = 128) stays in L2 between the two GEMMs, and the second half overwrites the
            // first half's dirty lines before they are written back -- the 135 MB hidden never travels to HBM and back.
            const ddb_model::HalfOps& ho = (*split)[i];
            for (int hlf = 0; hlf < 2; ++hlf) {
                const int row0 = hlf ? rows_h0 : 0;
                GemmArgs g1 = ho.fc1[hlf], g2 = ho.fc2[hlf];
                g1.stats = stp + (size_t)row0 * np_p, g1.nparts = np_p;
                g2.stats_out = stp + (size_t)row0 * np_p;
                if (g_alt_dir) g1.reverse = 0, g2.reverse = 1;
                {
                    ProfScope ps(PC_GEMM_FC1);
                    DDB_TRY(launch_gemm2(g1, EPI_LN_GELU, nsm, st));
                }
                {
                    ProfScope ps(PC_GEMM_FC2);
                    DDB_TRY(launch_gemm2(g2, EPI_RES, nsm, st));
                }
            }
        } else {
            DDB_TRY(run_gemm(op.fc1, EPI_LN_GELU, PC_GEMM_FC1, true, false));
            if (ee && pair && i + 1 < c.depth) probe_layer = (eed & 4) ? -1 : i + 1, probe_ready = true;
            DDB_TRY(run_gemm(op.fc2, EPI_RES, PC_GEMM_FC2, false, true));
            probe_layer = -1;
        }
        kind = pair ? 2 : 0;
        cur = m->xo[i]->as<__nv_bfloat16>();
    }
    (void)half;
    if (kind == 0) {
        DDB_TRY(launch_ln_stats(cur, M, D, nullptr, st2, nullptr, nullptr, st));
        kind = 1;
    }
    {
        GemmArgs g = m->final_dec;
        // fused early-exit step: the stayers are un-patchified at their ORIGINAL slots, next to the leavers (below)
        if (cp && fuse) g.dec_slot = m->ee_slot->as<int>();
        DDB_TRY(run_gemm(g, EPI_DECODE, PC_GEMM_DECODE, true, false));
    }
    if (fuse && !cp) return launch_step_tail(m, fuse->tail, B, st);
    if (cp && fuse) {
        // every sample that left, at whatever layer: one grouped decode into the same image buffer, then the step tail
        // with per-sample conv weights (head of layer exit_idx[b], or final_layer for the samples that never left)
        GemmArgs g = m->head_grp;
        g.grp_layer = cp->exit_idx, g.grp_B = B, g.nparts = np_exit;
        {
            ProfScope ps(PC_GEMM_DECODE);
            DDB_TRY(launch_gemm(g, EPI_DECODE, nsm, st));
        }
        return launch_step_tail(m, fuse->tail, B, st);
    }
    if (cp) {
        // the samples that never left: full-model output, written to their original slots ...
        DDB_TRY(run_conv(m, m->final_head, m->img_pre->as<float>(), eps, B, st, een, m->ee_slot->as<int>()));
        // ... and every sample that left, at whatever layer: ONE grouped decode (the head of sample b's exit layer is
        // selected through the stacked weight map) + one conv with per-sample weights
        GemmArgs g = m->head_grp;
        g.grp_layer = cp->exit_idx, g.grp_B = B, g.nparts = np_exit;
        {
            ProfScope ps(PC_GEMM_DECODE);
            DDB_TRY(launch_gemm(g, EPI_DECODE, nsm, st));
        }
        return run_conv(m, m->final_head, m->img_pre->as<float>(), eps, B, st, nullptr, nullptr, cp->exit_idx);
    } else
        DDB_TRY(run_conv(m, m->final_head, m->img_pre->as<float>(), eps, B, st));
    return DDB_OK;
}

static int ee_forward_impl(ddb_model* m, const float* x, const float* t, const int64_t* y, int B, float threshold,
                           int mode, float* eps, int32_t* exit_idx, float* scores_out, float* outputs_out,
                           const int* t_dev, int32_t* exit_log, float* score_log, cudaStream_t st) {
    if (!m->cfg.early_exit) return fail(DDB_ERR_INVALID, "model was not created with early_exit=1");
    if (mode != 0 && mode != 1) return fail(DDB_ERR_INVALID, "ee mode must be 0 (simulate) or 1 (compact)");
    const int depth = m->cfg.depth;
    if (mode == 1) {
        if (outputs_out) return fail(DDB_ERR_INVALID, "compact mode does not produce the per-layer head outputs");
        EeCompact cp{threshold, exit_idx ? exit_idx : m->exit_idx->as<int32_t>(), t_dev, exit_log, score_log};
        DDB_TRY(forward_impl(m, x, t, y, B, eps, true, st, &cp));
        if (scores_out)
            CUDA_TRY(cudaMemcpyAsync(scores_out, m->scores->p, (size_t)depth * B * 4, cudaMemcpyDeviceToDevice, st));
        return DDB_OK;
    }
    float* full = m->outputs->as<float>() + (size_t)depth * B * m->chw;
    DDB_TRY(forward_impl(m, x, t, y, B, full, true, st));
    int32_t* idx = exit_idx ? exit_idx : m->exit_idx->as<int32_t>();
    dim3 grid((unsigned)((m->chw / 4 + 255) / 256), (unsigned)B);
    ee_select_kernel<<<grid, 256, 0, st>>>(m->scores->as<float>(), m->outputs->as<float>(), depth, B, m->chw,
                                           threshold, eps, idx, t_dev, exit_log);
    LAUNCH_CHECK();
    if (scores_out)
        CUDA_TRY(cudaMemcpyAsync(scores_out, m->scores->p, (size_t)depth * B * 4, cudaMemcpyDeviceToDevice, st));
    if (outputs_out)
        CUDA_TRY(cudaMemcpyAsync(outputs_out, m->outputs->p, (size_t)(depth + 1) * B * m->chw * 4,
                                 cudaMemcpyDeviceToDevice, st));
    return DDB_OK;
}

// ------------------------------------------------------------------------------------------------ sampler
struct ddb_sampler {
    ddb_model* early = nullptr;
    ddb_model* late = nullptr;
    int switch_t = -1, B = 0, step_mode = 0, ee_mode = -1;
    float ee_threshold = 0.f;  // any value is meaningful (eesampler.py:67); early exit is switched by ee_mode >= 0
    size_t n = 0;
    unsigned long long noise_row0 = 0;  // index of this shard's first sample in the global batch (Philox keying)
    Buf coef, t_dev, t_vec, eps, x_buf, seed_dev, next_t, ticket;
    // sampler-owned staging, so that a captured step never depends on caller pointers: labels, early-exit logs
    Buf y_buf, exit_log, score_log;
    std::vector<int> next_host, next_uploaded;  // [0,1000) successor of t, [1000,2000) backbone of the successor step
    // One captured step per backbone.  The graph works on the sampler-owned x_buf / y_buf / logs and reads t and the
    // Philox key from device memory, so it is captured once and replayed for every call / seed / caller buffer.  It is
    // re-captured when the injected-noise pointer, the presence of labels or a ddb_set_option() switch changes.
    cudaGraphExec_t graph[2] = {nullptr, nullptr};
    long long graph_nodes[2] = {0, 0};
    struct Key {
        const void* z_all = nullptr;
        int has_y = 0, epoch = -1, guide = 0;
        float scale = 0.f;
        bool operator==(const Key& o) const {
            return z_all == o.z_all && has_y == o.has_y && epoch == o.epoch && guide == o.guide && scale == o.scale;
        }
    } graph_key[2];
    // classifier-free guidance (ddb_sampler_set_guidance): every forward runs on 2B rows, y_buf holds [y ; null...]
    int guide = 0;
    float cfg_scale = 0.f;
    // DPM-Solver++(2M) (step_mode 3) and SDE-DPM-Solver++(2M) (step_mode 5): the previous step's data prediction
    // [B,C,H,W], kept across runs (an order-1 row starts a new history), and the order column of the table (0: no
    // step starts at t)
    Buf d_prev;
    std::vector<float> ms_order;
    // UniPC (step_mode 4): d_prev holds D1; D2 and the corrected x of the previous step, kept across runs like d_prev
    // (a corrector-0 row starts a new history).  ms_order is the predictor order column
    Buf d_prev2, x_base;
    bool early_exit() const { return ee_mode >= 0 && early->cfg.early_exit; }
    // every step ends in step_tail_kernel, which also prepares the head of the next step (plain backbones always;
    // early exit in compaction mode on the CTA-pair path, option "ee_fuse")
    bool fused() const { return !early_exit() || (ee_mode == 1 && g_ee_fuse != 0 && g_gemm_variant == 2 && early->Np == 256); }
};

__global__ void set_t_kernel(int* t_dev, int t) { *t_dev = t; }
__global__ void set_seed_kernel(unsigned long long* p, unsigned long long seed, unsigned long long off4) {
    p[0] = seed, p[1] = off4;
}
// eesampler.py:71  error_prediction_by_timestep[t] = classifier_outputs.mean(axis=1)[:depth]
__global__ void score_mean_kernel(const float* __restrict__ scores, int depth, int B, const int* __restrict__ t_dev,
                                  float* __restrict__ out /*[1000,depth] by t*/) {
    const int i = blockIdx.x;
    float s = 0.f;
    for (int b = threadIdx.x; b < B; b += 32) s += scores[(size_t)i * B + b];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) out[(size_t)ld_state(t_dev) * depth + i] = s / (float)B;
}

static void tail_target(TailTarget& tg, const ddb_model* m) {
    tg.a_patch = m->a_patch->as<__nv_bfloat16>();
    tg.tokens = m->x0->as<__nv_bfloat16>();
    tg.stats_p = m->stats_p->as<float2>();
    tg.pos = m->pos->as<float>();
    tg.label_emb = m->label_emb ? m->label_emb->as<float>() : nullptr;
    tg.time_tab = m->time_tab ? m->time_tab->as<float>() : nullptr;
    tg.P = m->cfg.patch_size, tg.D = m->D, tg.L = m->L, tg.extras = m->extras;
    tg.normalize_t = m->cfg.normalize_timesteps, tg.num_classes = m->cfg.num_classes;
}

// One sampling step on the stream: forward + update + bookkeeping.  t comes from s->t_dev, the Philox key from
// s->seed_dev (device memory), labels from s->y_buf.
//   plain U-ViT:  embed GEMM -> blocks -> decode GEMM -> step_tail_kernel (conv + update + head of the next step)
//   early exit, compaction:  the same, with the probes / decisions / row moves between the blocks, a second (grouped)
//                 decode GEMM for the samples that left, and per-sample conv weights in the tail
//   early exit, simulate (or ee_fuse = 0):  fill_t -> EarlyExitUViT forward + selection -> ddpm_step -> next_t
static int sampler_step(ddb_sampler* s, ddb_model* m, float* x, bool has_y, const float* z_all, float* eps_save,
                        float* x_save, cudaStream_t st) {
    const int B = s->B;  // samples; a guided forward runs on 2B rows
    const int64_t* y = has_y ? s->y_buf->as<int64_t>() : nullptr;
    const bool ee_on = s->early_exit() && m->cfg.early_exit;
    if (ee_on && !s->fused()) {
        fill_t_kernel<<<(B + 127) / 128, 128, 0, st>>>(s->t_dev->as<int>(), s->t_vec->as<float>(), B);
        LAUNCH_CHECK();
        float* eps = eps_save ? eps_save : s->eps->as<float>();
        DDB_TRY(ee_forward_impl(m, x, s->t_vec->as<float>(), y, B, s->ee_threshold, s->ee_mode, eps, nullptr, nullptr,
                                nullptr, s->t_dev->as<int>(), s->exit_log->as<int32_t>(), s->score_log->as<float>(),
                                st));
        if (s->ee_mode == 0) {
            score_mean_kernel<<<m->cfg.depth, 32, 0, st>>>(m->scores->as<float>(), m->cfg.depth, B,
                                                           s->t_dev->as<int>(), s->score_log->as<float>());
            LAUNCH_CHECK();
        }
        {
            ProfScope ps(PC_DDPM);
            CUDA_TRY(launch_pdl(ddpm_step_kernel, dim3((unsigned)((s->n / 4 + 255) / 256)), dim3(256), 0, st, x,
                                (const float*)eps, z_all, s->n, s->n, (const float*)s->coef->as<float>(),
                                (const int*)s->t_dev->as<int>(), 0, s->step_mode, 0ull,
                                (const unsigned long long*)s->seed_dev->as<unsigned long long>(), x_save));
            LAUNCH_CHECK();
        }
        next_t_kernel<<<1, 32, 0, st>>>(s->t_dev->as<int>(), s->next_t->as<int>());
        LAUNCH_CHECK();
        return DDB_OK;
    }
    StepFuse f;
    memset(&f, 0, sizeof(f));
    TailArgs& ta = f.tail;
    ta.img_pre = m->img_pre->as<float>();
    ta.conv_w = m->final_head.conv_w->as<float>(), ta.conv_b = m->final_head.conv_b->as<float>();
    ta.x = x, ta.z_all = z_all, ta.coef = s->coef->as<float>();
    ta.t_dev = s->t_dev->as<int>(), ta.next_t = s->next_t->as<int>();
    ta.seed_dev = s->seed_dev->as<unsigned long long>();
    ta.y = reinterpret_cast<const long long*>(y);
    ta.eps_out = eps_save, ta.x_save = x_save;
    ta.ticket = s->ticket->as<unsigned>();
    ta.n = s->n, ta.H = m->cfg.img_size, ta.W = m->cfg.img_size, ta.mode = s->step_mode;
    tail_target(ta.tgt[0], s->early);
    tail_target(ta.tgt[1], s->late ? s->late : s->early);
    ta.guide = s->guide, ta.scale = s->cfg_scale, ta.B = B;
    ta.d_prev = s->d_prev ? s->d_prev->as<float>() : nullptr;
    ta.d_prev2 = s->d_prev2 ? s->d_prev2->as<float>() : nullptr;
    ta.x_base = s->x_base ? s->x_base->as<float>() : nullptr;
    if (s->guide) return forward_impl(m, x, nullptr, y, 2 * B, nullptr, false, st, nullptr, &f);
    if (ee_on) {
        // early exit with compaction: the same fused step; the tail picks every sample's conv weights by its exit layer
        EeCompact cp{s->ee_threshold, m->exit_idx->as<int32_t>(), s->t_dev->as<int>(), s->exit_log->as<int32_t>(),
                     s->score_log->as<float>()};
        ta.layer_idx = cp.exit_idx, ta.depth = m->cfg.depth;
        ta.grp_w = m->hg_conv_w->as<float>(), ta.grp_b = m->hg_conv_b->as<float>();
        return forward_impl(m, x, nullptr, y, B, nullptr, true, st, &cp, &f);
    }
    return forward_impl(m, x, nullptr, y, B, nullptr, false, st, nullptr, &f);
}

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

const char* ddb_version(void) {
#ifdef DDB_EXPERIMENTAL
    return "duodiff_b200 0.2.0 (sm_100a) +experimental";
#else
    return "duodiff_b200 0.2.0 (sm_100a)";
#endif
}
const char* ddb_last_error(void) { return g_err; }
int64_t ddb_launch_count(void) { return g_launches.load(); }
int ddb_set_option(const char* name, int32_t value) {
    if (!name) return fail(DDB_ERR_INVALID, "null option name");
    g_option_epoch.fetch_add(1);  // captured step graphs bake the options in: re-capture on the next run
#ifndef DDB_EXPERIMENTAL
    for (const char* ex : {"gemm_ts", "attn_x2", "gemm_bn128", "gemm_ln_cfg"})
        if (!strcmp(name, ex) && value != 0) DDB_NEEDS_EXPERIMENTAL(name);
    if (!strcmp(name, "gemm_variant") && value == 1) DDB_NEEDS_EXPERIMENTAL("gemm_variant = 1");
#endif
    if (!strcmp(name, "gemm_variant")) {
        if (value != 1 && value != 2) return fail(DDB_ERR_INVALID, "gemm_variant must be 1 or 2");
        g_gemm_variant = value;
        return DDB_OK;
    }
    if (!strcmp(name, "ee_fuse")) {
        g_ee_fuse = value != 0;
        return DDB_OK;
    }
    if (!strcmp(name, "ee_debug")) {
        g_ee_debug = value;
        return DDB_OK;
    }
    if (!strcmp(name, "gemm_debug")) {
        g_gemm_debug = value;
        return DDB_OK;
    }
    if (!strcmp(name, "gemm_ts")) {
        g_gemm_ts = value != 0;
        return DDB_OK;
    }
    if (!strcmp(name, "attn_x2")) {
        g_attn_x2 = value != 0;
        return DDB_OK;
    }
    if (!strcmp(name, "attn_direct")) {
        g_attn_direct = value != 0;
        return DDB_OK;
    }
    if (!strcmp(name, "attn_token")) {
        g_attn_token = value;  // bit 0: token; bits 1-3: bench-only experiments (attention.cuh)
        return DDB_OK;
    }
    if (!strcmp(name, "attn_discard")) {
        g_attn_discard = value != 0;
        return DDB_OK;
    }
    if (!strcmp(name, "mlp_split")) {
        g_mlp_split = value != 0;
        return DDB_OK;
    }
    if (!strcmp(name, "l2_hints")) {
        g_l2_hints = value;
        return DDB_OK;
    }
    if (!strcmp(name, "gemm_ln_cfg")) {
        g_gemm_ln_cfg = value;
        return DDB_OK;
    }
    if (!strcmp(name, "alt_dir")) {
        g_alt_dir = value != 0;
        return DDB_OK;
    }
    if (!strcmp(name, "gemm_bn128")) {
        g_gemm_bn128 = value != 0;
        return DDB_OK;
    }
    if (!strcmp(name, "pdl")) {
        g_use_pdl = value != 0;
        return DDB_OK;
    }
    if (ddb_host::ae_set_option(name, value)) return DDB_OK;
    return fail(DDB_ERR_INVALID, "unknown option '%s'", name);
}

int ddb_debug_set_ptr(const char* name, void* p) {
    if (name && !strcmp(name, "gemm_trace")) {
        g_gemm_trace = reinterpret_cast<long long*>(p);
        return DDB_OK;
    }
    if (name && !strcmp(name, "attn_trace")) {
        g_attn_trace = reinterpret_cast<long long*>(p);
        return DDB_OK;
    }
    return fail(DDB_ERR_INVALID, "unknown debug pointer '%s'", name ? name : "(null)");
}

int ddb_model_create(const ddb_uvit_config* cfg, const ddb_tensor* tensors, int32_t n_tensors, ddb_model** out) {
    if (!cfg || !tensors || !out) return fail(DDB_ERR_INVALID, "null argument");
    ddb_model* m = new ddb_model();
    int r = model_create_impl(cfg, tensors, n_tensors, m);
    if (r != DDB_OK) {
        delete m;
        *out = nullptr;
        return r;
    }
    *out = m;
    return DDB_OK;
}
void ddb_model_destroy(ddb_model* m) {
    if (m) {
        cudaDeviceSynchronize();
        delete m;
    }
}

int ddb_uvit_forward(ddb_model* m, const float* x_dev, const float* t_dev, const int64_t* y_dev, int32_t B,
                     float* eps_dev, void* stream) {
    if (!m || !x_dev || !t_dev || !eps_dev) return fail(DDB_ERR_INVALID, "null argument");
    return forward_impl(m, x_dev, t_dev, y_dev, B, eps_dev, false, (cudaStream_t)stream);
}

int ddb_profile_forward(ddb_model* m, const float* x_dev, const float* t_dev, const int64_t* y_dev, int32_t B,
                        float* eps_dev, int32_t ee, float* ms_host, int32_t* launches_host, void* stream) {
    if (!m || !x_dev || !t_dev || !eps_dev || !ms_host || !launches_host) return fail(DDB_ERR_INVALID, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    g_prof.active = true, g_prof.st = st, g_prof.used = 0;
    g_prof.cats.clear();
    int r = forward_impl(m, x_dev, t_dev, y_dev, B, eps_dev, ee != 0, st);
    g_prof.active = false;
    if (r != DDB_OK) return r;
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int i = 0; i < PC_COUNT; ++i) ms_host[i] = 0.f, launches_host[i] = 0;
    for (size_t i = 0; i < g_prof.cats.size(); ++i) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, g_prof.pool[2 * i], g_prof.pool[2 * i + 1]));
        ms_host[g_prof.cats[i]] += ms;
        launches_host[g_prof.cats[i]] += 1;
    }
    return DDB_OK;
}

int ddb_ee_forward(ddb_model* m, const float* x_dev, const float* t_dev, const int64_t* y_dev, int32_t B,
                   float threshold, int32_t mode, float* eps_dev, int32_t* exit_idx_dev, float* scores_dev,
                   float* outputs_dev, void* stream) {
    if (!m || !x_dev || !t_dev || !eps_dev) return fail(DDB_ERR_INVALID, "null argument");
    return ee_forward_impl(m, x_dev, t_dev, y_dev, B, threshold, mode, eps_dev, exit_idx_dev, scores_dev, outputs_dev,
                           nullptr, nullptr, nullptr, (cudaStream_t)stream);
}

int ddb_ddpm_step(float* x_dev, const float* model_out_dev, const float* z_dev, const float* coef_dev, int32_t t,
                  int32_t mode, uint64_t seed, int64_t n, void* stream) {
    if (!x_dev || !model_out_dev || !coef_dev) return fail(DDB_ERR_INVALID, "null argument");
    if (t < 0 || t > 999 || n <= 0 || n % 4) return fail(DDB_ERR_INVALID, "bad t=%d or n=%lld", t, (long long)n);
    if (mode == 3)
        return fail(DDB_ERR_INVALID, "mode 3 (DPM-Solver++) needs the previous step's data prediction: run it "
                                     "through a sampler");
    if (mode == 4)
        return fail(DDB_ERR_INVALID, "mode 4 (UniPC) needs the previous steps' data predictions: run it through a "
                                     "sampler");
    if (mode == 5)
        return fail(DDB_ERR_INVALID, "mode 5 (SDE-DPM-Solver++) needs the previous step's data prediction: run it "
                                     "through a sampler");
    // z_dev is this step's tensor: stride 0 makes z_all + t*stride land on it
    ddpm_step_kernel<<<(unsigned)((n / 4 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        x_dev, model_out_dev, z_dev, (size_t)n, (size_t)0, coef_dev, nullptr, t, mode, seed, nullptr, nullptr);
    LAUNCH_CHECK();
    return DDB_OK;
}

int ddb_sampler_create(ddb_model* early, ddb_model* late, int32_t switch_t, int32_t B, const float* coef_host,
                       int32_t step_mode, float ee_threshold, int32_t ee_mode, ddb_sampler** out) {
    if (!early || !coef_host || !out) return fail(DDB_ERR_INVALID, "null argument");
    if (B < 1 || B > early->cfg.max_batch || (late && B > late->cfg.max_batch))
        return fail(DDB_ERR_INVALID, "batch %d exceeds a model's max_batch", B);
    if (late && (late->cfg.in_chans != early->cfg.in_chans || late->cfg.img_size != early->cfg.img_size))
        return fail(DDB_ERR_SHAPE, "early/late models disagree on the sample shape [C,H,W]");
    if (ee_mode < -1 || ee_mode > 1) return fail(DDB_ERR_INVALID, "ee_mode must be -1 (off), 0 (simulate) or 1 (compact)");
    if (ee_mode >= 0 && !early->cfg.early_exit)
        return fail(DDB_ERR_INVALID, "early exit requested but the model was not created with early_exit=1");
    if (step_mode < 0 || step_mode > 5) return fail(DDB_ERR_INVALID, "step_mode must be 0, 1, 2, 3, 4 or 5");
    if (step_mode == 3 && ee_mode >= 0)
        return fail(DDB_ERR_INVALID, "step_mode 3 (DPM-Solver++) is not supported with early exit");
    if (step_mode == 4 && ee_mode >= 0)
        return fail(DDB_ERR_INVALID, "step_mode 4 (UniPC) is not supported with early exit");
    if (step_mode == 5 && ee_mode >= 0)
        return fail(DDB_ERR_INVALID, "step_mode 5 (SDE-DPM-Solver++) is not supported with early exit");
    std::unique_ptr<ddb_sampler> s(new ddb_sampler());
    s->early = early, s->late = late, s->switch_t = switch_t, s->B = B, s->step_mode = step_mode;
    s->ee_threshold = ee_threshold, s->ee_mode = ee_mode;
    s->n = (size_t)B * early->chw;
    const int row = step_mode == 4 ? 12 : step_mode >= 3 ? 8 : 4;  // floats per timestep of the coefficient table
    DDB_TRY(new_buf(s->coef, (size_t)1000 * row * 4));
    CUDA_TRY(cudaMemcpy(s->coef->p, coef_host, (size_t)1000 * row * 4, cudaMemcpyHostToDevice));
    if (step_mode >= 3) {
        DDB_TRY(new_buf(s->d_prev, s->n * 4));
        s->ms_order.resize(1000);
        const int col = step_mode == 4 ? 10 : 6;  // the (predictor) order column
        for (int t = 0; t < 1000; ++t) s->ms_order[t] = coef_host[t * row + col];
    }
    if (step_mode == 4) {
        DDB_TRY(new_buf(s->d_prev2, s->n * 4));
        DDB_TRY(new_buf(s->x_base, s->n * 4));
    }
    DDB_TRY(new_buf(s->t_dev, 4));
    DDB_TRY(new_buf(s->t_vec, (size_t)B * 4));
    DDB_TRY(new_buf(s->eps, s->n * 4));
    DDB_TRY(new_buf(s->x_buf, s->n * 4));
    DDB_TRY(new_buf(s->seed_dev, 16));
    DDB_TRY(new_buf(s->next_t, 2000 * 4));
    DDB_TRY(new_buf(s->ticket, 4));
    DDB_TRY(new_buf(s->y_buf, (size_t)B * 8));
    if (ee_mode >= 0) {
        DDB_TRY(new_buf(s->exit_log, (size_t)1000 * B * 4));
        DDB_TRY(new_buf(s->score_log, (size_t)1000 * early->cfg.depth * 4));
    }
    s->next_host.assign(2000, 0);
    *out = s.release();
    return DDB_OK;
}
void ddb_sampler_destroy(ddb_sampler* s) {
    if (!s) return;
    cudaDeviceSynchronize();
    for (int i = 0; i < 2; ++i)
        if (s->graph[i]) cudaGraphExecDestroy(s->graph[i]);
    delete s;
}
int ddb_sampler_set_guidance(ddb_sampler* s, float scale, int64_t null_label) {
    if (!s) return fail(DDB_ERR_INVALID, "null argument");
    if (!std::isfinite(scale)) return fail(DDB_ERR_INVALID, "guidance scale %g is not finite", (double)scale);
    if (s->ee_mode >= 0)
        return fail(DDB_ERR_INVALID, "guidance is not supported with early exit (the conditional and unconditional "
                                     "rows would leave at different layers)");
    for (const ddb_model* m : {s->early, s->late}) {
        if (!m) continue;
        if (m->cfg.num_classes <= 0) return fail(DDB_ERR_INVALID, "guidance needs class-conditional models");
        if (null_label < 0 || null_label >= m->cfg.num_classes)
            return fail(DDB_ERR_INVALID, "null label %lld outside [0, %d)", (long long)null_label, m->cfg.num_classes);
        if (m->cfg.max_batch < 2 * s->B)
            return fail(DDB_ERR_INVALID, "guidance runs the forward on 2B = %d rows but a model has max_batch = %d",
                        2 * s->B, m->cfg.max_batch);
    }
    // captured steps bake in the label buffer and the scale: they are captured again on the next run
    CUDA_TRY(cudaDeviceSynchronize());
    for (int i = 0; i < 2; ++i)
        if (s->graph[i]) cudaGraphExecDestroy(s->graph[i]), s->graph[i] = nullptr;
    // labels [y ; null x B]: the run copies y into the first half, the null half is written once here
    Buf y2;
    DDB_TRY(new_buf(y2, (size_t)2 * s->B * 8));
    std::vector<int64_t> nulls((size_t)s->B, null_label);
    CUDA_TRY(cudaMemcpy(y2->as<int64_t>() + s->B, nulls.data(), (size_t)s->B * 8, cudaMemcpyHostToDevice));
    s->y_buf = std::move(y2);
    s->guide = 1, s->cfg_scale = scale;
    return DDB_OK;
}
int ddb_sampler_set_noise_offset(ddb_sampler* s, uint64_t first_row) {
    if (!s) return fail(DDB_ERR_INVALID, "null argument");
    s->noise_row0 = first_row;
    return DDB_OK;
}

// Runs the model at the timesteps t_list[0..n) (late[k] != 0: on the late backbone) with the sampler's update rule.
// The early-exit log rows of the visited timesteps are copied to the caller's buffers afterwards (when given).
static int sampler_run_impl(ddb_sampler* s, float* x_dev, const int64_t* y_dev, const float* z_all_dev, uint64_t seed,
                            const int32_t* t_list, const uint8_t* late, int n, float* eps_trace_dev, float* x_trace_dev,
                            int32_t* exit_idx_trace_dev, float* score_mean_trace_dev, int32_t use_graph,
                            cudaStream_t st) {
    if (n <= 0) return DDB_OK;
    for (int k = 0; k < n; ++k) {
        if (t_list[k] < 0 || t_list[k] > 999) return fail(DDB_ERR_INVALID, "timestep %d outside [0, 999]", t_list[k]);
        if (late[k] && !s->late) return fail(DDB_ERR_INVALID, "step %d asks for the late model but none was given", k);
        if (s->step_mode == 3 && s->ms_order[t_list[k]] == 0.f)
            return fail(DDB_ERR_INVALID, "timestep %d is not a step of the DPM-Solver++ grid (order 0 in the table)",
                        t_list[k]);
        if (s->step_mode == 4 && s->ms_order[t_list[k]] == 0.f)
            return fail(DDB_ERR_INVALID, "timestep %d is not a step of the UniPC grid (predictor order 0 in the table)",
                        t_list[k]);
        if (s->step_mode == 5 && s->ms_order[t_list[k]] == 0.f)
            return fail(DDB_ERR_INVALID,
                        "timestep %d is not a step of the SDE-DPM-Solver++ grid (order 0 in the table)", t_list[k]);
    }
    if (use_graph && (eps_trace_dev || x_trace_dev))
        return fail(DDB_ERR_INVALID, "per-step eps/x traces need use_graph=0");
    if ((exit_idx_trace_dev || score_mean_trace_dev) && !s->early_exit())
        return fail(DDB_ERR_INVALID, "early-exit logs requested from a sampler without early exit");
    const bool has_y = y_dev != nullptr;
    if (!has_y && ((s->early->extras == 2) || (s->late && s->late->extras == 2)))
        return fail(DDB_ERR_INVALID, "class-conditional model needs y (models/uvit.py:361)");
    // the timestep sequence as device-side tables, so that a captured step needs no host argument: the successor of
    // every t and the backbone the successor step runs on (the tail of a step prepares the head of the next one)
    for (int k = 0; k < n; ++k) {
        s->next_host[t_list[k]] = (k + 1 < n) ? t_list[k + 1] : t_list[k];
        s->next_host[1000 + t_list[k]] = (k + 1 < n) ? (late[k + 1] ? 1 : 0) : (late[k] ? 1 : 0);
    }
    if (s->next_host != s->next_uploaded) {  // unchanged for repeated runs of the same schedule: no host sync
        CUDA_TRY(cudaMemcpyAsync(s->next_t->p, s->next_host.data(), 2000 * 4, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaStreamSynchronize(st));  // the staging vector is pageable host memory owned by the handle
        s->next_uploaded = s->next_host;
    }
    set_t_kernel<<<1, 1, 0, st>>>(s->t_dev->as<int>(), t_list[0]);
    LAUNCH_CHECK();
    set_seed_kernel<<<1, 1, 0, st>>>(s->seed_dev->as<unsigned long long>(), seed,
                                     (unsigned long long)(s->noise_row0 * (s->early->chw / 4)));
    LAUNCH_CHECK();
    if (has_y) CUDA_TRY(cudaMemcpyAsync(s->y_buf->p, y_dev, (size_t)s->B * 8, cudaMemcpyDeviceToDevice, st));
    // graph replay works on the sampler-owned copy of x; eager steps work in place
    float* xw = x_dev;
    if (use_graph) {
        xw = s->x_buf->as<float>();
        CUDA_TRY(cudaMemcpyAsync(xw, x_dev, s->n * 4, cudaMemcpyDeviceToDevice, st));
    }
    if (s->fused()) {
        // head of the first step (every later step's head is written by its predecessor's tail kernel); guided: x in
        // both halves of the patch matrix, token rows for [y ; null]
        ddb_model* m0 = late[0] ? s->late : s->early;
        DDB_TRY(launch_patch_gather(m0, xw, s->B, st));
        if (s->guide) DDB_TRY(launch_patch_gather(m0, xw, s->B, st, s->B));
        DDB_TRY(launch_token_extras(m0, nullptr, s->t_dev->as<int>(), has_y ? s->y_buf->as<int64_t>() : nullptr,
                                    s->guide ? 2 * s->B : s->B, st));
    }
    if (!use_graph) {
        for (int k = 0; k < n; ++k) {
            ddb_model* m = late[k] ? s->late : s->early;
            DDB_TRY(sampler_step(s, m, xw, has_y, z_all_dev, eps_trace_dev ? eps_trace_dev + (size_t)k * s->n : nullptr,
                                 x_trace_dev ? x_trace_dev + (size_t)k * s->n : nullptr, st));
        }
    } else {
        // ---- one captured step per backbone
        ddb_sampler::Key key;
        key.z_all = z_all_dev, key.has_y = has_y ? 1 : 0, key.epoch = g_option_epoch.load();
        key.guide = s->guide, key.scale = s->cfg_scale;
        for (int which = 0; which < 2; ++which) {
            ddb_model* m = which == 0 ? s->early : s->late;
            if (!m) continue;
            if (s->graph[which] && !(key == s->graph_key[which])) {
                cudaGraphExecDestroy(s->graph[which]);
                s->graph[which] = nullptr;
            }
            if (s->graph[which]) continue;
            cudaStream_t cs;
            CUDA_TRY(cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking));
            cudaGraph_t g = nullptr;
            CUDA_TRY(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
            const long long before = g_launches.load();
            int r = sampler_step(s, m, xw, has_y, z_all_dev, nullptr, nullptr, cs);
            g_launches.store(before);  // captured, not executed: replays are counted below
            cudaError_t e = cudaStreamEndCapture(cs, &g);
            if (r != DDB_OK) {
                if (g) cudaGraphDestroy(g);
                cudaStreamDestroy(cs);
                return r;
            }
            if (e != cudaSuccess) {
                cudaStreamDestroy(cs);
                return fail(DDB_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(e));
            }
            size_t n_nodes = 0;
            cudaGraphGetNodes(g, nullptr, &n_nodes);
            s->graph_nodes[which] = (long long)n_nodes;
            e = cudaGraphInstantiate(&s->graph[which], g, 0);
            cudaGraphDestroy(g);
            cudaStreamDestroy(cs);
            if (e != cudaSuccess) return fail(DDB_ERR_CUDA, "graph instantiate failed: %s", cudaGetErrorString(e));
            s->graph_key[which] = key;
        }
        for (int k = 0; k < n; ++k) {
            const int which = late[k] ? 1 : 0;
            CUDA_TRY(cudaGraphLaunch(s->graph[which], st));
            g_launches.fetch_add(s->graph_nodes[which], std::memory_order_relaxed);
        }
        CUDA_TRY(cudaMemcpyAsync(x_dev, xw, s->n * 4, cudaMemcpyDeviceToDevice, st));
    }
    // early-exit logs: the rows of the timesteps this call visited, from the sampler-owned buffers; a run of
    // consecutive timesteps (t, t-1, ...) is one copy, so a DDPM range is a single copy per log
    if (exit_idx_trace_dev || score_mean_trace_dev) {
        const int depth = s->early->cfg.depth;
        for (int k = 0; k < n;) {
            int j = k;
            while (j + 1 < n && t_list[j + 1] == t_list[j] - 1) ++j;
            const size_t lo = (size_t)t_list[j], rows = (size_t)(j - k + 1);
            if (exit_idx_trace_dev)
                CUDA_TRY(cudaMemcpyAsync(exit_idx_trace_dev + lo * s->B, s->exit_log->as<int32_t>() + lo * s->B,
                                         rows * s->B * 4, cudaMemcpyDeviceToDevice, st));
            if (score_mean_trace_dev)
                CUDA_TRY(cudaMemcpyAsync(score_mean_trace_dev + lo * depth, s->score_log->as<float>() + lo * depth,
                                         rows * depth * 4, cudaMemcpyDeviceToDevice, st));
            k = j + 1;
        }
    }
    return DDB_OK;
}

int ddb_sampler_run(ddb_sampler* s, float* x_dev, const int64_t* y_dev, const float* z_all_dev, uint64_t seed,
                    int32_t t_first, int32_t t_last, float* eps_trace_dev, float* x_trace_dev,
                    int32_t* exit_idx_trace_dev, float* score_mean_trace_dev, int32_t use_graph, void* stream) {
    if (!s || !x_dev) return fail(DDB_ERR_INVALID, "null argument");
    if (t_first > 999 || t_last < 0 || t_last > t_first) return fail(DDB_ERR_INVALID, "bad step range");
    if (s->step_mode == 3)
        return fail(DDB_ERR_INVALID, "DPM-Solver++ (step_mode 3) runs over its grid only: use ddb_sampler_run_list");
    if (s->step_mode == 4)
        return fail(DDB_ERR_INVALID, "UniPC (step_mode 4) runs over its grid only: use ddb_sampler_run_list");
    if (s->step_mode == 5)
        return fail(DDB_ERR_INVALID,
                    "SDE-DPM-Solver++ (step_mode 5) runs over its grid only: use ddb_sampler_run_list");
    std::vector<int32_t> ts;
    std::vector<uint8_t> late;
    for (int t = t_first; t >= t_last; --t) {
        ts.push_back(t);
        late.push_back((s->late && t < s->switch_t) ? 1 : 0);  // sampler.py:135-136
    }
    return sampler_run_impl(s, x_dev, y_dev, z_all_dev, seed, ts.data(), late.data(), (int)ts.size(), eps_trace_dev,
                            x_trace_dev, exit_idx_trace_dev, score_mean_trace_dev, use_graph, (cudaStream_t)stream);
}

int ddb_sampler_run_list(ddb_sampler* s, float* x_dev, const int64_t* y_dev, const float* z_all_dev, uint64_t seed,
                         const int32_t* t_list_host, const uint8_t* late_host, int32_t n_steps, float* eps_trace_dev,
                         float* x_trace_dev, int32_t use_graph, void* stream) {
    if (!s || !x_dev || !t_list_host || !late_host) return fail(DDB_ERR_INVALID, "null argument");
    return sampler_run_impl(s, x_dev, y_dev, z_all_dev, seed, t_list_host, late_host, n_steps, eps_trace_dev,
                            x_trace_dev, nullptr, nullptr, use_graph, (cudaStream_t)stream);
}

int ddb_sampler_run_list_logs(ddb_sampler* s, float* x_dev, const int64_t* y_dev, const float* z_all_dev,
                              uint64_t seed, const int32_t* t_list_host, const uint8_t* late_host, int32_t n_steps,
                              float* eps_trace_dev, float* x_trace_dev, int32_t* exit_idx_trace_dev,
                              float* score_mean_trace_dev, int32_t use_graph, void* stream) {
    if (!s || !x_dev || !t_list_host || !late_host) return fail(DDB_ERR_INVALID, "null argument");
    return sampler_run_impl(s, x_dev, y_dev, z_all_dev, seed, t_list_host, late_host, n_steps, eps_trace_dev,
                            x_trace_dev, exit_idx_trace_dev, score_mean_trace_dev, use_graph, (cudaStream_t)stream);
}

int ddb_sampler_profile_step(ddb_sampler* s, float* x_dev, const int64_t* y_dev, int32_t t, int32_t late,
                             float* ms_host, int32_t* launches_host, void* stream) {
    if (!s || !x_dev || !ms_host || !launches_host) return fail(DDB_ERR_INVALID, "null argument");
    cudaStream_t st = (cudaStream_t)stream;
    const int32_t tl[1] = {t};
    const uint8_t lf[1] = {(uint8_t)(late ? 1 : 0)};
    g_prof.active = true, g_prof.st = st, g_prof.used = 0;
    g_prof.cats.clear();
    int r = sampler_run_impl(s, x_dev, y_dev, nullptr, 0, tl, lf, 1, nullptr, nullptr, nullptr, nullptr, 0, st);
    g_prof.active = false;
    if (r != DDB_OK) return r;
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int i = 0; i < PC_COUNT; ++i) ms_host[i] = 0.f, launches_host[i] = 0;
    for (size_t i = 0; i < g_prof.cats.size(); ++i) {
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, g_prof.pool[2 * i], g_prof.pool[2 * i + 1]));
        ms_host[g_prof.cats[i]] += ms;
        launches_host[g_prof.cats[i]] += 1;
    }
    return DDB_OK;
}

int ddb_finalize_nhwc(const float* x_dev, float* out_dev, int32_t B, int32_t C, int32_t H, int32_t W, void* stream) {
    if (!x_dev || !out_dev) return fail(DDB_ERR_INVALID, "null argument");
    const size_t n = (size_t)B * C * H * W;
    finalize_nhwc_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x_dev, out_dev, B, C, H, W);
    LAUNCH_CHECK();
    return DDB_OK;
}

// ---- single-operator entry points
int ddb_op_gemm(const void* a0_dev, const void* a1_dev, const void* w_dev, const float* bias_dev,
                const float* colsum_dev, const float* stats_dev, int32_t nparts, int32_t ln_dim,
                const void* residual_dev, void* out_dev, float* stats_out_dev, int32_t M, int32_t N, int32_t K0,
                int32_t K1, int32_t epi, int32_t variant, void* stream) {
    if (!a0_dev || !w_dev || !out_dev) return fail(DDB_ERR_INVALID, "null argument");
    if (variant == 0) variant = g_gemm_variant;
    if (variant != 1 && variant != 2) return fail(DDB_ERR_INVALID, "variant must be 0, 1 or 2");
#ifndef DDB_EXPERIMENTAL
    if (variant == 1) DDB_NEEDS_EXPERIMENTAL("the single-CTA GEMM for the block linears");
#endif
    if (stats_out_dev && (variant != 2 || (epi != EPI_BIAS && epi != EPI_RES)))
        return fail(DDB_ERR_INVALID, "stats_out needs the CTA-pair kernel with a bias or residual epilogue");
    if (epi < 0 || epi > EPI_RES) return fail(DDB_ERR_INVALID, "epi must be 0..3");
    if (N % 256 || K0 % 64 || K1 % 64 || M < 1) return fail(DDB_ERR_INVALID, "need N%%256==0, K%%64==0, M>=1");
    if ((epi == EPI_LN || epi == EPI_LN_GELU) && (!colsum_dev || !stats_dev))
        return fail(DDB_ERR_INVALID, "LN epilogue needs colsum and stats");
    if (epi == EPI_RES && !residual_dev) return fail(DDB_ERR_INVALID, "residual epilogue needs residual");
    DeviceInfo di;
    DDB_TRY(device_info(di));
    GemmArgs g;
    memset(&g, 0, sizeof(g));
    g.M = M, g.N = N, g.K0 = K0, g.K1 = K1;
    g.bias = bias_dev, g.colsum = colsum_dev, g.stats = reinterpret_cast<const float2*>(stats_dev);
    g.nparts = nparts > 0 ? nparts : 1, g.ln_dim = ln_dim, g.ln_eps = 1e-5f;
    DDB_TRY(make_tmap_bf16(&g.tmA0, a0_dev, M, K0, K0, 128));
    if (K1 > 0) DDB_TRY(make_tmap_bf16(&g.tmA1, a1_dev, M, K1, K1, 128));
    DDB_TRY(make_tmap_bf16(&g.tmB, w_dev, N, K0 + K1, K0 + K1, 256));
    DDB_TRY(make_tmap_bf16(&g.tmB2, w_dev, N, K0 + K1, K0 + K1, 128));
    DDB_TRY(make_tmap_bf16(&g.tmB3, w_dev, N, K0 + K1, K0 + K1, 64));
    DDB_TRY(make_tmap_bf16(&g.tmOut, out_dev, M, N, N, 128));
    if (residual_dev) DDB_TRY(make_tmap_bf16(&g.tmRes, residual_dev, M, N, N, 128));
    DDB_TRY(make_tmap_bf16_sw64(&g.tmOut2, out_dev, M, N, N, 128));
    if (residual_dev) DDB_TRY(make_tmap_bf16_sw64(&g.tmRes2, residual_dev, M, N, N, 128));
    g.stats_out = reinterpret_cast<float2*>(stats_out_dev);
    return variant == 2 ? launch_gemm2(g, epi, di.num_sms, (cudaStream_t)stream)
                        : launch_gemm(g, epi, di.num_sms, (cudaStream_t)stream);
}

int ddb_op_attention(const void* qkv_dev, void* out_dev, int32_t B, int32_t L, int32_t H, int32_t variant,
                     void* stream) {
    if (!qkv_dev || !out_dev) return fail(DDB_ERR_INVALID, "null argument");
    DeviceInfo di;
    DDB_TRY(device_info(di));
    const bool tc_ok = (L == 257 || L == 258);
    if ((variant == 2 || variant == 3) && !tc_ok) return fail(DDB_ERR_INVALID, "tcgen05 attention needs L = 256 + {1,2}");
    if (variant == 2 || variant == 3 || (variant == 0 && tc_ok)) {
        AttnArgs a;
        DDB_TRY(plan_attention(a, reinterpret_cast<const __nv_bfloat16*>(qkv_dev),
                               reinterpret_cast<__nv_bfloat16*>(out_dev), B, L, H));
        return launch_attention_tc(a, B, di.num_sms, (cudaStream_t)stream, variant == 0 ? -1 : (variant == 3));
    }
    return launch_attention(reinterpret_cast<const __nv_bfloat16*>(qkv_dev),
                            reinterpret_cast<__nv_bfloat16*>(out_dev), B, L, H, (cudaStream_t)stream);
}

int ddb_op_ln_stats(const void* x_dev, int32_t M, int32_t D, float* stats_dev, void* stream) {
    if (!x_dev || !stats_dev) return fail(DDB_ERR_INVALID, "null argument");
    return launch_ln_stats(reinterpret_cast<const __nv_bfloat16*>(x_dev), M, D, nullptr,
                           reinterpret_cast<float2*>(stats_dev), nullptr, nullptr, (cudaStream_t)stream);
}

int ddb_op_pack_linear(const float* w_dev, const float* bias_dev, const float* gamma_dev, const float* beta_dev,
                       int32_t N, int32_t K, void* wp_dev, float* colsum_dev, float* bias_out_dev, void* stream) {
    if (!w_dev || !wp_dev) return fail(DDB_ERR_INVALID, "null argument");
    pack_linear_kernel<<<N, 256, 0, (cudaStream_t)stream>>>(w_dev, bias_dev, gamma_dev, beta_dev, N, K,
                                                            reinterpret_cast<__nv_bfloat16*>(wp_dev), colsum_dev,
                                                            bias_out_dev);
    LAUNCH_CHECK();
    return DDB_OK;
}

}  // extern "C"
