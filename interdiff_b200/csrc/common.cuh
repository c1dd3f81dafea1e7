// Shared internals of libinterdiff_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <cmath>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "../../include/interdiff_b200.h"

#define IDB_OK 0
#define IDB_ERR_CUDA 1
#define IDB_ERR_ARG 2
#define IDB_ERR_STATE 3

struct DevTensor {
    float* p = nullptr;
    std::vector<int64_t> shape;
    size_t numel() const { size_t n = 1; for (auto s : shape) n *= (size_t)s; return n; }
};

struct StepParams {      // one row per diffusion step index i (device table)
    long long t;         // timestep passed to the model (timestep_map[i])
    float c1, c2;        // posterior_mean_coef1/2[i]
    float sigma_nz;      // (i != 0) * exp(0.5 * posterior_log_variance_clipped[i])
    float pad;
};

struct DenoiserLayer {
    bool qan = false;
    // standard self-attention
    float *w_qkv = nullptr, *b_qkv = nullptr, *w_o = nullptr, *b_o = nullptr;
    // folded self-attention: [Wq; Wk; (Wo_h Wv_h) for h] (1536 x 256), bias [bq; bk; 0], bo' = bo + sum_h Wo_h bv_h
    float *w_qkvf = nullptr, *b_qkvf = nullptr, *bo_f = nullptr;
    // (big, small) splits of the GEMM weights for the tensor-core path
    __half* qt_pack = nullptr;                                     // folded queries [2 (hi, lo)][3N][D + 8]: the kernels' staged layout
    __half* mem_pack = nullptr;                                    // bound: per sample keys hi | lo, value words hi | lo, kc (mem_block_bytes)
    __half *w_qkvf_b = nullptr, *w_qkvf_s = nullptr, *w1_b = nullptr, *w1_s = nullptr,
           *w2_b = nullptr, *w2_s = nullptr;
    // QaN
    float *qt = nullptr, *wk = nullptr;  // qt: [3*N][D] folded queries
    // cross attention
    float *w_qc = nullptr, *b_qc = nullptr, *w_kvc = nullptr, *b_kvc = nullptr, *w_oc = nullptr, *b_oc = nullptr;
    float *w1 = nullptr, *b1 = nullptr, *w2 = nullptr, *b2 = nullptr;
    float *ln1w = nullptr, *ln1b = nullptr, *ln2w = nullptr, *ln2b = nullptr, *ln3w = nullptr, *ln3b = nullptr;
    float* kv_mem = nullptr;  // [Tm*B][2D] cross-attention K|V of the bound memory
    float* vp_mem = nullptr;  // [Tm*B][H*D] values folded with the out-projection: (V_h Wo_h^T)
    float* kp_mem = nullptr;  // [Tm*B][H*D] keys folded with the query projection: (K_h Wq_h) / sqrt(hd)
    float* kc_mem = nullptr;  // [Tm*B][H]   constant logit term (bq_h . K_h) / sqrt(hd)
    float* w_qcT = nullptr;   // [D][D] transposed cross-attention query weight (for the key fold)
};

struct Denoiser {
    idb_denoiser_config cfg{};
    bool configured = false, committed = false;
    std::map<std::string, DevTensor> raw;   // reference state_dict name -> device copy
    std::vector<DenoiserLayer> layers;
    std::vector<DenoiserLayer> enc_layers;        // conditioning encoder (empty unless its weights were loaded)
    // encoder workspace (rows m = b*Tp + t), grown on demand by idb_encode_condition
    int enc_cap = 0;
    float *e_add = nullptr, *e_h = nullptr, *e_h2 = nullptr, *e_z = nullptr, *e_qkv = nullptr;
    __half *e_xtok_b = nullptr, *e_xtok_s = nullptr, *e_h_b = nullptr, *e_h_s = nullptr, *e_h2_b = nullptr, *e_h2_s = nullptr,
           *e_ff_b = nullptr, *e_ff_s = nullptr;
    std::vector<void*> enc_owned;
    float *w_shapeT = nullptr, *b_shape = nullptr;   // skeleton: shapeEmbedding k-major [3 n_points][D] + bias (null unless loaded)
    // PointNet++ point-cloud encoder (pointnet.cu): folded weights + workspace; optional like the encoder
    bool pn_ready = false; int pn_cap = 0;
    float *pn_w1 = nullptr, *pn_w2 = nullptr, *pn_xyz1 = nullptr, *pn_feat1 = nullptr;
    std::vector<float*> owned;              // packed buffers to free
    float *w_inT = nullptr, *b_in = nullptr;      // [C][D] k-major input embedding, summed bias
    float *w_in = nullptr, *w_out = nullptr;      // nn.Linear layouts for the GEMM: [D][C], [Clin][D]
    float *w_outT = nullptr, *b_out = nullptr;    // [D][Clin] k-major output heads
    float *pe = nullptr; int pe_rows = 0;         // sinusoid table [rows][D]
    float *te_w0T = nullptr, *te_b0 = nullptr, *te_w2T = nullptr, *te_b2 = nullptr;
    float *temb_tab = nullptr;                    // [pe_rows][D]: timestep MLP of every table row + b_in
    // bound problem
    int B = 0, T = 0, M = 0, Tm = 0;
    float *cond = nullptr, *zero_pose = nullptr;
    float *temb = nullptr, *h = nullptr, *h2 = nullptr, *qkv = nullptr, *att = nullptr, *ff = nullptr, *qc = nullptr;
    float *addend = nullptr, *lin = nullptr, *z = nullptr;
    __half *w_in_b = nullptr, *w_in_s = nullptr, *w_out_b = nullptr, *w_out_s = nullptr;
    // fp16 (hi, lo) copies of the activations that feed GEMMs  (_b = hi, _s = lo)
    __half *h_b = nullptr, *h_s = nullptr, *h2_b = nullptr, *h2_s = nullptr, *ff_b = nullptr, *ff_s = nullptr, *xtok_b = nullptr,
           *xtok_s = nullptr;
    std::vector<void*> bound_h;
    int* step_cur = nullptr;      // device: diffusion step index i of the step in flight (moved by the step's last kernel)
    int* ticket = nullptr;        // device: block counter of that last kernel
    std::vector<float*> bound;              // workspaces to free on rebind
};

struct Diffusion {
    int n = 0;
    std::vector<StepParams> host;
    StepParams* tbl = nullptr;
};

struct BodyModel;     // lbs.cu
struct Projector;     // correction.cu
struct Sampler;       // sampler.cu

struct idb_handle {
    std::string err;
    int device = 0, sm_count = 148;
    long long epoch = 0;      // bumped whenever a buffer / table / launch attribute that captured graphs reference changes
    long long launches = 0;   // kernels launched through this handle (bench's gpu_launches)
    int gemm_backend = 1;     // 0 = fp32 SIMT (debug / bisect), 1 = tcgen05 split-fp16 (default)
    int pdl = 1;              // programmatic dependent launch between the kernels of a sampling step
    unsigned attr_mask = 0;   // kernels whose > 48 KB shared-memory opt-in was done on this handle's device (bit 0 GEMM, 1 MLP, 2 NN)
    double last_ms = 0.0;     // mean launch time of the last timed debug hook
    int gemm_multicast = 1;   // long wide GEMMs (SMPL-H blend): row-tile pairs share the W tile by TMA multicast (idb_debug_set_gemm_multicast)
    int nn_pruning = 1;       // cluster-pruned nearest-neighbour search for body-mesh targets (identical results)
    int fuse_attn = 1;        // standard decoder layers: self-attention + cross-attention in one launch (idb_set_fused_mlp(h, 10 / 11) = off / on)
    int fused_mlp = 2;        // feed-forward block as ONE cluster kernel (tensor backend, d_model 256, d_ff 1024); 2 = incl. the layer's final norm;
                              // 3 = a layer's attention half runs in the same kernel on sample-aligned tiles (one launch per layer):
                              // measured NOT faster (288.6 vs 282.3 us per step at B=60: programmatic dependent launch already hides the
                              // boundary) and at B=64 it needs 16 clusters where the device holds 15 (profiles/README.md) - kept as an option
    void* metrics_ws = nullptr; size_t metrics_bytes = 0;        // workspace of idb_metrics (posed object points, normals, signed distances)
    void* scratch = nullptr; size_t scratch_bytes = 0;   // on-the-fly operand splits of idb_gemm
    Denoiser den;
    Diffusion diff;
    BodyModel* body = nullptr;
    Projector* proj = nullptr;
    Sampler* sampler = nullptr;
};

int idb_fail(idb_handle* h, int code, const char* fmt, ...);

// Every C-ABI entry point runs on the handle's device whatever device is current in the calling thread
// (one handle per device; the veneer keeps one Engine per device) and restores the caller's device on exit.
struct IdbDeviceGuard {
    int prev = -1;
    explicit IdbDeviceGuard(const idb_handle* h) {
        if (!h) return;
        int cur = -1;
        if (cudaGetDevice(&cur) == cudaSuccess && cur != h->device) { prev = cur; cudaSetDevice(h->device); }
    }
    ~IdbDeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
    IdbDeviceGuard(const IdbDeviceGuard&) = delete;
    IdbDeviceGuard& operator=(const IdbDeviceGuard&) = delete;
};
#define IDB_ENTER(h) IdbDeviceGuard _idb_device_guard(h)

#define CUDA_TRY(h, expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess)                                                              \
            return idb_fail((h), IDB_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,              \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                    \
    } while (0)

#define LAUNCH_CHECK(h)                                                                     \
    do {                                                                                    \
        (h)->launches++;                                                                    \
        cudaError_t _e = cudaGetLastError();                                                \
        if (_e != cudaSuccess)                                                              \
            return idb_fail((h), IDB_ERR_CUDA, "kernel launch failed: %s (%s:%d)",          \
                            cudaGetErrorString(_e), __FILE__, __LINE__);                    \
    } while (0)

// ---------------------------------------------------------------- device helpers
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// Exact (erf) GELU, F.gelu default (model/layers.py / nn.TransformerDecoderLayer activation="gelu").
// erf(t) = 1 - 2^(-t q(t)) with a degree-7 minimax fit of q(t) = -log2(erfc(t)) / t on (0, 4] (erf(4) rounds to
// 1 in fp32), branch-free: 7 FMA + one MUFU.EX2.  Max abs error of erf 1.0e-7 (libdevice erff: 6e-8; the fit
// is in profiles/README.md), i.e. fp32-rounding level for the GELU output, at less than half the instructions
// of erff's two-sided evaluation under divergence.
__device__ __forceinline__ float erf_fast(float x) {
    const float t = fminf(fabsf(x), 4.0f);
    float p = 4.5338660129345953e-05f;
    p = fmaf(p, t, -0.0004454450972843915f);
    p = fmaf(p, t, 0.0014896064531058073f);
    p = fmaf(p, t, 0.0007736838888376951f);
    p = fmaf(p, t, -0.028252195566892624f);
    p = fmaf(p, t, 0.1484806090593338f);
    p = fmaf(p, t, 0.9184166789054871f);
    p = fmaf(p, t, 1.6279085874557495f);
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-t * p));
    return copysignf(1.0f - e, x);
}
__device__ __forceinline__ float gelu_erf(float x) {
    const float hx = 0.5f * x;
    return fmaf(hx, erf_fast(x * 0.70710678118654752440f), hx);
}
// ---- packed fp32 pairs (fma / mul / add .f32x2, sm_100): the same IEEE operations as the scalar code, two per issue slot
typedef unsigned long long f32x2_t;
__device__ __forceinline__ f32x2_t pk2(float a, float b) { f32x2_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk2(f32x2_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2_t fma2(f32x2_t a, f32x2_t b, f32x2_t c) { f32x2_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2_t mul2(f32x2_t a, f32x2_t b) { f32x2_t d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2_t add2(f32x2_t a, f32x2_t b) { f32x2_t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
// two elements of the feed-forward block's hidden layer: v = gelu_erf(fmaf(small, 2^-11, main) + bias), returned as the fp16
// (hi, lo) words of split_f16x2(v0, v1).  Operation for operation the scalar gelu_erf / erf_fast / split_f16x2 (bit-identical),
// with every fp32 multiply / add / fma issued as a packed pair: the phase is bound by the SM's instruction issue rate.
__device__ __forceinline__ void gelu_split_x2(float m0, float m1, float s0, float s1, float2 bias, uint32_t& hi_w, uint32_t& lo_w) {
    const f32x2_t x = add2(fma2(pk2(s0, s1), pk2(1.0f / 2048.0f, 1.0f / 2048.0f), pk2(m0, m1)), pk2(bias.x, bias.y));
    const f32x2_t hx = mul2(x, pk2(0.5f, 0.5f));
    const f32x2_t y = mul2(x, pk2(0.70710678118654752440f, 0.70710678118654752440f));
    float y0, y1;
    upk2(y, y0, y1);
    const float t0 = fminf(fabsf(y0), 4.0f), t1 = fminf(fabsf(y1), 4.0f);
    const f32x2_t t = pk2(t0, t1);
    f32x2_t p = pk2(4.5338660129345953e-05f, 4.5338660129345953e-05f);
    p = fma2(p, t, pk2(-0.0004454450972843915f, -0.0004454450972843915f));
    p = fma2(p, t, pk2(0.0014896064531058073f, 0.0014896064531058073f));
    p = fma2(p, t, pk2(0.0007736838888376951f, 0.0007736838888376951f));
    p = fma2(p, t, pk2(-0.028252195566892624f, -0.028252195566892624f));
    p = fma2(p, t, pk2(0.1484806090593338f, 0.1484806090593338f));
    p = fma2(p, t, pk2(0.9184166789054871f, 0.9184166789054871f));
    p = fma2(p, t, pk2(1.6279085874557495f, 1.6279085874557495f));
    float a0, a1, e0, e1;
    upk2(mul2(t, p), a0, a1);          // erf_fast evaluates (-t) * p: the sign moves into the MUFU operand
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e0) : "f"(-a0));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e1) : "f"(-a1));
    float r0, r1;
    upk2(fma2(pk2(e0, e1), pk2(-1.0f, -1.0f), pk2(1.0f, 1.0f)), r0, r1);      // 1 - e (one rounding, like the scalar subtraction)
    const f32x2_t v = fma2(hx, pk2(copysignf(r0, y0), copysignf(r1, y1)), hx);
    float v0, v1;
    upk2(v, v0, v1);
    const __half2 hh = __floats2half2_rn(v0, v1);
    const float2 f = __half22float2(hh);
    float l0, l1;
    upk2(mul2(fma2(pk2(f.x, f.y), pk2(-1.0f, -1.0f), v), pk2(2048.0f, 2048.0f)), l0, l1);      // (v - hi) * 2^11, v - hi exact
    const __half2 ll = __floats2half2_rn(l0, l1);
    hi_w = *reinterpret_cast<const uint32_t*>(&hh); lo_w = *reinterpret_cast<const uint32_t*>(&ll);
}
__device__ __forceinline__ float silu(float x) { return x / (1.0f + expf(-x)); }

// Programmatic dependent launch: every kernel of the sampling step releases its successor at once
// (pdl_trigger) and blocks (pdl_wait) before its first access to data produced by earlier kernels, so
// the successor's launch latency, barrier/TMEM setup and constant-weight prefetch overlap the
// predecessor's tail.  Both are no-ops for launches without the attribute.  Every kernel in the
// chain executes pdl_wait, which makes completion transitive along the stream.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Chain timeline probe (profiles/chain_probe.py): when idb_debug_chain_trace has installed a buffer, a mark appends
// (kind, event, grid size, block | %globaltimer) to one of 64 lanes of the buffer (lane = block & 63, so that the marks of a
// launch do not serialise on one counter): lane l = buf + l * (2 + 2 * cap) words: [0] record count, [1] capacity, then records.
// Events: 0 entry, 1 dependency wait done, 2 exit.  Off (null) in production: one constant load and a branch per mark.  One
// copy of the pointer per translation unit (CHAIN_SETTER defines the unit's installer).
static __constant__ unsigned long long* c_chain = nullptr;
__device__ __forceinline__ void chain_mark(int kind, int ev) {
    unsigned long long* p = c_chain;
    if (p) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        const unsigned long long nb = (unsigned long long)gridDim.x * gridDim.y * gridDim.z;
        const unsigned long long bid = ((unsigned long long)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        const unsigned long long cap = p[1];
        p += (bid & 63) * (2 + 2 * cap);
        const unsigned long long i = atomicAdd(p, 1ull);
        if (i < cap) {
            p[2 + 2 * i] = ((unsigned long long)kind << 56) | ((unsigned long long)ev << 52) | (nb << 26) | bid;
            p[3 + 2 * i] = t;
        }
    }
}
#define CHAIN_SETTER(name) \
    int name(unsigned long long* buf) { return cudaMemcpyToSymbol(c_chain, &buf, sizeof(buf)) == cudaSuccess ? 0 : 1; }

template <typename... KArgs, typename... Args>
inline cudaError_t idb_launch(bool pdl, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}


// GEMM front door (gemm.cu): C[M,N] = epi(A[M,K] * W[N,K]^T)   (nn.Linear layout, all row-major)
enum { EPI_BIAS = 1, EPI_GELU = 2, EPI_RES = 4, EPI_SILU = 8 };
int idb_gemm(idb_handle* h, const float* A, int lda, const float* W, int ldw, const float* bias,
             const float* res, int ldr, float* C, int ldc, int M, int N, int K, int epi, cudaStream_t st);

// Split-precision operands for the tensor-core path: x = hi + lo * 2^-11 with hi = fp16_rn(x),
// lo = fp16_rn((x - hi) * 2^11) (x - hi is exact in fp32; the scale keeps lo a normal fp16 number).
// An operand is given either as full fp32 (A / W; SIMT path, or split on the fly into scratch) or as
// an fp16 pair; an output may be requested as full fp32 and/or as a pair for the next GEMM.
struct GemmArgs {
    const float* A = nullptr; const __half* A_hi = nullptr; const __half* A_lo = nullptr; int lda = 0;
    const float* W = nullptr; const __half* W_hi = nullptr; const __half* W_lo = nullptr; int ldw = 0;
    const float* bias = nullptr; const float* res = nullptr; int ldr = 0;
    float* C = nullptr; __half* C_hi = nullptr; __half* C_lo = nullptr; int ldc = 0;
    int M = 0, N = 0, K = 0, epi = 0;
    int ksplit = 1;                                     // 2: split-K onto a C zeroed by an earlier kernel (tensor path only)
    float* zero = nullptr; int zero_ld = 0, zero_cols = 0;   // aux [M][zero_cols] matrix to clear as a side job
    int pdl = 0;   // 1: programmatic dependent launch; REQUIRES W_hi/W_lo to be complete before the previous kernel started
    int single_acc = 0;   // 1: ONE main accumulator is accurate enough for the caller whatever K is (e.g. the mm-scale pose
                          //    blend added to metre-scale vertices): allows the 256-column tiles for long reductions
};
int idb_gemm_ex(idb_handle* h, const GemmArgs& g, cudaStream_t st);
// fused feed-forward block on the tensor path (gemm_tcgen05.cu)
bool idb_mlp_tcgen05_supported(int d_model, int d_ff);
int idb_mlp_tcgen05(idb_handle* h, const __half* x_hi, const __half* x_lo, const __half* w1_hi, const __half* w1_lo, const float* b1,
                    const __half* w2_hi, const __half* w2_lo, const float* b2, const float* res, int ldr, float* Z, int ldz, int M,
                    int pdl, cudaStream_t st, const float* ln_w = nullptr, const float* ln_b = nullptr, __half* Z_hi = nullptr,
                    __half* Z_lo = nullptr);
// x[rows][cols] (row stride ld_src) -> fp16 pairs [rows][ld_dst] (columns >= cols zero-filled)
int idb_split_tensor(idb_handle* h, const float* x, int ld_src, __half* hi, __half* lo, int ld_dst, int rows, int cols, cudaStream_t st);

__device__ __forceinline__ void split_f16(float x, __half& hi, __half& lo) {
    hi = __float2half_rn(x);
    lo = __float2half_rn((x - __half2float(hi)) * 2048.0f);
}
__device__ __forceinline__ void split_f16x2(float x, float y, __half2& hi, __half2& lo) {
    hi = __floats2half2_rn(x, y);
    const float2 f = __half22float2(hi);
    lo = __floats2half2_rn((x - f.x) * 2048.0f, (y - f.y) * 2048.0f);
}
__device__ __forceinline__ float join_f16(__half hi, __half lo) { return fmaf(__half2float(lo), 1.0f / 2048.0f, __half2float(hi)); }

// allocation helpers
int idb_dev_alloc(idb_handle* h, float** p, size_t n_floats);
int idb_upload(idb_handle* h, float** p, const float* host, size_t n_floats);
