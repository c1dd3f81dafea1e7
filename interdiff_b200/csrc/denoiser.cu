// Denoiser (MDM decoder path): per-timestep transformer over (batch, frames, channels).
// Replaces reference model/diffusion_smpl.py:226-246, model/diffusion_skeleton.py:218-257,
// model/layers.py:24-26,42-43,258-264, model/sublayers.py:18-35,295-375 and the
// torch.nn.TransformerDecoderLayer instances of layers 0/7.
//
// Token layout in HBM: row m = b*T + t (batch-major; a sample's frames are adjacent rows, which
// is what the 3-tap QaN filter and the per-sample attention want), features contiguous.
// All arithmetic fp32 (see gemm.cu header for why).
#include "common.cuh"
#include "tc_mlp.cuh"

#include <cstdarg>

// ------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------
namespace {

constexpr int D = 256;    // d_model is fixed at 256 for both shipped models (checked at init)
constexpr int HD = 64;    // head dim
constexpr int SLAB = 16;  // query rows per block in the per-sample attention kernels
constexpr int LDZ = D + 4;

// Step-invariant cross-attention operands of one sample, split into fp16 (hi, lo) once per bind and stored as ONE block in
// exactly the (padded, bank-conflict-free) layout the attention kernels keep in shared memory, so that a CTA stages them with
// a single bulk copy:  keys hi [HT][KPH] | keys lo [HT][KPH] (row hj = h*Tk + j, fp16) | values hi [HT/2][VPW] | values lo
// (word i = (V[2i][n], V[2i+1][n])) | kc [HT] fp32 (constant logit term).  kp / vp rows are (j*B + b) x [H][D]; kc [Tk*B][H].
// The pad columns are never read.  grid (H*Tk, B), block D.
constexpr int KPH = D + 8;     // halfs per staged row of a pre-split "rows" operand
constexpr int VPW = D + 8;     // words per staged row of a k-pair-packed K x N operand
__host__ __device__ constexpr size_t mem_block_bytes(int HT) {
    return (size_t)2 * HT * KPH * 2 + (size_t)2 * (HT >> 1) * VPW * 4 + (size_t)((HT + 3) & ~3) * 4;
}
__global__ void k_pack_memory(const float* __restrict__ kp, const float* __restrict__ vp, const float* __restrict__ kc,
                              uint8_t* __restrict__ pack, int B, int Tk, int H) {
    const int hj = blockIdx.x, b = blockIdx.y, n = threadIdx.x, HT = H * Tk, HP = HT >> 1;
    uint8_t* blk = pack + (size_t)b * mem_block_bytes(HT);
    __half* kph = reinterpret_cast<__half*>(blk); __half* kpl = kph + (size_t)HT * KPH;
    uint32_t* vph = reinterpret_cast<uint32_t*>(kpl + (size_t)HT * KPH); uint32_t* vpl = vph + (size_t)HP * VPW;
    float* kco = reinterpret_cast<float*>(vpl + (size_t)HP * VPW);
    auto src = [&](int q) { return ((size_t)((q % Tk) * B + b) * H + q / Tk) * D + n; };
    split_f16(kp[src(hj)], kph[(size_t)hj * KPH + n], kpl[(size_t)hj * KPH + n]);
    if ((hj & 1) == 0 && (hj >> 1) < HP) {
        const float v0 = vp[src(hj)], v1 = hj + 1 < HT ? vp[src(hj + 1)] : 0.f;
        __half2 h2, l2;
        split_f16x2(v0, v1, h2, l2);
        vph[(size_t)(hj >> 1) * VPW + n] = *reinterpret_cast<uint32_t*>(&h2);
        vpl[(size_t)(hj >> 1) * VPW + n] = *reinterpret_cast<uint32_t*>(&l2);
    }
    if (n == 0) kco[hj] = kc[(size_t)((hj % Tk) * B + b) * H + hj / Tk];
}

// bind-time: scale the folded keys by 1/sqrt(hd) and compute the constant logit term
//   kc[row][h] = (bq_h . K_h[row]) / 8.   One warp per (row, head).
__global__ void k_fold_scale(float* __restrict__ kp, const float* __restrict__ kv, const float* __restrict__ bq,
                             float* __restrict__ kc, int rows, int H) {
    const int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= rows * H) return;
    const int row = w / H, hh = w % H;
    float* p = kp + (size_t)row * H * D + (size_t)hh * D;
    for (int c = lane; c < D; c += 32) p[c] *= 0.125f;
    const float* kr = kv + (size_t)row * 2 * D + hh * HD;
    float a = kr[lane] * bq[hh * HD + lane] + kr[lane + 32] * bq[hh * HD + lane + 32];
    a = warp_sum(a);
    if (lane == 0) kc[(size_t)row * H + hh] = a * 0.125f;
}

// TimestepEmbedder.forward (model/layers.py:42-43): pe[t] -> Linear -> SiLU -> Linear is a pure function
// of the integer timestep, so it is tabulated once at commit for every row of the sinusoid table:
// tab[t][:] = MLP(pe[t]) + b_in  (grid pe_rows, block 256).  The sampling step only gathers from it.
// Thread (cg = tid & 63, kg = tid >> 6) accumulates columns 4cg..4cg+3 over k in [64kg, 64kg+64):
// float4 weight loads, 1 KB contiguous per k across the 64 column groups, 16 loads in flight.
__device__ __forceinline__ float4 mlp_partial(const float* __restrict__ wT, const float* __restrict__ s_x, int cg, int kg) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* w4 = reinterpret_cast<const float4*>(wT) + cg;
#pragma unroll 16
    for (int k = kg * 64; k < kg * 64 + 64; k++) {
        const float4 w = __ldg(w4 + (size_t)k * (D / 4));
        const float x = s_x[k];
        a.x = fmaf(w.x, x, a.x); a.y = fmaf(w.y, x, a.y); a.z = fmaf(w.z, x, a.z); a.w = fmaf(w.w, x, a.w);
    }
    return a;
}
__global__ void __launch_bounds__(256)
k_temb_table(const float* __restrict__ pe, const float* __restrict__ w0T, const float* __restrict__ b0,
             const float* __restrict__ w2T, const float* __restrict__ b2, const float* __restrict__ b_in,
             float* __restrict__ tab) {
    __shared__ float s_in[D], s_h[D];
    __shared__ float4 s_part[4][64];
    const int row = blockIdx.x, n = threadIdx.x, cg = n & 63, kg = n >> 6;
    s_in[n] = pe[(size_t)row * D + n];
    __syncthreads();
    s_part[kg][cg] = mlp_partial(w0T, s_in, cg, kg);
    __syncthreads();
    {
        const float* p = reinterpret_cast<const float*>(s_part);
        s_h[n] = silu(((p[n] + p[256 + n]) + (p[512 + n] + p[768 + n])) + b0[n]);
    }
    __syncthreads();
    s_part[kg][cg] = mlp_partial(w2T, s_h, cg, kg);
    __syncthreads();
    {
        const float* p = reinterpret_cast<const float*>(s_part);
        tab[(size_t)row * D + n] = (((p[n] + p[256 + n]) + (p[512 + n] + p[768 + n])) + b2[n]) + b_in[n];
    }
}

// store two float4 (columns 4*lane.. and 128+4*lane.. of a 256-wide row) as fp16 (hi, lo) pairs
__device__ __forceinline__ void store_pairs(const float4& o0, const float4& o1, __half* __restrict__ hi, __half* __restrict__ lo, int lane) {
    __half2 h0, h1, h2, h3, l0, l1, l2, l3;
    split_f16x2(o0.x, o0.y, h0, l0); split_f16x2(o0.z, o0.w, h1, l1);
    split_f16x2(o1.x, o1.y, h2, l2); split_f16x2(o1.z, o1.w, h3, l3);
    *reinterpret_cast<uint2*>(hi + lane * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
    *reinterpret_cast<uint2*>(hi + 128 + lane * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&h2), *reinterpret_cast<uint32_t*>(&h3));
    *reinterpret_cast<uint2*>(lo + lane * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&l0), *reinterpret_cast<uint32_t*>(&l1));
    *reinterpret_cast<uint2*>(lo + 128 + lane * 4) = make_uint2(*reinterpret_cast<uint32_t*>(&l2), *reinterpret_cast<uint32_t*>(&l3));
}

// out[m,:] = LayerNorm(a[m,:]) * w + b.  warp per row, D = 256.
__global__ void k_ln(const float* __restrict__ a, const float* __restrict__ w, const float* __restrict__ bb,
                     float* __restrict__ out, __half* __restrict__ out_b, __half* __restrict__ out_s, int M) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    pdl_wait();
    if (warp >= M) return;
    const float4* pa = reinterpret_cast<const float4*>(a + (size_t)warp * D);
    float v[8];
    float4 u0 = pa[lane], u1 = pa[lane + 32];
    v[0] = u0.x; v[1] = u0.y; v[2] = u0.z; v[3] = u0.w; v[4] = u1.x; v[5] = u1.y; v[6] = u1.z; v[7] = u1.w;
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) s += v[i];
    const float mean = warp_sum(s) * (1.0f / D);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) { const float d = v[i] - mean; q = fmaf(d, d, q); }
    const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / D) + 1e-5f);
    const float4* pw = reinterpret_cast<const float4*>(w);
    const float4* pb = reinterpret_cast<const float4*>(bb);
    float4 w0 = pw[lane], w1 = pw[lane + 32], b0 = pb[lane], b1 = pb[lane + 32];
    float4 o0, o1;
    o0.x = (v[0] - mean) * rstd * w0.x + b0.x; o0.y = (v[1] - mean) * rstd * w0.y + b0.y;
    o0.z = (v[2] - mean) * rstd * w0.z + b0.z; o0.w = (v[3] - mean) * rstd * w0.w + b0.w;
    o1.x = (v[4] - mean) * rstd * w1.x + b1.x; o1.y = (v[5] - mean) * rstd * w1.y + b1.y;
    o1.z = (v[6] - mean) * rstd * w1.z + b1.z; o1.w = (v[7] - mean) * rstd * w1.w + b1.w;
    float4* po = reinterpret_cast<float4*>(out + (size_t)warp * D);
    po[lane] = o0; po[lane + 32] = o1;
    if (out_b) store_pairs(o0, o1, out_b + (size_t)warp * D, out_s + (size_t)warp * D, lane);
}

// LayerNorm of one 256-wide row held in shared memory by one warp (lane holds cols 4*lane.. and 128+4*lane..)
__device__ __forceinline__ void warp_ln_row(const float* __restrict__ zrow, const float* __restrict__ w, const float* __restrict__ bb,
                                            float* __restrict__ dst, int lane, __half* __restrict__ dst_b = nullptr,
                                            __half* __restrict__ dst_s = nullptr) {
    const float4 u0 = *reinterpret_cast<const float4*>(zrow + lane * 4), u1 = *reinterpret_cast<const float4*>(zrow + 128 + lane * 4);
    float v[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) s += v[i];
    const float mean = warp_sum(s) * (1.0f / D);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) { const float d = v[i] - mean; q = fmaf(d, d, q); }
    const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / D) + 1e-5f);
    const float4 w0 = *reinterpret_cast<const float4*>(w + lane * 4), w1 = *reinterpret_cast<const float4*>(w + 128 + lane * 4);
    const float4 b0 = *reinterpret_cast<const float4*>(bb + lane * 4), b1 = *reinterpret_cast<const float4*>(bb + 128 + lane * 4);
    float4 o0, o1;
    o0.x = (v[0] - mean) * rstd * w0.x + b0.x; o0.y = (v[1] - mean) * rstd * w0.y + b0.y;
    o0.z = (v[2] - mean) * rstd * w0.z + b0.z; o0.w = (v[3] - mean) * rstd * w0.w + b0.w;
    o1.x = (v[4] - mean) * rstd * w1.x + b1.x; o1.y = (v[5] - mean) * rstd * w1.y + b1.y;
    o1.z = (v[6] - mean) * rstd * w1.z + b1.z; o1.w = (v[7] - mean) * rstd * w1.w + b1.w;
    *reinterpret_cast<float4*>(dst + lane * 4) = o0;
    *reinterpret_cast<float4*>(dst + 128 + lane * 4) = o1;
    if (dst_b) store_pairs(o0, o1, dst_b, dst_s, lane);
}


// ---------------------------------------------------------------------------------------------
// Attention kernels.  One CTA = a slab of <= 16 rows of one sample, 512 threads (16 warps, 4 per
// scheduler): these kernels are chains of short, latency-bound phases between block barriers, so
// the win comes from more warps per phase, fewer phases, and issuing every global read up front.
// phase timeline of the fused QaN kernel (clock64 of CTA (0,0) thread 0 at the phase boundaries); read with
// idb_debug_attn_trace.  One predicated store per phase.
__device__ long long g_attn_trace[16];
#define ATRACE(slot) do { if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0) g_attn_trace[slot] = clock64(); } while (0)
constexpr int ANT = 512;   // threads per attention CTA
constexpr int ANW = 16;    // warps

// --- staging: 1-D bulk copies (TMA) of whole rows, completion counted on an mbarrier.  A CTA needs ~170 KB
// (folded queries, folded memory keys / values, parameter vectors, its input rows); as per-thread 16-byte
// cp.async that is ~11 K instructions with index arithmetic per CTA, as bulk copies ~150 instructions.
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mb_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(smem_addr(bar)), "r"(parity) : "memory");
    }
}
// dst/src 16-byte aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_addr(dst)), "l"(src), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}
constexpr uint32_t ROW_BYTES = D * sizeof(float);

// --- 16-row tensor-core fragments.  The three small products of the fused QaN / cross-attention kernel
// ([18 x 256] x [256 x 30], [16 x 256] x [256 x 40], [16 x 40] x [40 x 256]) are far too small for a
// tcgen05 tile (M = 128) but are exactly one mma.sync m16n8k16 row block.  fp32 operands are read from
// shared memory straight into fragments (row strides of 8 mod 32 floats for the float2 k-pairs, 4 mod 16
// for the K x N values, make every fragment load conflict-free), split on the fly into the same fp16
// (hi, lo * 2^11) pairs as the big GEMMs and multiplied as hi*hi (main accumulator) and lo*hi + hi*lo
// (small accumulator, folded in with 2^-11): fp32-grade, ~3e-7 over K = 256 with the 4-way k-split.
// History (profiles/README.md): the register-tiled SIMT version was bound by shared-memory wavefronts
// (4-way replays of its 128-bit operand loads); a 3xTF32 m16n8k8 version was no faster because legacy
// TF32 mma.sync issues at ~30 cycles per instruction and scheduler on this part (= the FFMA rate).
constexpr int LDX = D + 8;     // row stride of fragment-A / row-dot operands (x rows, folded queries / keys): 8 mod 32
constexpr int VLD = D + 4;     // row stride of the folded values (K x N fragments): 4 mod 16
constexpr int PLD = 72;        // row stride of the probabilities: 8 mod 32
constexpr int XLDP = 64;       // row stride of the cross-attention logit partials
constexpr int P1LD = 32;       // row stride of the QaN logit partials

__device__ __forceinline__ uint32_t h2u(const __half2& h) { return *reinterpret_cast<const uint32_t*>(&h); }
__device__ __forceinline__ void split_pair(float x, float y, uint32_t& hi, uint32_t& lo) {
    __half2 h, l;
    split_f16x2(x, y, h, l);
    hi = h2u(h); lo = h2u(l);
}
__device__ __forceinline__ void mma_f16(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// main += hi*hi ; small += lo*hi + hi*lo   (result = main + small / 2048)
__device__ __forceinline__ void mma_pairs(float (&cm)[4], float (&cs)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4],
                                          const uint32_t (&bh)[2], const uint32_t (&bl)[2]) {
    mma_f16(cs, al, bh); mma_f16(cs, ah, bl); mma_f16(cm, ah, bh);
}
// A fragment (16 x 16): rows row0 + g, row0 + g + 8 (clamped to nrows - 1), k-pairs k0 + 2c, k0 + 2c + 8
__device__ __forceinline__ void load_a_frag(const float* __restrict__ s, int ld, int row0, int nrows, int k0, int lane,
                                            uint32_t (&hi)[4], uint32_t (&lo)[4]) {
    const int g = lane >> 2, c = lane & 3;
    const float* p0 = s + min(row0 + g, nrows - 1) * ld + k0 + 2 * c;
    const float* p1 = s + min(row0 + g + 8, nrows - 1) * ld + k0 + 2 * c;
    const float2 v0 = *reinterpret_cast<const float2*>(p0), v1 = *reinterpret_cast<const float2*>(p1);
    const float2 v2 = *reinterpret_cast<const float2*>(p0 + 8), v3 = *reinterpret_cast<const float2*>(p1 + 8);
    split_pair(v0.x, v0.y, hi[0], lo[0]); split_pair(v1.x, v1.y, hi[1], lo[1]);
    split_pair(v2.x, v2.y, hi[2], lo[2]); split_pair(v3.x, v3.y, hi[3], lo[3]);
}
// B fragment (16 x 8) of "dot products against the rows of Mx": B[k][n] = Mx[n0 + n][k0 + k]   (rows clamped)
__device__ __forceinline__ void load_b_frag_rows(const float* __restrict__ s, int ld, int n0, int nrows, int k0, int lane,
                                                 uint32_t (&hi)[2], uint32_t (&lo)[2]) {
    const float* p = s + min(n0 + (lane >> 2), nrows - 1) * ld + k0 + 2 * (lane & 3);
    const float2 v0 = *reinterpret_cast<const float2*>(p), v1 = *reinterpret_cast<const float2*>(p + 8);
    split_pair(v0.x, v0.y, hi[0], lo[0]); split_pair(v1.x, v1.y, hi[1], lo[1]);
}
// B fragment (16 x 8) of a row-major K x N matrix: B[k][n] = Mx[k0 + k][n0 + n]   (rows clamped to nk - 1)
__device__ __forceinline__ void load_b_frag_cols(const float* __restrict__ s, int ld, int k0, int nk, int n0, int lane,
                                                 uint32_t (&hi)[2], uint32_t (&lo)[2]) {
    const int g = lane >> 2, c = lane & 3;
    const float* q = s + n0 + g;
    const int r = k0 + 2 * c;
    split_pair(q[min(r, nk - 1) * ld], q[min(r + 1, nk - 1) * ld], hi[0], lo[0]);
    split_pair(q[min(r + 8, nk - 1) * ld], q[min(r + 9, nk - 1) * ld], hi[1], lo[1]);
}

// Self-attention core + out-projection (folded into the values) + residual + LayerNorm.
// grid (B, ceil(T/16)), block 512.
//   q rows  : q[(b*T + r) * ldq + h*64 + d]                          (pre-projected queries)
//   keys    : k[(b*T + j) * ldk + h*64 + d], j < T
//   values' : v[(b*T + j) * ldv + h*256 + n]  = (V_h W_o,h^T)[j][n]: value vectors already
//             multiplied by the head's out-proj block
//   out[r]  = LN( res[r] + bo + sum_h sum_j softmax_j(q_h[r].k_h[j] / 8) v'_h[j] )
// Both products run on fp16-pair fragments: logits = 16 (head, 8-key tile) units of 4 k-steps, one
// per warp; values = [16 x 4T] x [4T x 256], two 8-column tiles per warp.
struct AttnArgs {
    const float* q; int ldq; const float* k; int ldk; const float* v; int ldv; const float *res, *bo, *lnw, *lnb;
    float* out; __half *out_b, *out_s; int T, H;
};
// slab (sample b, rows r0 ..) on caller-provided shared memory (attn_smem() bytes); also phase A1 of the fused standard layer
__device__ __forceinline__ void attn_body(const AttnArgs& aa, float* sm, const int b, const int r0) {
    const float* __restrict__ q = aa.q; const float* __restrict__ k = aa.k; const float* __restrict__ v = aa.v;
    const float* __restrict__ res = aa.res; const float* __restrict__ bo = aa.bo; const float* __restrict__ lnw = aa.lnw;
    const float* __restrict__ lnb = aa.lnb; float* __restrict__ out = aa.out; __half* __restrict__ out_b = aa.out_b;
    __half* __restrict__ out_s = aa.out_s;
    const int ldq = aa.ldq, ldk = aa.ldk, ldv = aa.ldv, T = aa.T, H = aa.H;
    constexpr int LDK = HD + 8;            // key-slice stride (8 mod 32)
    const int Tk = T, HT = H * Tk, HT16 = (HT + 15) & ~15, pld = ((HT16 + 23) / 32) * 32 + 8;   // pld: >= HT16, 8 mod 32
    uint64_t* bar = reinterpret_cast<uint64_t*>(sm);   // [0]: parameters, [1]: activations
    float* s_par = sm + 4;                 // bo, lnw, lnb
    float* s_q = s_par + 3 * D;            // [SLAB][LDX]   query rows
    float* s_z = s_q + SLAB * LDX;         // [SLAB][LDZ]   residual rows, then the pre-LayerNorm sums
    float* s_v = s_z + SLAB * LDZ;         // [H*Tk][VLD]   folded values
    float* s_k = s_v + (size_t)HT * VLD;   // [H*Tk][LDK]   key head slices ...
    float* s_p = s_k;                      // [SLAB][pld]   ... then (after a barrier) logits / probabilities
    const int nr = min(SLAB, T - r0), tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, c = lane & 3;
    pdl_trigger();
    if (tid == 0) {
        mb_init(bar, 1); mb_init(bar + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // barrier [0]: parameter rows + the folded value rows (120 KB, needed only by the value product: their copy overlaps the
    // logits and the softmax); barrier [1]: query / residual rows and key slices (needed at once)
    if (tid == 0) {
        mb_expect_tx(bar, (uint32_t)(3 + HT) * ROW_BYTES);
        bulk_g2s(s_par, bo, ROW_BYTES, bar); bulk_g2s(s_par + D, lnw, ROW_BYTES, bar); bulk_g2s(s_par + 2 * D, lnb, ROW_BYTES, bar);
    }
    pdl_wait();
    if (tid == 0) chain_mark(0, 1);
    if (tid == 0) mb_expect_tx(bar + 1, (uint32_t)(2 * nr + Tk) * ROW_BYTES);
    __syncwarp();
    // one copy per thread and round: query + residual rows, key head slices (256 B), folded value rows
    for (int i = tid; i < 2 * nr + 2 * HT; i += ANT) {
        if (i < nr) bulk_g2s(s_q + i * LDX, q + (size_t)(b * T + r0 + i) * ldq, ROW_BYTES, bar + 1);
        else if (i < 2 * nr) bulk_g2s(s_z + (i - nr) * LDZ, res + (size_t)(b * T + r0 + i - nr) * D, ROW_BYTES, bar + 1);
        else if (i < 2 * nr + HT) {
            const int hj = i - 2 * nr, hh = hj / Tk, j = hj - hh * Tk;
            bulk_g2s(s_k + hj * LDK, k + (size_t)(b * T + j) * ldk + hh * HD, HD * sizeof(float), bar + 1);
        } else {
            const int hj = i - 2 * nr - HT, hh = hj / Tk, j = hj - hh * Tk;
            bulk_g2s(s_v + (size_t)hj * VLD, v + (size_t)(b * T + j) * ldv + hh * D, ROW_BYTES, bar);
        }
    }
    mb_wait(bar + 1, 0);
    // logits: unit u = (head, 8-key tile); the accumulators stay in registers across the barrier that
    // retires the key slices, then land (scaled by 1/sqrt(64)) in the same memory as [row][head*Tk + key]
    const int ntk = (Tk + 7) >> 3, units = H * ntk;          // <= 20 for T <= 36: at most two units per warp
    float lg[2][4];
#pragma unroll
    for (int uu = 0; uu < 2; uu++) {
        const int u = warp + uu * ANW;
        float m[4] = {0.f, 0.f, 0.f, 0.f}, sq[4] = {0.f, 0.f, 0.f, 0.f};
        if (u < units) {
            const int hh = u / ntk, nt = u - hh * ntk;
#pragma unroll
            for (int kk = 0; kk < HD / 16; kk++) {
                uint32_t ah[4], al[4], bh[2], bl[2];
                load_a_frag(s_q, LDX, 0, nr, hh * HD + kk * 16, lane, ah, al);
                load_b_frag_rows(s_k + (size_t)hh * Tk * LDK, LDK, nt * 8, Tk, kk * 16, lane, bh, bl);
                mma_pairs(m, sq, ah, al, bh, bl);
            }
        }
#pragma unroll
        for (int e = 0; e < 4; e++) lg[uu][e] = fmaf(sq[e], 1.0f / 2048.0f, m[e]) * 0.125f;
    }
    __syncthreads();
#pragma unroll
    for (int uu = 0; uu < 2; uu++) {
        const int u = warp + uu * ANW;
        if (u < units) {
            const int hh = u / ntk, nt = u - hh * ntk, j = nt * 8 + 2 * c;
            float* pr = s_p + hh * Tk + j;
            if (j < Tk) { pr[g * pld] = lg[uu][0]; pr[(g + 8) * pld] = lg[uu][2]; }
            if (j + 1 < Tk) { pr[g * pld + 1] = lg[uu][1]; pr[(g + 8) * pld + 1] = lg[uu][3]; }
        }
    }
    __syncthreads();
    // one warp per (row, head): softmax over the Tk keys (contiguous); rows >= nr and the padding columns are zero
    for (int p = warp; p < SLAB * H; p += ANW) {
        const int r = p / H, hh = p - r * H;
        float* row = s_p + r * pld + hh * Tk;
        const float a0 = lane < Tk ? row[lane] : -INFINITY, a1 = lane + 32 < Tk ? row[lane + 32] : -INFINITY;
        float mx = fmaxf(a0, a1);
#pragma unroll
        for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float e0 = lane < Tk ? expf(a0 - mx) : 0.f, e1 = lane + 32 < Tk ? expf(a1 - mx) : 0.f;
        const float inv = r < nr ? 1.0f / warp_sum(e0 + e1) : 0.f;
        if (lane < Tk) row[lane] = e0 * inv;
        if (lane + 32 < Tk) row[lane + 32] = e1 * inv;
    }
    for (int i = tid; i < SLAB * (HT16 - HT); i += ANT) s_p[(i / (HT16 - HT)) * pld + HT + i % (HT16 - HT)] = 0.f;
    mb_wait(bar, 0);
    __syncthreads();
    // values: z[16 x 256] = P[16 x HT] V'[HT x 256]; warp w owns output columns 16w .. 16w+15
    {
        float m0[4] = {0.f, 0.f, 0.f, 0.f}, m1[4] = {0.f, 0.f, 0.f, 0.f}, q0[4] = {0.f, 0.f, 0.f, 0.f}, q1[4] = {0.f, 0.f, 0.f, 0.f};
        const int n0 = warp * 16;
#pragma unroll 2
        for (int kk = 0; kk < HT16 / 16; kk++) {
            uint32_t ah[4], al[4], bh[2], bl[2];
            load_a_frag(s_p, pld, 0, SLAB, kk * 16, lane, ah, al);
            load_b_frag_cols(s_v, VLD, kk * 16, HT, n0, lane, bh, bl);
            mma_pairs(m0, q0, ah, al, bh, bl);
            load_b_frag_cols(s_v, VLD, kk * 16, HT, n0 + 8, lane, bh, bl);
            mma_pairs(m1, q1, ah, al, bh, bl);
        }
        const float sc = 1.0f / 2048.0f;
#pragma unroll
        for (int t = 0; t < 2; t++) {
            const float* am = t ? m1 : m0;
            const float* aq = t ? q1 : q0;
            const int n = n0 + t * 8 + 2 * c;
            const float2 bb = *reinterpret_cast<const float2*>(s_par + n);
            if (g < nr) {
                float2* zz = reinterpret_cast<float2*>(s_z + g * LDZ + n);
                const float2 rr = *zz;
                *zz = make_float2((fmaf(aq[0], sc, am[0]) + bb.x) + rr.x, (fmaf(aq[1], sc, am[1]) + bb.y) + rr.y);
            }
            if (g + 8 < nr) {
                float2* zz = reinterpret_cast<float2*>(s_z + (g + 8) * LDZ + n);
                const float2 rr = *zz;
                *zz = make_float2((fmaf(aq[2], sc, am[2]) + bb.x) + rr.x, (fmaf(aq[3], sc, am[3]) + bb.y) + rr.y);
            }
        }
    }
    __syncthreads();
    for (int r = warp; r < nr; r += ANW) {
        const size_t o = (size_t)(b * T + r0 + r) * D;
        warp_ln_row(s_z + r * LDZ, s_par + D, s_par + 2 * D, out + o, lane, out_b ? out_b + o : nullptr, out_s ? out_s + o : nullptr);
    }
}

__global__ void __launch_bounds__(ANT)
k_attn_ln(const AttnArgs aa) {
    extern __shared__ __align__(16) float sm[];
    if (threadIdx.x == 0) chain_mark(4, 0);
    attn_body(aa, sm, blockIdx.x, blockIdx.y * SLAB);
    if (c_chain) { __syncthreads(); if (threadIdx.x == 0) chain_mark(4, 2); }
}

// Step-invariant B operands (folded queries, folded memory keys / values) are split into fp16 (hi, lo) ONCE (at
// commit / bind) so that their fragments are plain 32-bit loads: rows operands as fp16 [rows][KPH] (k contiguous),
// K x N operands with the two k-neighbours of a column packed in one word, [K/2][VPW].  Strides: KPH/2 = 4 mod 32
// words, VPW = 8 mod 32 words (conflict-free).
__device__ __forceinline__ void load_b_frag_rows_pk(const __half* __restrict__ sh, const __half* __restrict__ sl, int n0, int nrows,
                                                    int k0, int lane, uint32_t (&hi)[2], uint32_t (&lo)[2]) {
    const int off = min(n0 + (lane >> 2), nrows - 1) * KPH + k0 + 2 * (lane & 3);
    hi[0] = *reinterpret_cast<const uint32_t*>(sh + off); hi[1] = *reinterpret_cast<const uint32_t*>(sh + off + 8);
    lo[0] = *reinterpret_cast<const uint32_t*>(sl + off); lo[1] = *reinterpret_cast<const uint32_t*>(sl + off + 8);
}
__device__ __forceinline__ void load_b_frag_cols_pk(const uint32_t* __restrict__ sh, const uint32_t* __restrict__ sl, int k0, int nkp,
                                                    int n0, int lane, uint32_t (&hi)[2], uint32_t (&lo)[2]) {
    const int g = lane >> 2, c = lane & 3;
    const int o0 = min((k0 >> 1) + c, nkp - 1) * VPW + n0 + g, o1 = min((k0 >> 1) + c + 4, nkp - 1) * VPW + n0 + g;
    hi[0] = sh[o0]; hi[1] = sh[o1]; lo[0] = sl[o0]; lo[1] = sl[o1];
}

// ---------------------------------------------------------------------------------------------
// Cross-attention block with BOTH projections folded into the step-invariant memory tensors:
//   logit[t,h,j] = x1[t] . kp[h,j] + kc[h,j]      kp = (K_h Wq_h)/8 (256-vector), kc = (bq_h . K_h)/8
//   out[t] = LN2( x1[t] + bo + sum_{h,j} softmax_j(logit)[t,h,j] vp[h,j] )      vp = V_h Wo_h^T
// so no query GEMM is needed and the block can run right after the layer's first sub-block while its
// x1 rows are still in shared memory.  s_kph/s_kpl [HT][KPH] fp16, s_kc [HT], s_vph/s_vpl [HT/2][VPW] and the parameter rows
// s_bo / s_lnw / s_lnb must already be staged.  Tk <= 16, H*Tk <= 64.
__device__ __forceinline__ void cross_attention_tail(const float* __restrict__ s_x1, const __half* __restrict__ s_kph,
                                                     const __half* __restrict__ s_kpl, const float* __restrict__ s_kc,
                                                     const uint32_t* __restrict__ s_vph, const uint32_t* __restrict__ s_vpl,
                                                     float* __restrict__ s_p, float* __restrict__ s_z, int nr, int HT, int Tk, int H,
                                                     const float* __restrict__ s_bo, const float* __restrict__ s_lnw,
                                                     const float* __restrict__ s_lnb, float* __restrict__ out,
                                                     __half* __restrict__ out_b, __half* __restrict__ out_s, size_t row0,
                                                     bool trace = false) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, c = lane & 3;
    // logits: warp (ks = warp & 3, ng = warp >> 2) accumulates the 8-key column tiles ng and ng + 4 over the
    // 16-wide k-steps [4 ks, 4 ks + 4); the k-slice partial tiles go to s_z (free until the value pass)
    {
        const int ks = warp & 3, ng = warp >> 2, ntiles = (HT + 7) >> 3;
        const bool t1 = ng + 4 < ntiles;
        if (ng < ntiles) {
            float m0[4] = {0.f, 0.f, 0.f, 0.f}, m1[4] = {0.f, 0.f, 0.f, 0.f}, q0[4] = {0.f, 0.f, 0.f, 0.f}, q1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
            for (int kk = ks * 4; kk < ks * 4 + 4; kk++) {
                uint32_t ah[4], al[4], bh[2], bl[2];
                load_a_frag(s_x1, LDX, 0, nr, kk * 16, lane, ah, al);
                load_b_frag_rows_pk(s_kph, s_kpl, ng * 8, HT, kk * 16, lane, bh, bl);
                mma_pairs(m0, q0, ah, al, bh, bl);
                if (t1) {
                    load_b_frag_rows_pk(s_kph, s_kpl, (ng + 4) * 8, HT, kk * 16, lane, bh, bl);
                    mma_pairs(m1, q1, ah, al, bh, bl);
                }
            }
            const float sc = 1.0f / 2048.0f;
            float* pp = s_z + (ks * SLAB + g) * XLDP + ng * 8 + 2 * c;
            *reinterpret_cast<float2*>(pp) = make_float2(fmaf(q0[0], sc, m0[0]), fmaf(q0[1], sc, m0[1]));
            *reinterpret_cast<float2*>(pp + 8 * XLDP) = make_float2(fmaf(q0[2], sc, m0[2]), fmaf(q0[3], sc, m0[3]));
            if (t1) {
                *reinterpret_cast<float2*>(pp + 32) = make_float2(fmaf(q1[0], sc, m1[0]), fmaf(q1[1], sc, m1[1]));
                *reinterpret_cast<float2*>(pp + 8 * XLDP + 32) = make_float2(fmaf(q1[2], sc, m1[2]), fmaf(q1[3], sc, m1[3]));
            }
        }
    }
    __syncthreads();
    if (trace) ATRACE(7);
    // one warp per row, 8 lanes per head (H <= 4), lane `sub` holds keys sub and sub + 8 (Tk <= 16): fixed-order sum of
    // the 4 k-slices + constant term, softmax over the Tk memory slots with 3-step shuffles inside the 8-lane group;
    // probabilities row-major [row][hj] (zero for rows >= nr and for the padding columns up to a multiple of 16) as
    // the A operand of the value product
    {
        const int r = warp, hh = lane >> 3, sub = lane & 7;
        const bool on0 = hh < H && sub < Tk, on1 = hh < H && sub + 8 < Tk;
        const int hj0 = hh * Tk + sub, hj1 = hj0 + 8;
        float a0 = -INFINITY, a1 = -INFINITY;
        if (on0) {
            const float* pp = s_z + r * XLDP + hj0;
            a0 = (((pp[0] + pp[SLAB * XLDP]) + pp[2 * SLAB * XLDP]) + pp[3 * SLAB * XLDP]) + s_kc[hj0];
        }
        if (on1) {
            const float* pp = s_z + r * XLDP + hj1;
            a1 = (((pp[0] + pp[SLAB * XLDP]) + pp[2 * SLAB * XLDP]) + pp[3 * SLAB * XLDP]) + s_kc[hj1];
        }
        float mx = fmaxf(a0, a1);
#pragma unroll
        for (int o = 4; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        const float e0 = on0 ? expf(a0 - mx) : 0.f, e1 = on1 ? expf(a1 - mx) : 0.f;
        float sum = e0 + e1;
#pragma unroll
        for (int o = 4; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
        const float inv = r < nr ? 1.0f / sum : 0.f;
        if (on0) s_p[r * PLD + hj0] = e0 * inv;
        if (on1) s_p[r * PLD + hj1] = e1 * inv;
        const int pad = ((HT + 15) & ~15) - HT;
        for (int i = tid; i < SLAB * pad; i += ANT) s_p[(i / pad) * PLD + HT + i % pad] = 0.f;
    }
    __syncthreads();
    if (trace) ATRACE(8);
    // values: z[16 x 256] = P[16 x HT] V'[HT x 256]; warp w owns output columns 16w .. 16w+15 (two n-tiles),
    // then bias + residual straight from the accumulator fragments
    {
        float m0[4] = {0.f, 0.f, 0.f, 0.f}, m1[4] = {0.f, 0.f, 0.f, 0.f}, q0[4] = {0.f, 0.f, 0.f, 0.f}, q1[4] = {0.f, 0.f, 0.f, 0.f};
        const int n0 = warp * 16, nks = (HT + 15) >> 4;
        for (int kk = 0; kk < nks; kk++) {
            uint32_t ah[4], al[4], bh[2], bl[2];
            load_a_frag(s_p, PLD, 0, SLAB, kk * 16, lane, ah, al);
            load_b_frag_cols_pk(s_vph, s_vpl, kk * 16, HT >> 1, n0, lane, bh, bl);
            mma_pairs(m0, q0, ah, al, bh, bl);
            load_b_frag_cols_pk(s_vph, s_vpl, kk * 16, HT >> 1, n0 + 8, lane, bh, bl);
            mma_pairs(m1, q1, ah, al, bh, bl);
        }
        const float sc = 1.0f / 2048.0f;
#pragma unroll
        for (int t = 0; t < 2; t++) {
            const float* am = t ? m1 : m0;
            const float* aq = t ? q1 : q0;
            const int n = n0 + t * 8 + 2 * c;
            const float2 bb = *reinterpret_cast<const float2*>(s_bo + n);
            if (g < nr) {
                const float2 rr = *reinterpret_cast<const float2*>(s_x1 + g * LDX + n);
                *reinterpret_cast<float2*>(s_z + g * LDZ + n) = make_float2((fmaf(aq[0], sc, am[0]) + bb.x) + rr.x, (fmaf(aq[1], sc, am[1]) + bb.y) + rr.y);
            }
            if (g + 8 < nr) {
                const float2 rr = *reinterpret_cast<const float2*>(s_x1 + (g + 8) * LDX + n);
                *reinterpret_cast<float2*>(s_z + (g + 8) * LDZ + n) = make_float2((fmaf(aq[2], sc, am[2]) + bb.x) + rr.x, (fmaf(aq[3], sc, am[3]) + bb.y) + rr.y);
            }
        }
    }
    __syncthreads();
    if (trace) ATRACE(9);
    for (int r = warp; r < nr; r += ANW) {
        const size_t o = (row0 + r) * D;
        warp_ln_row(s_z + r * LDZ, s_lnw, s_lnb, out + o, lane, out_b ? out_b + o : nullptr, out_s ? out_s + o : nullptr);
    }
}

// stage the packed folded memory tensors of sample b (k_pack_memory's block): ONE bulk copy, issued by the calling thread
__device__ __forceinline__ void stage_memory(const uint8_t* __restrict__ mpack, __half* __restrict__ s_kph, int b, int HT, uint64_t* bar) {
    bulk_g2s(s_kph, mpack + (size_t)b * mem_block_bytes(HT), (uint32_t)mem_block_bytes(HT), bar);
}

// standalone cross-attention block (layers whose first sub-block is the standard self-attention)
struct XattnArgs {
    const float* x1; const uint8_t* mpack; const float *bo, *lnw, *lnb;      // mpack: k_pack_memory's per-sample blocks
    float* out; __half *out_b, *out_s; int T, B, Tk, H;
};
// own_rows: the x1 rows were written by THIS CTA with plain stores just before (fused standard layer): read them back with
// plain L2 loads instead of bulk copies (which would need a proxy fence)
__device__ __forceinline__ void xattn_body(const XattnArgs& xa, float* sm, const int b, const int r0, const bool own_rows) {
    const float* __restrict__ x1 = xa.x1;
    const float* __restrict__ bo = xa.bo; const float* __restrict__ lnw = xa.lnw; const float* __restrict__ lnb = xa.lnb;
    float* __restrict__ out = xa.out; __half* __restrict__ out_b = xa.out_b; __half* __restrict__ out_s = xa.out_s;
    const int T = xa.T, Tk = xa.Tk, H = xa.H;
    const int HT = H * Tk;
    uint64_t* bar = reinterpret_cast<uint64_t*>(sm);   // [0]: step-invariant tensors, [1]: input rows
    float* s_par = sm + 4;                  // bo, lnw, lnb
    float* s_x1 = s_par + 3 * D;            // [SLAB][LDX]
    __half* s_kph = reinterpret_cast<__half*>(s_x1 + SLAB * LDX);      // [HT][KPH] fp16, hi then lo     } one block, laid out like
    __half* s_kpl = s_kph + HT * KPH;                                  //                                 } k_pack_memory's
    uint32_t* s_vph = reinterpret_cast<uint32_t*>(s_kpl + HT * KPH);   // [HT/2][VPW] k-pair words, hi then lo
    uint32_t* s_vpl = s_vph + (HT >> 1) * VPW;
    float* s_kc = reinterpret_cast<float*>(s_vpl + (HT >> 1) * VPW);   // [HT] (padded to a multiple of 4)
    float* s_a = s_kc + ((HT + 3) & ~3);    // [SLAB][PLD]     probabilities
    float* s_z = s_a + SLAB * PLD;          // [SLAB][LDZ]
    const int nr = min(SLAB, T - r0), tid = threadIdx.x;
    pdl_trigger();
    if (tid == 0) {
        // the initialising thread issues every step-invariant copy itself, at once (they overlap the previous kernel under
        // programmatic dependent launch, or - when this CTA only got an SM after the previous kernel left it - the row loads)
        mb_init(bar, 1); mb_init(bar + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mb_expect_tx(bar, 3u * ROW_BYTES + (uint32_t)mem_block_bytes(HT));
        bulk_g2s(s_par, bo, ROW_BYTES, bar); bulk_g2s(s_par + D, lnw, ROW_BYTES, bar); bulk_g2s(s_par + 2 * D, lnb, ROW_BYTES, bar);
        stage_memory(xa.mpack, s_kph, b, HT, bar);
    }
    __syncthreads();
    pdl_wait();
    if (tid == 0) chain_mark(0, 1);
    if (own_rows) {
        for (int i = tid; i < nr * (D / 4); i += ANT) {
            const int l = i / (D / 4), c = i % (D / 4);
            *reinterpret_cast<float4*>(s_x1 + l * LDX + c * 4) = __ldcg(reinterpret_cast<const float4*>(x1 + (size_t)(b * T + r0 + l) * D) + c);
        }
    } else {
        if (tid == 0) mb_expect_tx(bar + 1, (uint32_t)nr * ROW_BYTES);
        __syncwarp();
        if (tid < nr) bulk_g2s(s_x1 + tid * LDX, x1 + (size_t)(b * T + r0 + tid) * D, ROW_BYTES, bar + 1);
    }
    mb_wait(bar, 0);
    if (!own_rows) mb_wait(bar + 1, 0);
    __syncthreads();     // own rows were written with plain stores
    cross_attention_tail(s_x1, s_kph, s_kpl, s_kc, s_vph, s_vpl, s_a, s_z, nr, HT, Tk, H, s_par, s_par + D, s_par + 2 * D, out, out_b,
                         out_s, (size_t)b * T + r0);
}

__global__ void __launch_bounds__(ANT)
k_xattn_ln(const XattnArgs xa) {
    extern __shared__ __align__(16) float sm[];
    if (threadIdx.x == 0) chain_mark(5, 0);
    xattn_body(xa, sm, blockIdx.x, blockIdx.y * SLAB, false);
    if (c_chain) { __syncthreads(); if (threadIdx.x == 0) chain_mark(5, 2); }
}

// Standard decoder layer, attention half in ONE launch: self-attention + LN1 (attn_body) and - on the rows this CTA has just
// written - cross-attention + LN2 (xattn_body), on the same shared memory one after the other.  Saves the kernel boundary
// between the two (hand-off, CTA launch, a second prologue: ~3 us of a step's critical path per layer).
__global__ void __launch_bounds__(ANT)
k_attn_xattn_ln(const AttnArgs aa, const XattnArgs xa) {
    extern __shared__ __align__(16) float sm[];
    if (threadIdx.x == 0) chain_mark(4, 0);
    attn_body(aa, sm, blockIdx.x, blockIdx.y * SLAB);
    __syncthreads();                 // every warp's LN1 rows are in global memory (this CTA reads them back below)
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr(sm)) : "memory");
        asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr(sm) + 8u) : "memory");
    }
    __syncthreads();
    xattn_body(xa, sm, blockIdx.x, blockIdx.y * SLAB, true);
    if (c_chain) { __syncthreads(); if (threadIdx.x == 0) chain_mark(4, 2); }
}

// QaN block + residual + LayerNorm1 (model/sublayers.py:343-352 + :332) for a slab of <= 16 rows of
// one sample, with an optional LayerNorm applied to the input rows first (the previous layer's
// pending norm3).   grid (B, ceil(T/16)), block 512.
//   x = pre ? LN_pre(zin) : zin
//   logit[t,n,s] = x[t+s-1] . Qt[s][n]   (Qt = rotary-folded, 1/16-scaled normalised queries; s = key slot)
//   a = softmax over the valid slots;  y[t] = sum_s (sum_n wk[n] a[t,n,s]) x[t+s-1];  out = LN1(x + y)
// ... followed, in the same kernel, by the layer's cross-attention block (cross_attention_tail) on the
// LN1 rows, which never leave shared memory.
struct QanArgs {
    const float *zin, *prew, *preb; const __half* qpack; const float *wk, *lnw, *lnb;      // qpack: [2 (hi, lo)][3N][KPH] folded queries
    const uint8_t* mpack; const float *bo2, *ln2w, *ln2b; float* out; __half *out_b, *out_s; int T, N, B, Tk, H;   // mpack: k_pack_memory's blocks
};
// the slab (sample b, rows r0 .. r0 + 15) of the kernel below as a device function on caller-provided shared memory `sm`
// (16-byte aligned, qan_smem() bytes): also phase A of the fused decoder-layer kernel
// PRELN = false: instantiated without the pending-LayerNorm code (the fused feed-forward kernel applies the previous layer's
// norm3 itself, so the hot path never has one pending; a skipped block of ~150 instructions still costs its instruction fetches)
template <bool XATTN, bool PRELN = true>
__device__ __forceinline__ void qan_xattn_body(const QanArgs& qa, float* sm, const int b, const int r0) {
    const float* __restrict__ zin = qa.zin; const float* __restrict__ prew = PRELN ? qa.prew : nullptr; const float* __restrict__ preb = qa.preb;
    const float* __restrict__ wk = qa.wk;
    const float* __restrict__ lnw = qa.lnw; const float* __restrict__ lnb = qa.lnb;
    const float* __restrict__ bo2 = qa.bo2; const float* __restrict__ ln2w = qa.ln2w;
    const float* __restrict__ ln2b = qa.ln2b; float* __restrict__ out = qa.out; __half* __restrict__ out_b = qa.out_b;
    __half* __restrict__ out_s = qa.out_s;
    const int T = qa.T, N = qa.N, Tk = qa.Tk, H = qa.H;
    const int HT = H * Tk, NQ = 3 * N;
    uint64_t* bar = reinterpret_cast<uint64_t*>(sm);   // [0]: step-invariant tensors, [1]: input rows
    float* s_par = sm + 4;                  // pre w, pre b, ln1 w, ln1 b, bo2, ln2 w, ln2 b
    float* s_x = s_par + 7 * D;             // [SLAB+2][LDX]   rows r0-1 .. r0+nr
    __half* s_qth = reinterpret_cast<__half*>(s_x + (SLAB + 2) * LDX);   // [NQ <= 30][KPH] fp16 folded queries, hi then lo (= qpack)
    __half* s_qtl = s_qth + NQ * KPH;
    float* s_x1 = reinterpret_cast<float*>(s_qth + 2 * 30 * KPH);       // [SLAB][LDX]     LN1 rows (input of the cross-attention block)
    __half* s_kph = reinterpret_cast<__half*>(s_x1 + SLAB * LDX);        // [HT][KPH]       } one block, laid out like
    __half* s_kpl = s_kph + HT * KPH;                                    //                 } k_pack_memory's
    uint32_t* s_vph = reinterpret_cast<uint32_t*>(s_kpl + HT * KPH);     // [HT/2][VPW]
    uint32_t* s_vpl = s_vph + (HT >> 1) * VPW;
    float* s_kc = reinterpret_cast<float*>(s_vpl + (HT >> 1) * VPW);     // [HT] (padded to a multiple of 4)
    float* s_a = s_kc + ((HT + 3) & ~3);                                 // [SLAB][PLD]     probabilities
    float* s_z = XATTN ? s_a + SLAB * PLD : s_x1;   // [SLAB][LDZ]  (encoder variant: no cross-attention buffers at all)
    const int nr = min(SLAB, T - r0), tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    // Everything step-invariant (parameter rows, the folded queries as ONE block, the sample's folded memory keys / values / kc
    // as ONE block) is requested by the thread that initialises the barriers, before the CTA-wide barrier: the copies
    // overlap the previous kernel's tail under programmatic dependent launch, or - when this CTA only got its SM after the
    // previous kernel left it - the loads of the input rows r0-1 .. r0+nr (halo of one on each side, l = t - (r0 - 1)).
    // Two barriers: [0] parameters + folded queries (needed by the QaN block right away), [1] the memory block (84 KB, needed
    // only by the cross-attention block: its copy overlaps the QaN block).
    pdl_trigger();
    ATRACE(0);
    if (tid == 0) {
        mb_init(bar, 1); mb_init(bar + 1, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        const int npar = (prew ? 2 : 0) + 2 + (XATTN ? 3 : 0);
        const uint32_t qbytes = (uint32_t)(2 * NQ * KPH * sizeof(__half));
        mb_expect_tx(bar, (uint32_t)npar * ROW_BYTES + qbytes);
        bulk_g2s(s_qth, qa.qpack, qbytes, bar);
        if (prew) { bulk_g2s(s_par, prew, ROW_BYTES, bar); bulk_g2s(s_par + D, preb, ROW_BYTES, bar); }
        bulk_g2s(s_par + 2 * D, lnw, ROW_BYTES, bar); bulk_g2s(s_par + 3 * D, lnb, ROW_BYTES, bar);
        if (XATTN) {
            bulk_g2s(s_par + 4 * D, bo2, ROW_BYTES, bar); bulk_g2s(s_par + 5 * D, ln2w, ROW_BYTES, bar); bulk_g2s(s_par + 6 * D, ln2b, ROW_BYTES, bar);
            mb_expect_tx(bar + 1, (uint32_t)mem_block_bytes(HT));
            stage_memory(qa.mpack, s_kph, b, HT, bar + 1);
        }
    }
    __syncthreads();
    const float wk_n = lane < N ? wk[lane] : 0.f;
    ATRACE(1);
    pdl_wait();
    if (tid == 0) chain_mark(0, 1);
    ATRACE(2);
    {
        // the input rows were just written by the previous kernel (L2 resident): plain 16-byte loads straight into the
        // padded shared-memory rows cost one L2 round trip, about half the latency of a bulk copy + mbarrier
        for (int i = tid; i < (nr + 2) * (D / 4); i += ANT) {
            const int l = i / (D / 4), c = i % (D / 4), t = r0 - 1 + l;
            if (t >= 0 && t < T)
                *reinterpret_cast<float4*>(s_x + l * LDX + c * 4) = __ldcg(reinterpret_cast<const float4*>(zin + (size_t)(b * T + t) * D) + c);
        }
    }
    mb_wait(bar, 0);
    __syncthreads();     // s_x rows were written with plain stores
    ATRACE(3);
    if (prew) {   // the previous layer's pending LayerNorm3, in place on the staged rows
        for (int l = warp; l < nr + 2; l += ANW) {
            const int t = r0 - 1 + l;
            if (t >= 0 && t < T) warp_ln_row(s_x + l * LDX, s_par, s_par + D, s_x + l * LDX, lane);
        }
        __syncthreads();
    }
    // part[ks][l][j] = (k-slice of) x[row l] . Qt[j] for all nr+2 staged rows and the 3N folded queries
    // on the tensor cores (fp16-pair fragments); s_z is free until the cross-attention block and holds the partials.
    ATRACE(4);
    {
        // warp (mt = warp & 1, np = (warp >> 1) & 1, ks = warp >> 2): row tile mt (rows 16 mt ..), query tiles
        // 2 np, 2 np + 1, 16-wide k-steps [4 ks, 4 ks + 4)
        const int mt = warp & 1, np = (warp >> 1) & 1, ks = warp >> 2, g = lane >> 2, c = lane & 3;
        float m0[4] = {0.f, 0.f, 0.f, 0.f}, m1[4] = {0.f, 0.f, 0.f, 0.f}, q0[4] = {0.f, 0.f, 0.f, 0.f}, q1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 2
        for (int kk = ks * 4; kk < ks * 4 + 4; kk++) {
            uint32_t ah[4], al[4], bh[2], bl[2];
            load_a_frag(s_x, LDX, mt * 16, nr + 2, kk * 16, lane, ah, al);
            load_b_frag_rows_pk(s_qth, s_qtl, np * 16, NQ, kk * 16, lane, bh, bl);
            mma_pairs(m0, q0, ah, al, bh, bl);
            load_b_frag_rows_pk(s_qth, s_qtl, np * 16 + 8, NQ, kk * 16, lane, bh, bl);
            mma_pairs(m1, q1, ah, al, bh, bl);
        }
        const float sc = 1.0f / 2048.0f;
        float* pp = s_z + (ks * 32 + mt * 16 + g) * P1LD + np * 16 + 2 * c;
        *reinterpret_cast<float2*>(pp) = make_float2(fmaf(q0[0], sc, m0[0]), fmaf(q0[1], sc, m0[1]));
        *reinterpret_cast<float2*>(pp + 8 * P1LD) = make_float2(fmaf(q0[2], sc, m0[2]), fmaf(q0[3], sc, m0[3]));
        *reinterpret_cast<float2*>(pp + 8) = make_float2(fmaf(q1[0], sc, m1[0]), fmaf(q1[1], sc, m1[1]));
        *reinterpret_cast<float2*>(pp + 8 * P1LD + 8) = make_float2(fmaf(q1[2], sc, m1[2]), fmaf(q1[3], sc, m1[3]));
    }
    __syncthreads();
    ATRACE(5);
    // One warp per output row: lane n < N sums the k-slices of its 3 slot logits (row l = r + slot feeds
    // output row r), softmax over the valid slots, times wk[n]; three warp sums give the row's tap
    // weights c[slot] = sum_n wk[n] a[n][slot]; then y = 3-tap filter, residual and LayerNorm1 in registers.
    for (int r = warp; r < nr; r += ANW) {
        const int t = r0 + r;
        const bool v0 = t > 0, v2 = t < T - 1;
        float w0 = 0.f, w1 = 0.f, w2 = 0.f;
        if (lane < N) {
            float lg[3];
#pragma unroll
            for (int sl = 0; sl < 3; sl++) {
                const float* pp = s_z + (r + sl) * P1LD + sl * N + lane;
                lg[sl] = ((pp[0] + pp[32 * P1LD]) + pp[2 * 32 * P1LD]) + pp[3 * 32 * P1LD];
            }
            const float l1 = lg[1], l0 = v0 ? lg[0] : -INFINITY, l2 = v2 ? lg[2] : -INFINITY;
            const float mx = fmaxf(l1, fmaxf(l0, l2));
            const float e0 = v0 ? expf(l0 - mx) : 0.f, e1 = expf(l1 - mx), e2 = v2 ? expf(l2 - mx) : 0.f;
            const float wn = wk_n / (e0 + e1 + e2);
            w0 = wn * e0; w1 = wn * e1; w2 = wn * e2;
        }
        const float c0 = warp_sum(w0), c1 = warp_sum(w1), c2 = warp_sum(w2);
        const float* xm = s_x + (r + 1) * LDX;          // row t
        float v[8];
#pragma unroll
        for (int half = 0; half < 2; half++) {
            const int c = half * 128 + lane * 4;
            const float4 x1 = *reinterpret_cast<const float4*>(xm + c);
            float4 y = make_float4(c1 * x1.x, c1 * x1.y, c1 * x1.z, c1 * x1.w);
            if (v0) {
                const float4 x0 = *reinterpret_cast<const float4*>(xm - LDX + c);
                y.x = fmaf(c0, x0.x, y.x); y.y = fmaf(c0, x0.y, y.y); y.z = fmaf(c0, x0.z, y.z); y.w = fmaf(c0, x0.w, y.w);
            }
            if (v2) {
                const float4 x2 = *reinterpret_cast<const float4*>(xm + LDX + c);
                y.x = fmaf(c2, x2.x, y.x); y.y = fmaf(c2, x2.y, y.y); y.z = fmaf(c2, x2.z, y.z); y.w = fmaf(c2, x2.w, y.w);
            }
            v[half * 4 + 0] = x1.x + y.x; v[half * 4 + 1] = x1.y + y.y; v[half * 4 + 2] = x1.z + y.z; v[half * 4 + 3] = x1.w + y.w;
        }
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < 8; i++) s += v[i];
        const float mean = warp_sum(s) * (1.0f / D);
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < 8; i++) { const float d = v[i] - mean; q = fmaf(d, d, q); }
        const float rstd = 1.0f / sqrtf(warp_sum(q) * (1.0f / D) + 1e-5f);
        float4 o[2];
#pragma unroll
        for (int half = 0; half < 2; half++) {
            const int c = half * 128 + lane * 4;
            const float4 w4 = *reinterpret_cast<const float4*>(s_par + 2 * D + c), b4 = *reinterpret_cast<const float4*>(s_par + 3 * D + c);
            o[half].x = (v[half * 4 + 0] - mean) * rstd * w4.x + b4.x; o[half].y = (v[half * 4 + 1] - mean) * rstd * w4.y + b4.y;
            o[half].z = (v[half * 4 + 2] - mean) * rstd * w4.z + b4.z; o[half].w = (v[half * 4 + 3] - mean) * rstd * w4.w + b4.w;
            if (XATTN) *reinterpret_cast<float4*>(s_x1 + r * LDX + c) = o[half];
        }
        if (!XATTN) {      // encoder layer: LayerNorm1 rows are the kernel's output (fp32 + fp16 pairs for the feed-forward block)
            const size_t orow = ((size_t)b * T + r0 + r) * D;
            *reinterpret_cast<float4*>(out + orow + lane * 4) = o[0];
            *reinterpret_cast<float4*>(out + orow + 128 + lane * 4) = o[1];
            if (out_b) store_pairs(o[0], o[1], out_b + orow, out_s + orow, lane);
        }
    }
    if (!XATTN) return;
    mb_wait(bar + 1, 0);     // memory keys / values have landed (copied while the QaN block ran)
    __syncthreads();
    ATRACE(6);
    cross_attention_tail(s_x1, s_kph, s_kpl, s_kc, s_vph, s_vpl, s_a, s_z, nr, HT, Tk, H, s_par + 4 * D, s_par + 5 * D, s_par + 6 * D,
                         out, out_b, out_s, (size_t)b * T + r0, true);
    ATRACE(11);
}

template <bool XATTN, bool PRELN = true>
__global__ void __launch_bounds__(ANT)
k_qan_xattn_ln(const QanArgs qa) {
    extern __shared__ __align__(16) float sm[];
    if (threadIdx.x == 0) chain_mark(3, 0);
    qan_xattn_body<XATTN, PRELN>(qa, sm, blockIdx.x, blockIdx.y * SLAB);
    if (c_chain) { __syncthreads(); if (threadIdx.x == 0) chain_mark(3, 2); }
}

// ---------------------------------------------------------------------------------------------
// One QaN decoder layer in ONE launch: QaN block + LN1 + cross-attention + LN2 (phase A, the kernel above as a device
// function) and the feed-forward block + the layer's final LayerNorm (phase B, tc::mlp_run).  A cluster of 8 CTAs owns G whole
// samples (G = 8 / ceil(T / 16): 4 samples = 120 rows for T = 30): in phase A CTA c takes slab c % nslabs of the cluster's
// sample c / nslabs; the LN2 rows (fp32 for the residual, fp16 pairs for the tensor core) go to global memory (L2); after a
// cluster barrier the same 8 CTAs run the feed-forward block on the cluster's rows as one 128-row tile (rows past G T belong to
// the next cluster: computed, never reduced or stored).  Tiles aligned to samples mean NO dependency between clusters, so the
// kernel boundary between the two halves of a layer disappears.  The attention phase uses the operand region of the
// feed-forward block as its shared memory; the feed-forward barriers and the TMEM allocation sit above it and are set up at entry.
__global__ void __cluster_dims__(tc::mlp::CLUSTER, 1, 1) __launch_bounds__(ANT, 1)
k_layer_qan_fused(const QanArgs qa, const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w1,
                  const __grid_constant__ CUtensorMap map_xl, const __grid_constant__ CUtensorMap map_w1l,
                  const __grid_constant__ CUtensorMap map_w2, const __grid_constant__ CUtensorMap map_w2l,
                  const float* __restrict__ b1, const float* __restrict__ b2, const float* __restrict__ res, float* __restrict__ Z,
                  const float* __restrict__ ln_w, const float* __restrict__ ln_b, __half* __restrict__ Zh, __half* __restrict__ Zl,
                  int M, int G, int nslabs) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    pdl_trigger();
    const int c = blockIdx.x, cl = blockIdx.y, tid = threadIdx.x;
    tc::MlpArgs a{&map_x, &map_w1, &map_xl, &map_w1l, &map_w2, &map_w2l, b1, b2, res, D, Z, D, ln_w, ln_b, Zh, Zl, nullptr};
    const uint32_t tmem_base = tc::mlp_setup<8>(smem_raw, a);
    // ---- phase A
    const int sl = c / nslabs, b = cl * G + sl;
    const bool attend = sl < G && b < qa.B;
    if (attend) qan_xattn_body<true>(qa, reinterpret_cast<float*>(smem_raw), b, (c % nslabs) * SLAB);
    else pdl_wait();
    // this CTA's rows (plain stores) must be visible to the TMA reads and plain loads of the whole cluster
    __threadfence();
    asm volatile("fence.proxy.async;" ::: "memory");
    __syncthreads();
    if (tid == 0 && attend) {   // the attention phase's two mbarriers sit in memory the operand ring is about to overwrite
        asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr(smem_raw)) : "memory");
        asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr(smem_raw) + 8u) : "memory");
    }
    tc::cluster_sync_all();
    asm volatile("fence.proxy.async;" ::: "memory");
    // ---- phase B
    const int m0 = cl * G * qa.T;
    tc::mlp_run<8>(smem_raw, a, c, m0, min(M, m0 + G * qa.T), tmem_base, false, nullptr);
    tc::mlp_teardown(tmem_base);
}

// The same for a standard decoder layer (layers 0 and 7): self-attention + LN1 (phase A1, on the folded-QKV projection a
// GEMM launch produced), cross-attention + LN2 (phase A2, on the rows phase A1 just wrote), feed-forward + LN3 (phase B).
__global__ void __cluster_dims__(tc::mlp::CLUSTER, 1, 1) __launch_bounds__(ANT, 1)
k_layer_std_fused(const AttnArgs aa, const XattnArgs xa, const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_w1,
                  const __grid_constant__ CUtensorMap map_xl, const __grid_constant__ CUtensorMap map_w1l,
                  const __grid_constant__ CUtensorMap map_w2, const __grid_constant__ CUtensorMap map_w2l,
                  const float* __restrict__ b1, const float* __restrict__ b2, const float* __restrict__ res, float* __restrict__ Z,
                  const float* __restrict__ ln_w, const float* __restrict__ ln_b, __half* __restrict__ Zh, __half* __restrict__ Zl,
                  int M, int G, int nslabs) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    pdl_trigger();
    const int c = blockIdx.x, cl = blockIdx.y, tid = threadIdx.x;
    tc::MlpArgs a{&map_x, &map_w1, &map_xl, &map_w1l, &map_w2, &map_w2l, b1, b2, res, D, Z, D, ln_w, ln_b, Zh, Zl, nullptr};
    const uint32_t tmem_base = tc::mlp_setup<8>(smem_raw, a);
    const int sl = c / nslabs, b = cl * G + sl, r0 = (c % nslabs) * SLAB;
    const bool attend = sl < G && b < xa.B;
    float* sm = reinterpret_cast<float*>(smem_raw);
    if (attend) {
        attn_body(aa, sm, b, r0);
        __syncthreads();                 // every warp's LN1 rows are in global memory (same CTA reads them back below)
        if (tid == 0) {
            asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr(smem_raw)) : "memory");
            asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr(smem_raw) + 8u) : "memory");
        }
        __syncthreads();
        xattn_body(xa, sm, b, r0, true);
    } else {
        pdl_wait();
    }
    __threadfence();
    asm volatile("fence.proxy.async;" ::: "memory");
    __syncthreads();
    if (tid == 0 && attend) {
        asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr(smem_raw)) : "memory");
        asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(smem_addr(smem_raw) + 8u) : "memory");
    }
    tc::cluster_sync_all();
    asm volatile("fence.proxy.async;" ::: "memory");
    const int m0 = cl * G * xa.T;
    tc::mlp_run<8>(smem_raw, a, c, m0, min(M, m0 + G * xa.T), tmem_base, false, nullptr);
    tc::mlp_teardown(tmem_base);
}

// ---------------------------------------------------------------------------------------------
// Step input / output kernel.  The sample tensors live as (B,1,C,T); the decoder works on token rows
// [B*T][.].  One kernel covers both ends of a sampling step so a plain step is "decoder GEMMs/attention
// + ONE tail kernel":
//   HEADS  (mode & 1): lin[(b*T+t)][Clin] -> x0 (B,1,C,T) with the skeleton's keypoint re-derivation and
//                      the inpainting blend (model/diffusion_smpl.py:245; model/diffusion_skeleton.py:218-248;
//                      diffusion/gaussian_diffusion.py:307-311)
//   FINISH (mode & 2): x_{t-1} = c1[i] x0 + c2[i] x_t + sigma[i] eps   (gaussian_diffusion.py:253-275,537-547),
//                      then - when emit_next - the NEXT step's token pairs and embedding addend, and the
//                      device step counter moves to i-1 (last block to finish, so nobody still reads it)
//   TOKENS (mode == 4): x (B,1,C,T) -> token pairs [B*T][Cp] + addend rows, for the first step of a loop and
//                      for the stand-alone forward
// addend[b*T+t][:] = (MLP(pe[t_b]) + b_in) + pe[t]  = table row + positional row (model/diffusion_smpl.py:227-232).
// grid (B, parts): a block owns a channel range of one sample, all T frames; every global load of the
// element phase is independent and issued in batches of 5 per thread.
struct StepIO {
    // heads
    const float* lin; const float* zero_pose; const float* gt; const unsigned char* mask; float* x0_out;
    // finish
    const float* x0_in; const float* xt; const float* noise; float* x_next;
    const StepParams* tbl; int* step_cur; int* ticket;
    int tape_mode, n_steps, emit_next;
    int i_host;     // >= 0: the step index, known when the launch is enqueued (else read from step_cur after the dependency wait)
    // tokens
    const float* x_in; const long long* tstep;
    __half* xtok_b; __half* xtok_s; const float* tab; const float* pe; float* add;
    int pe_rows, T, Clin, C, Cp, variant, c_body, n_points;
};

template <int MODE>
__global__ void __launch_bounds__(256) k_step_io(const StepIO a) {
    extern __shared__ float sm[];
    const int b = blockIdx.x, part = blockIdx.y, NP = gridDim.y, T = a.T, tid = threadIdx.x;
    const int ncp = (a.Cp + NP - 1) / NP, c0 = part * ncp, c1 = min(c0 + ncp, a.Cp);   // token columns (incl. zero padding)
    const int nc = max(min(c1, a.C) - c0, 0);                                            // real channels of this block
    const int LT = T + 1;
    float* tile = sm;                 // [ncp][T+1]
    float* pose = sm + ncp * LT;      // [T][8]  (skeleton: object translation + quaternion per frame)
    if (tid == 0) chain_mark(6, 0);
    pdl_trigger();
    const int n = nc * T;
    constexpr int KM = 5, NA = 3;
    float v_in[KM], v_xt[KM], v_nz[KM], v_gt[KM];
    unsigned char v_m[KM];
    int i_step = 0;
    StepParams sp = {};
    const float* nz = nullptr;
    // the loads of a batch of KM elements per thread, in two groups: "static" operands exist before the loop's first kernel
    // (noise tape, inpainting ground truth / mask), "dynamic" ones are written by earlier kernels of the chain
    auto step_setup = [&]() {
        sp = a.tbl[i_step];
        // tape_mode 0: `noise` is this step's eps; 1: `noise` is the tape (n_steps + 1 entries, [0] = x_T); 2: `noise` is a
        // device slot holding the tape pointer (captured graphs stay valid when the caller passes a new tape tensor)
        const float* base = a.tape_mode == 2 ? *reinterpret_cast<const float* const*>(a.noise) : a.noise;
        nz = a.tape_mode ? base + (size_t)(a.n_steps - i_step) * ((size_t)gridDim.x * a.C * T) : base;
    };
    auto load_static = [&](int base) {
#pragma unroll
        for (int k = 0; k < KM; k++) {
            const int e = base + tid + k * 256;
            v_nz[k] = v_gt[k] = 0.f; v_m[k] = 0;
            if (e < n) {
                const size_t o = ((size_t)b * a.C + c0) * T + e;        // (B,1,C,T): the block's channels are contiguous
                if (MODE & 2) v_nz[k] = nz[o];
                if ((MODE & 1) && a.mask) { v_m[k] = a.mask[o]; v_gt[k] = a.gt[o]; }
            }
        }
    };
    auto load_dynamic = [&](int base) {
#pragma unroll
        for (int k = 0; k < KM; k++) {
            const int e = base + tid + k * 256;
            v_in[k] = v_xt[k] = 0.f;
            if (e < n) {
                const size_t o = ((size_t)b * a.C + c0) * T + e;
                if (MODE == 2) v_in[k] = a.x0_in[o];
                if (MODE == 4) v_in[k] = a.x_in[o];
                if (MODE & 2) v_xt[k] = a.xt[o];
            }
        }
    };
    // When the host knows the step index at enqueue time (plain launches, whole-loop graph) nothing "static" depends on an
    // earlier kernel of the chain: the table entry, the noise / ground truth / mask of the first batch and the rows of the
    // next step's embedding addend are loaded BEFORE the dependency wait, under the previous kernel's tail (this kernel's
    // blocks are small enough to be resident next to it).
    const bool early = (MODE & 2) && a.i_host >= 0;
    const int nq = T * (D / 4), per = (nq + NP - 1) / NP, q1 = min(nq, (part + 1) * per);
    float4 add_pre[NA];
    bool add_early = false;
    if (early) {
        i_step = a.i_host;
        step_setup();
        load_static(0);
        if (a.emit_next && i_step > 0 && per <= NA * 256) {
            long long ti = a.tbl[i_step - 1].t;
            if (ti < 0) ti = 0;
            if (ti >= a.pe_rows) ti = a.pe_rows - 1;
            const float4* trow = reinterpret_cast<const float4*>(a.tab + (size_t)ti * D);
#pragma unroll
            for (int k = 0; k < NA; k++) {
                const int i = part * per + tid + k * 256;
                add_pre[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (i < q1) {
                    const float4 p4 = reinterpret_cast<const float4*>(a.pe + (size_t)(i / (D / 4)) * D)[i % (D / 4)];
                    const float4 o4 = trow[i % (D / 4)];
                    add_pre[k] = make_float4(o4.x + p4.x, o4.y + p4.y, o4.z + p4.z, o4.w + p4.w);
                }
            }
            add_early = true;
        }
    }
    pdl_wait();
    if (tid == 0) chain_mark(6, 1);
    if ((MODE & 2) && !early) { i_step = *a.step_cur; step_setup(); }
    if (MODE & 1) {
        // stage the block's linear-head columns, transposed; derived keypoint channels are rebuilt from the pose
        const float* lrow = a.lin + (size_t)b * T * a.Clin;
        for (int j = tid; j < n; j += 256) {
            const int t = j / nc, cc = j % nc, c = c0 + cc;
            int src = c;
            if (a.variant != 0 && c >= a.c_body) src = c >= a.c_body + 3 * a.n_points ? c - 3 * a.n_points : -1;
            if (src >= 0) tile[cc * LT + t] = lrow[(size_t)t * a.Clin + src];
        }
        if (a.variant != 0)
            for (int j = tid; j < T * 7; j += 256) pose[(j / 7) * 8 + j % 7] = lrow[(size_t)(j / 7) * a.Clin + a.c_body + j % 7];
    }
    load_dynamic(0);
    if (!early) load_static(0);
    if (MODE & 1) __syncthreads();
    for (int base = 0; base < n; base += 256 * KM) {
        if (base) { load_dynamic(base); load_static(base); }
#pragma unroll
        for (int k = 0; k < KM; k++) {
            const int e = base + tid + k * 256;
            if (e >= n) continue;
            const int cc = e / T, t = e % T, c = c0 + cc;
            const size_t o = ((size_t)b * a.C + c0) * T + e;
            float val = v_in[k];
            if (MODE & 1) {
                if (a.variant == 0 || c < a.c_body || c >= a.c_body + 3 * a.n_points) {
                    val = tile[cc * LT + t];
                } else {
                    // calc_obj_pred: pose = [trans3, quat xyzw]; quaternion_to_matrix on (w,x,y,z), un-normalised
                    const int p = (c - a.c_body) / 3, ax = (c - a.c_body) % 3;
                    const float* ps = pose + t * 8;
                    const float tx = ps[0], ty = ps[1], tz = ps[2], qi = ps[3], qj = ps[4], qk = ps[5], qr = ps[6];
                    const float two_s = 2.0f / (qr * qr + qi * qi + qj * qj + qk * qk);
                    float r0, r1, r2, tr;
                    if (ax == 0) { r0 = 1 - two_s * (qj * qj + qk * qk); r1 = two_s * (qi * qj - qk * qr); r2 = two_s * (qi * qk + qj * qr); tr = tx; }
                    else if (ax == 1) { r0 = two_s * (qi * qj + qk * qr); r1 = 1 - two_s * (qi * qi + qk * qk); r2 = two_s * (qj * qk - qi * qr); tr = ty; }
                    else { r0 = two_s * (qi * qk - qj * qr); r1 = two_s * (qj * qk + qi * qr); r2 = 1 - two_s * (qi * qi + qj * qj); tr = tz; }
                    const float* zp = a.zero_pose + ((size_t)b * a.n_points + p) * 3;
                    val = (r0 * zp[0] + r1 * zp[1] + r2 * zp[2]) + tr;
                }
                if (v_m[k]) val = v_gt[k];
                if (a.x0_out) a.x0_out[o] = val;
            }
            if (MODE & 2) {
                const float mean = sp.c1 * val + sp.c2 * v_xt[k];
                val = mean + sp.sigma_nz * v_nz[k];
                a.x_next[o] = val;
            }
            if (MODE != 1) tile[cc * LT + t] = val;      // tokens of the step that consumes this tensor
        }
    }
    if (MODE == 1) return;
    const bool emit = MODE == 4 || (a.emit_next && i_step > 0);
    if (emit) {
        __syncthreads();
        const int ncw = c1 - c0;
        for (int j = tid; j < T * ncw; j += 256) {
            const int t = j / ncw, cc = j % ncw;
            const size_t o = ((size_t)b * T + t) * a.Cp + c0 + cc;
            split_f16(cc < nc ? tile[cc * LT + t] : 0.f, a.xtok_b[o], a.xtok_s[o]);     // (hi, lo) fp16 pair; padding columns zero
        }
        if (add_early) {
#pragma unroll
            for (int k = 0; k < NA; k++) {
                const int i = part * per + tid + k * 256;
                if (i < q1) reinterpret_cast<float4*>(a.add + ((size_t)b * T + i / (D / 4)) * D)[i % (D / 4)] = add_pre[k];
            }
        } else {
            long long ti = MODE == 4 ? (a.tstep ? a.tstep[b] : a.tbl[*a.step_cur].t) : a.tbl[i_step - 1].t;
            if (ti < 0) ti = 0;
            if (ti >= a.pe_rows) ti = a.pe_rows - 1;
            const float4* trow = reinterpret_cast<const float4*>(a.tab + (size_t)ti * D);
            for (int i = part * per + tid; i < q1; i += 256) {
                const int tt = i / (D / 4), c = i % (D / 4);
                const float4 p4 = reinterpret_cast<const float4*>(a.pe + (size_t)tt * D)[c];
                const float4 o4 = trow[c];
                reinterpret_cast<float4*>(a.add + ((size_t)b * T + tt) * D)[c] = make_float4(o4.x + p4.x, o4.y + p4.y, o4.z + p4.z, o4.w + p4.w);
            }
        }
    }
    if ((MODE & 2) && a.emit_next && !early) {
        // (only when the step index comes from the device counter: with a host-known index nobody reads the counter until the
        // next loop's k_loop_begin sets it)  every thread of this block has read step_cur (before the first barrier-free use
        // above it sits in a register); the last block to get here moves the counter
        __syncthreads();
        if (tid == 0) {
            const int done = atomicAdd(a.ticket, 1);
            if (done == (int)(gridDim.x * gridDim.y) - 1) { *a.ticket = 0; *a.step_cur = i_step - 1; }
        }
    }
    if (c_chain) { __syncthreads(); if (tid == 0) chain_mark(6, 2); }
}

}  // namespace

CHAIN_SETTER(idb_chain_set_denoiser)

/* test / profiling hook: how many 8-CTA clusters of the fused decoder-layer kernel the device can hold at once */
extern "C" int idb_debug_max_layer_clusters(idb_handle* h) {
    IDB_ENTER(h);
    if (!h) return -1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(tc::mlp::CLUSTER, 64); cfg.blockDim = dim3(ANT); cfg.dynamicSmemBytes = tc::mlp::SMEM_BYTES;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = tc::mlp::CLUSTER; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = -1;
    if (cudaOccupancyMaxActiveClusters(&n, k_layer_qan_fused, &cfg) != cudaSuccess) { cudaGetLastError(); return -1; }
    return n;
}

extern "C" int idb_debug_attn_trace(long long* out16) {
    if (!out16) return IDB_ERR_ARG;
    return cudaMemcpyFromSymbol(out16, g_attn_trace, sizeof(long long) * 16) == cudaSuccess ? IDB_OK : IDB_ERR_CUDA;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------

int idb_pointnet_commit(idb_handle* h);
// six tensor maps of the feed-forward block (x hi/lo rows [M][256], w1 hi/lo [1024][256], w2 hi/lo [256][1024]); gemm_tcgen05.cu
int idb_mlp_make_maps(idb_handle* h, const __half* x_hi, const __half* x_lo, const __half* w1_hi, const __half* w1_lo, const __half* w2_hi,
                      const __half* w2_lo, int M, CUtensorMap* out6);
void idb_pointnet_release(idb_handle* h);

int idb_fail(idb_handle* h, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf;
    return code;
}

int idb_dev_alloc(idb_handle* h, float** p, size_t n) {
    CUDA_TRY(h, cudaMalloc((void**)p, (n ? n : 1) * sizeof(float)));
    return IDB_OK;
}
int idb_upload(idb_handle* h, float** p, const float* host, size_t n) {
    int rc = idb_dev_alloc(h, p, n);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpy(*p, host, n * sizeof(float), cudaMemcpyDefault));
    return IDB_OK;
}

static void denoiser_free_bound(Denoiser& d) {
    for (float* p : d.bound) cudaFree(p);
    d.bound.clear();
    for (void* p : d.bound_h) cudaFree(p);
    d.bound_h.clear();
    if (d.step_cur) { cudaFree(d.step_cur); d.step_cur = nullptr; d.ticket = nullptr; }
    d.B = d.T = d.M = 0;
}
void idb_sampler_drop_graphs(idb_handle* h);

void idb_denoiser_release(idb_handle* h) {
    Denoiser& d = h->den;
    idb_sampler_drop_graphs(h);      // captured step graphs hold the weight / workspace pointers freed below
    idb_pointnet_release(h);
    denoiser_free_bound(d);
    for (auto& kv : d.raw) cudaFree(kv.second.p);
    d.raw.clear();
    for (float* p : d.owned) cudaFree(p);
    d.owned.clear();
    d.layers.clear();
    d.enc_layers.clear();
    for (void* p : d.enc_owned) cudaFree(p);
    d.enc_owned.clear();
    d.enc_cap = 0;
    d.committed = false;
}

extern "C" int idb_denoiser_init(idb_handle* h, const idb_denoiser_config* cfg) {
    IDB_ENTER(h);
    if (!h || !cfg) return IDB_ERR_ARG;
    if (cfg->d_model != D) return idb_fail(h, IDB_ERR_ARG, "d_model must be 256 (got %d)", cfg->d_model);
    if (cfg->n_heads * 64 != cfg->d_model) return idb_fail(h, IDB_ERR_ARG, "head_dim must be 64");
    if (cfg->n_queries * 3 > 32) return idb_fail(h, IDB_ERR_ARG, "n_queries must be <= 10");
    if (cfg->d_ff % 4 || cfg->n_layers < 1 || cfg->n_layers > 32) return idb_fail(h, IDB_ERR_ARG, "bad d_ff / n_layers");
    if (cfg->variant == 1 && (cfg->c_obj != 3 * cfg->n_points || cfg->c_extra != 7))
        return idb_fail(h, IDB_ERR_ARG, "skeleton variant needs c_obj == 3*n_points and c_extra == 7");
    idb_denoiser_release(h);
    h->den.cfg = *cfg;
    h->den.configured = true;
    return IDB_OK;
}

extern "C" int idb_denoiser_load(idb_handle* h, const char* name, const float* data, const int64_t* shape, int ndim) {
    IDB_ENTER(h);
    if (!h || !name || !data) return IDB_ERR_ARG;
    Denoiser& d = h->den;
    if (!d.configured) return idb_fail(h, IDB_ERR_STATE, "idb_denoiser_init first");
    std::string s(name);
    // tensors of the sampling hot path and, when given, of the conditioning encoder (PointNet++ for SMPL, shapeEmbedding for
    // the skeleton model)
    bool want = s.rfind("decoder.layers.", 0) == 0 || s.rfind("encoder.layers.", 0) == 0 || s.rfind("pcEmbedding.", 0) == 0 ||
                s.rfind("shapeEmbedding.", 0) == 0 || s.rfind("bodyEmbedding.", 0) == 0 || s.rfind("objEmbedding.", 0) == 0 ||
                s.rfind("bodyFinalLinear.", 0) == 0 || s.rfind("objFinalLinear.", 0) == 0 ||
                s.rfind("embedTimeStep.time_embed.", 0) == 0 || s == "PositionalEmbedding.pe";
    if (!want || s.find("inv_freq") != std::string::npos) return IDB_OK;
    DevTensor t;
    t.shape.assign(shape, shape + ndim);
    auto it = d.raw.find(s);
    if (it != d.raw.end()) { cudaFree(it->second.p); d.raw.erase(it); }
    int rc = idb_upload(h, &t.p, data, t.numel());
    if (rc) return rc;
    d.raw[s] = t;
    d.committed = false;
    return IDB_OK;
}

namespace {
struct Packer {
    idb_handle* h;
    Denoiser& d;
    int rc = IDB_OK;
    const DevTensor* get(const std::string& n, std::initializer_list<int64_t> shape) {
        auto it = d.raw.find(n);
        if (it == d.raw.end()) { rc = idb_fail(h, IDB_ERR_STATE, "missing weight '%s'", n.c_str()); return nullptr; }
        std::vector<int64_t> want(shape);
        if (it->second.shape != want) {
            rc = idb_fail(h, IDB_ERR_STATE, "weight '%s' has the wrong shape", n.c_str());
            return nullptr;
        }
        return &it->second;
    }
    std::vector<float> host(const DevTensor* t) {
        std::vector<float> v(t->numel());
        cudaMemcpy(v.data(), t->p, v.size() * sizeof(float), cudaMemcpyDeviceToHost);
        return v;
    }
    float* up(const std::vector<float>& v) {
        float* p = nullptr;
        if (idb_upload(h, &p, v.data(), v.size())) { rc = IDB_ERR_CUDA; return nullptr; }
        d.owned.push_back(p);
        return p;
    }
};
}  // namespace

extern "C" int idb_denoiser_commit(idb_handle* h) {
    IDB_ENTER(h);
    if (!h) return IDB_ERR_ARG;
    Denoiser& d = h->den;
    if (!d.configured) return idb_fail(h, IDB_ERR_STATE, "idb_denoiser_init first");
    idb_sampler_drop_graphs(h);      // packed weights are (re)built below
    for (float* p : d.owned) cudaFree(p);
    d.owned.clear();
    d.layers.clear();
    const idb_denoiser_config& c = d.cfg;
    const int F = c.d_ff, N = c.n_queries, H = c.n_heads, HD = D / H;
    Packer P{h, d};
#define GET(var, name, ...) const DevTensor* var = P.get(name, {__VA_ARGS__}); if (!var) return P.rc;
    // input embedding: W_in^T [C][D] (zero rows for un-embedded channels), bias = b_body + b_obj
    {
        GET(wb, "bodyEmbedding.weight", D, c.c_body) GET(bb, "bodyEmbedding.bias", D)
        GET(wo, "objEmbedding.weight", D, c.c_obj) GET(bo, "objEmbedding.bias", D)
        const int C = c.c_body + c.c_obj + c.c_extra;
        auto hwb = P.host(wb), hbb = P.host(bb), hwo = P.host(wo), hbo = P.host(bo);
        std::vector<float> wT((size_t)C * D, 0.f), bsum(D);
        for (int n = 0; n < D; n++) {
            for (int k = 0; k < c.c_body; k++) wT[(size_t)k * D + n] = hwb[(size_t)n * c.c_body + k];
            for (int k = 0; k < c.c_obj; k++) wT[(size_t)(c.c_body + k) * D + n] = hwo[(size_t)n * c.c_obj + k];
            bsum[n] = hbb[n] + hbo[n];
        }
        d.w_inT = P.up(wT); d.b_in = P.up(bsum);
        const int Cp = (C + 3) & ~3;                      // row stride padded to 16 bytes for the GEMM
        std::vector<float> wcat((size_t)D * Cp, 0.f);    // [D][Cp]: [W_body | W_obj | 0]
        for (int n = 0; n < D; n++) {
            for (int k = 0; k < c.c_body; k++) wcat[(size_t)n * Cp + k] = hwb[(size_t)n * c.c_body + k];
            for (int k = 0; k < c.c_obj; k++) wcat[(size_t)n * Cp + c.c_body + k] = hwo[(size_t)n * c.c_obj + k];
        }
        d.w_in = P.up(wcat);
    }
    // output heads: [D][Clin] k-major; Clin = c_body + (variant 0 ? c_obj : 7)
    {
        const int c2 = c.variant == 0 ? c.c_obj : 7, Clin = c.c_body + c2;
        GET(wb, "bodyFinalLinear.weight", c.c_body, D) GET(bb, "bodyFinalLinear.bias", c.c_body)
        GET(wo, "objFinalLinear.weight", c2, D) GET(bo, "objFinalLinear.bias", c2)
        auto hwb = P.host(wb), hbb = P.host(bb), hwo = P.host(wo), hbo = P.host(bo);
        std::vector<float> wT((size_t)D * Clin), bcat(Clin);
        for (int n = 0; n < Clin; n++) {
            for (int k = 0; k < D; k++)
                wT[(size_t)k * Clin + n] = n < c.c_body ? hwb[(size_t)n * D + k] : hwo[(size_t)(n - c.c_body) * D + k];
            bcat[n] = n < c.c_body ? hbb[n] : hbo[n - c.c_body];
        }
        d.w_outT = P.up(wT); d.b_out = P.up(bcat);
        std::vector<float> wcat((size_t)Clin * D);        // [Clin][D]: [W_bodyFinal; W_objFinal]
        for (int n = 0; n < Clin; n++)
            for (int k = 0; k < D; k++) wcat[(size_t)n * D + k] = n < c.c_body ? hwb[(size_t)n * D + k] : hwo[(size_t)(n - c.c_body) * D + k];
        d.w_out = P.up(wcat);
    }
    // timestep MLP (k-major) + sinusoid table
    {
        GET(w0, "embedTimeStep.time_embed.0.weight", D, D) GET(b0, "embedTimeStep.time_embed.0.bias", D)
        GET(w2, "embedTimeStep.time_embed.2.weight", D, D) GET(b2, "embedTimeStep.time_embed.2.bias", D)
        auto tr = [&](const DevTensor* w) {
            auto hw = P.host(w);
            std::vector<float> t((size_t)D * D);
            for (int n = 0; n < D; n++) for (int k = 0; k < D; k++) t[(size_t)k * D + n] = hw[(size_t)n * D + k];
            return t;
        };
        d.te_w0T = P.up(tr(w0)); d.te_w2T = P.up(tr(w2));
        d.te_b0 = b0->p; d.te_b2 = b2->p;
        auto it = d.raw.find("PositionalEmbedding.pe");
        if (it == d.raw.end()) return idb_fail(h, IDB_ERR_STATE, "missing weight 'PositionalEmbedding.pe'");
        const DevTensor& pe = it->second;
        if (pe.shape.empty() || pe.shape.back() != D) return idb_fail(h, IDB_ERR_STATE, "pe has the wrong shape");
        d.pe = pe.p; d.pe_rows = (int)(pe.numel() / D);
        d.temb_tab = P.up(std::vector<float>((size_t)d.pe_rows * D, 0.f));
        k_temb_table<<<d.pe_rows, 256>>>(d.pe, d.te_w0T, d.te_b0, d.te_w2T, d.te_b2, d.b_in, d.temb_tab);
        LAUNCH_CHECK(h);
    }
    // one transformer layer of the decoder ("decoder.layers.") or of the conditioning encoder ("encoder.layers.": no
    // cross-attention block; its norm2 takes the place of the decoder's norm3 = the layer's final, "pending" norm)
    auto build_layer = [&](const std::string& stack, int l, bool is_dec, std::vector<DenoiserLayer>& dst) -> int {
        DenoiserLayer L;
        L.qan = (c.qan_mask >> l) & 1;
        const std::string p = stack + std::to_string(l) + ".";
        if (L.qan) {
            GET(q, p + "queries", N, D) GET(wk, p + "wk", N, 1)
            // fold: per-head unit norm (+1e-6), / sqrt(hd) (model/sublayers.py:18-35), * D^-0.5
            // (LocalAttention scale), rotate by o_s = q_pos - k_pos (rotary pairs (i, i+D/2))
            auto hq = P.host(q);
            std::vector<float> qt((size_t)3 * N * D);
            for (int n = 0; n < N; n++) {
                std::vector<double> qn(D);
                for (int hh = 0; hh < H; hh++) {
                    double nrm = 0;
                    for (int e = 0; e < HD; e++) { double v = hq[(size_t)n * D + hh * HD + e]; nrm += v * v; }
                    nrm = std::sqrt(nrm) + 1e-6;
                    for (int e = 0; e < HD; e++)
                        qn[hh * HD + e] = hq[(size_t)n * D + hh * HD + e] / nrm / std::sqrt((double)HD) * std::pow((double)D, -0.5);
                }
                for (int s = 0; s < 3; s++) {
                    const double o = c.rotary_offsets[s];
                    for (int i = 0; i < D / 2; i++) {
                        const double f = o * (double)(float)(1.0 / std::pow(10000.0, (double)(2 * i) / D));
                        const double cs = std::cos(f), sn = std::sin(f);
                        qt[((size_t)s * N + n) * D + i] = (float)(qn[i] * cs - qn[i + D / 2] * sn);
                        qt[((size_t)s * N + n) * D + i + D / 2] = (float)(qn[i + D / 2] * cs + qn[i] * sn);
                    }
                }
            }
            L.qt = P.up(qt); L.wk = wk->p;
        } else {
            GET(w, p + "self_attn.in_proj_weight", 3 * D, D) GET(b, p + "self_attn.in_proj_bias", 3 * D)
            GET(wo, p + "self_attn.out_proj.weight", D, D) GET(bo, p + "self_attn.out_proj.bias", D)
            L.w_qkv = w->p; L.b_qkv = b->p; L.w_o = wo->p; L.b_o = bo->p;
            // fold the out-projection into the value projection (exact algebra, float64 on the host):
            //   sum_j a_j (x_j Wv_h^T + bv_h) Wo_h^T = sum_j a_j x_j (Wo_h Wv_h)^T + Wo_h bv_h
            auto hw = P.host(w), hb = P.host(b), hwo = P.host(wo), hbo = P.host(bo);
            std::vector<float> wf((size_t)(2 * D + H * D) * D), bf((size_t)2 * D + H * D, 0.f), bof(D);
            std::copy(hw.begin(), hw.begin() + (size_t)2 * D * D, wf.begin());
            std::copy(hb.begin(), hb.begin() + 2 * D, bf.begin());
            for (int n = 0; n < D; n++) {
                double bacc = hbo[n];
                for (int hh = 0; hh < H; hh++) {
                    for (int k = 0; k < D; k++) {
                        double a = 0;
                        for (int e = 0; e < HD; e++) a += (double)hwo[(size_t)n * D + hh * HD + e] * hw[(size_t)(2 * D + hh * HD + e) * D + k];
                        wf[(size_t)(2 * D + hh * D + n) * D + k] = (float)a;
                    }
                    for (int e = 0; e < HD; e++) bacc += (double)hwo[(size_t)n * D + hh * HD + e] * hb[2 * D + hh * HD + e];
                }
                bof[n] = (float)bacc;
            }
            L.w_qkvf = P.up(wf); L.b_qkvf = P.up(bf); L.bo_f = P.up(bof);
        }
        if (is_dec) {
            GET(w, p + "multihead_attn.in_proj_weight", 3 * D, D) GET(b, p + "multihead_attn.in_proj_bias", 3 * D)
            GET(wo, p + "multihead_attn.out_proj.weight", D, D) GET(bo, p + "multihead_attn.out_proj.bias", D)
            L.w_qc = w->p; L.b_qc = b->p; L.w_kvc = w->p + (size_t)D * D; L.b_kvc = b->p + D; L.w_oc = wo->p; L.b_oc = bo->p;
            {   // Wq^T [k][h*64+d], for folding the query projection into the memory keys at bind time
                auto hwq = P.host(w);
                std::vector<float> wT((size_t)D * D);
                for (int o = 0; o < D; o++) for (int k = 0; k < D; k++) wT[(size_t)k * D + o] = hwq[(size_t)o * D + k];
                L.w_qcT = P.up(wT);
            }
        }
        {
            GET(w1, p + "linear1.weight", F, D) GET(b1, p + "linear1.bias", F)
            GET(w2, p + "linear2.weight", D, F) GET(b2, p + "linear2.bias", D)
            L.w1 = w1->p; L.b1 = b1->p; L.w2 = w2->p; L.b2 = b2->p;
            GET(n1w, p + "norm1.weight", D) GET(n1b, p + "norm1.bias", D) GET(n2w, p + "norm2.weight", D) GET(n2b, p + "norm2.bias", D)
            L.ln1w = n1w->p; L.ln1b = n1b->p;
            if (is_dec) {
                GET(n3w, p + "norm3.weight", D) GET(n3b, p + "norm3.bias", D)
                L.ln2w = n2w->p; L.ln2b = n2b->p; L.ln3w = n3w->p; L.ln3b = n3b->p;
            } else {
                L.ln3w = n2w->p; L.ln3b = n2b->p;
            }
        }
        dst.push_back(L);
        return IDB_OK;
    };
    for (int l = 0; l < c.n_layers; l++) {
        const int rc = build_layer("decoder.layers.", l, true, d.layers);
        if (rc) return rc;
    }
    // conditioning encoder (optional: present when its tensors were loaded; SURVEY 8f rank 1)
    d.enc_layers.clear();
    d.w_shapeT = d.b_shape = nullptr;
    if (d.raw.count("encoder.layers.0.linear1.weight")) {
        for (int l = 0; l < c.n_layers; l++) {
            const int rc = build_layer("encoder.layers.", l, false, d.enc_layers);
            if (rc) return rc;
        }
        if (c.variant == 1) {
            // skeleton: the object-shape embedding of the canonical keypoints (model/diffusion_skeleton.py:203), k-major
            GET(ws, "shapeEmbedding.weight", D, c.c_obj) GET(bs, "shapeEmbedding.bias", D)
            auto hws = P.host(ws);
            std::vector<float> wT((size_t)c.c_obj * D);
            for (int n = 0; n < D; n++) for (int k = 0; k < c.c_obj; k++) wT[(size_t)k * D + n] = hws[(size_t)n * c.c_obj + k];
            d.w_shapeT = P.up(wT); d.b_shape = bs->p;
        }
    }
#undef GET
    if (P.rc) return P.rc;
    // fp16 (hi, lo) copies of every GEMM weight for the tensor-core path
    {
        auto split = [&](const float* w, int rows, int cols, int ld_dst, __half** hi, __half** lo) -> int {
            const size_t n = (size_t)rows * ld_dst;
            CUDA_TRY(h, cudaMalloc((void**)hi, n * sizeof(__half)));
            d.owned.push_back(reinterpret_cast<float*>(*hi));
            CUDA_TRY(h, cudaMalloc((void**)lo, n * sizeof(__half)));
            d.owned.push_back(reinterpret_cast<float*>(*lo));
            return idb_split_tensor(h, w, cols, *hi, *lo, ld_dst, rows, cols, 0);
        };
        const int C = c.c_body + c.c_obj + c.c_extra, Cp = (C + 3) & ~3, Cp8 = (C + 7) & ~7;
        const int Clin = c.c_body + (c.variant == 0 ? c.c_obj : 7);
        (void)Cp;
        int rc = split(d.w_in, D, (C + 3) & ~3, Cp8, &d.w_in_b, &d.w_in_s);
        if (!rc) rc = split(d.w_out, Clin, D, D, &d.w_out_b, &d.w_out_s);
        for (auto* stack : {&d.layers, &d.enc_layers})
            for (auto& L : *stack) {
                if (!rc && !L.qan) rc = split(L.w_qkvf, 2 * D + H * D, D, D, &L.w_qkvf_b, &L.w_qkvf_s);
                if (!rc && L.qan) {
                    // folded queries as fp16 (hi, lo), rows padded to the stride the kernels keep in shared memory: one block
                    __half *qb = nullptr, *qs = nullptr;
                    rc = split(L.qt, 3 * N, D, D, &qb, &qs);
                    if (!rc) {
                        CUDA_TRY(h, cudaDeviceSynchronize());      // the split kernels ran on the handle's stream
                        const size_t half_bytes = (size_t)3 * N * KPH * sizeof(__half);
                        CUDA_TRY(h, cudaMalloc((void**)&L.qt_pack, 2 * half_bytes));
                        d.owned.push_back(reinterpret_cast<float*>(L.qt_pack));
                        CUDA_TRY(h, cudaMemset(L.qt_pack, 0, 2 * half_bytes));
                        CUDA_TRY(h, cudaMemcpy2D(L.qt_pack, KPH * sizeof(__half), qb, D * sizeof(__half), D * sizeof(__half), 3 * N, cudaMemcpyDeviceToDevice));
                        CUDA_TRY(h, cudaMemcpy2D(reinterpret_cast<uint8_t*>(L.qt_pack) + half_bytes, KPH * sizeof(__half), qs, D * sizeof(__half),
                                                 D * sizeof(__half), 3 * N, cudaMemcpyDeviceToDevice));
                    }
                }
                if (!rc) rc = split(L.w1, F, D, D, &L.w1_b, &L.w1_s);
                if (!rc) rc = split(L.w2, D, F, F, &L.w2_b, &L.w2_s);
            }
        if (rc) return rc;
        CUDA_TRY(h, cudaDeviceSynchronize());
    }
    {
        const int rc = idb_pointnet_commit(h);      // optional PointNet++ point-cloud encoder (pointnet.cu)
        if (rc) return rc;
    }
    d.committed = true;
    denoiser_free_bound(d);
    return IDB_OK;
}

extern "C" int idb_denoiser_bind(idb_handle* h, int B, int T, int Tm, const float* cond, const float* zero_pose_obj, void* stream) {
    IDB_ENTER(h);
    if (!h || !cond || B <= 0 || T <= 0 || Tm <= 0) return IDB_ERR_ARG;
    Denoiser& d = h->den;
    if (!d.committed) return idb_fail(h, IDB_ERR_STATE, "idb_denoiser_commit first");
    if (T > d.pe_rows) return idb_fail(h, IDB_ERR_ARG, "T exceeds the positional table");
    if (T > 36 || Tm > 16) return idb_fail(h, IDB_ERR_ARG, "supported window: T <= 36 frames (reference default 35), <= 16 memory tokens");
    if (d.cfg.variant == 1 && !zero_pose_obj) return idb_fail(h, IDB_ERR_ARG, "skeleton variant needs zero_pose_obj");
    cudaStream_t st = (cudaStream_t)stream;
    const idb_denoiser_config& c = d.cfg;
    const int M = B * T, F = c.d_ff, H = c.n_heads, C = c.c_body + c.c_obj + c.c_extra;
    const int Clin = c.c_body + (c.variant == 0 ? c.c_obj : 7);
    const int npts = c.n_points > 0 ? c.n_points : 1;
    if (B != d.B || T != d.T || Tm != d.Tm) {
        idb_sampler_drop_graphs(h);  // the workspaces below are baked into the captured graphs
        denoiser_free_bound(d);
        auto A = [&](float** p, size_t n) { int rc = idb_dev_alloc(h, p, n); if (!rc) d.bound.push_back(*p); return rc; };
        int rc = 0;
        rc |= A(&d.cond, (size_t)Tm * B * D); rc |= A(&d.h, (size_t)M * D); rc |= A(&d.h2, (size_t)M * D);
        rc |= A(&d.qkv, (size_t)M * (2 * D + H * D)); rc |= A(&d.qc, (size_t)M * D);
        rc |= A(&d.z, (size_t)M * D); rc |= A(&d.addend, (size_t)M * D);
        rc |= A(&d.lin, (size_t)M * Clin); rc |= A(&d.att, (size_t)Tm * B * D);
        auto AH = [&](__half** p, size_t n) {
            cudaError_t e = cudaMalloc((void**)p, n * sizeof(__half) + 16);
            if (e == cudaSuccess) d.bound_h.push_back(*p);
            return e == cudaSuccess ? 0 : idb_fail(h, IDB_ERR_CUDA, "cudaMalloc failed: %s", cudaGetErrorString(e));
        };
        const size_t Cp8 = (size_t)((C + 7) & ~7);
        rc |= AH(&d.h_b, (size_t)M * D); rc |= AH(&d.h_s, (size_t)M * D); rc |= AH(&d.h2_b, (size_t)M * D); rc |= AH(&d.h2_s, (size_t)M * D);
        rc |= AH(&d.ff_b, (size_t)M * F); rc |= AH(&d.ff_s, (size_t)M * F); rc |= AH(&d.xtok_b, (size_t)M * Cp8); rc |= AH(&d.xtok_s, (size_t)M * Cp8);
        rc |= A(&d.zero_pose, (size_t)B * npts * 3);
        for (auto& L : d.layers) {
            rc |= A(&L.kv_mem, (size_t)Tm * B * 2 * D); rc |= A(&L.vp_mem, (size_t)Tm * B * H * D);
            rc |= A(&L.kp_mem, (size_t)Tm * B * H * D); rc |= A(&L.kc_mem, (size_t)Tm * B * H);
            rc |= AH(&L.mem_pack, (size_t)B * mem_block_bytes(H * Tm) / sizeof(__half));
            if (!rc) cudaMemsetAsync(L.mem_pack, 0, (size_t)B * mem_block_bytes(H * Tm), st);      // pad columns
        }
        if (rc) return rc;
        CUDA_TRY(h, cudaMalloc((void**)&d.step_cur, 2 * sizeof(int)));
        CUDA_TRY(h, cudaMemset(d.step_cur, 0, 2 * sizeof(int)));
        d.ticket = d.step_cur + 1;
        d.B = B; d.T = T; d.M = M; d.Tm = Tm;
    }
    CUDA_TRY(h, cudaMemcpyAsync(d.cond, cond, sizeof(float) * (size_t)Tm * B * D, cudaMemcpyDefault, st));
    if (zero_pose_obj && c.n_points > 0)
        CUDA_TRY(h, cudaMemcpyAsync(d.zero_pose, zero_pose_obj, sizeof(float) * (size_t)B * c.n_points * 3, cudaMemcpyDefault, st));
    // Step-invariant cross-attention tensors of the memory (rows j*B + b, seq-first like the reference):
    //   kv_mem = mem [Wk;Wv]^T + b ;  vp_mem[:, h*D:(h+1)*D] = V_h Wo_h^T  (out-projection folded in)
    for (auto& L : d.layers) {
        int rc = idb_gemm(h, d.cond, D, L.w_kvc, D, L.b_kvc, nullptr, 0, L.kv_mem, 2 * D, Tm * B, 2 * D, D, EPI_BIAS, st);
        if (rc) return rc;
        for (int hh = 0; hh < H; hh++) {
            rc = idb_gemm(h, L.kv_mem + D + hh * HD, 2 * D, L.w_oc + hh * HD, D, nullptr, nullptr, 0, L.vp_mem + hh * D, H * D,
                          Tm * B, D, HD, 0, st);
            if (rc) return rc;
            // kp[:, h*D + k] = sum_d K[:, h*64+d] Wq[h*64+d][k]   (scaled by 1/sqrt(hd) in k_fold_scale)
            rc = idb_gemm(h, L.kv_mem + hh * HD, 2 * D, L.w_qcT + hh * HD, D, nullptr, nullptr, 0, L.kp_mem + hh * D, H * D,
                          Tm * B, D, HD, 0, st);
            if (rc) return rc;
        }
        k_fold_scale<<<(Tm * B * H + 7) / 8, 256, 0, st>>>(L.kp_mem, L.kv_mem, L.b_qc, L.kc_mem, Tm * B, H);
        LAUNCH_CHECK(h);
        k_pack_memory<<<dim3(H * Tm, B), D, 0, st>>>(L.kp_mem, L.vp_mem, L.kc_mem, reinterpret_cast<uint8_t*>(L.mem_pack), B, Tm, H);
        LAUNCH_CHECK(h);
    }
    return IDB_OK;
}

static size_t attn_smem(int Tk, int H) {   // barriers, 3 parameter rows, s_q, s_z, s_v, s_k (reused for the probabilities)
    const size_t HT = (size_t)H * Tk, HT16 = (HT + 15) & ~(size_t)15, pld = ((HT16 + 23) / 32) * 32 + 8;
    const size_t kreg = HT * (HD + 8) > SLAB * pld ? HT * (HD + 8) : SLAB * pld;
    return sizeof(float) * (4 + 3 * D + (size_t)SLAB * (D + 8) + (size_t)SLAB * LDZ + HT * (D + 4) + kreg);
}
static size_t xattn_tail_smem(int Tk, int H) {   // s_x1, s_kp, s_v, s_a, s_z, s_kc
    const size_t HT = (size_t)H * Tk;
    // s_x1, keys fp16 hi+lo [HT][264] (= HT*264 words), value k-pair words hi+lo [HT/2][264] (= HT*264 words), s_p, s_z, s_kc
    return sizeof(float) * ((size_t)SLAB * (D + 8) + HT * (D + 8) + HT * (D + 8) + (size_t)SLAB * 72 + (size_t)SLAB * LDZ + HT + 4);
}
static size_t xattn_smem(int Tk, int H) { return sizeof(float) * (4 + 3 * D) + xattn_tail_smem(Tk, H); }
static size_t qan_enc_smem() {      // encoder variant: barriers, parameter rows, s_x, s_qt, s_z
    return sizeof(float) * (4 + 7 * D + (size_t)(SLAB + 2) * (D + 8) + 30 * (D + 8) + (size_t)SLAB * LDZ + 4);
}
static size_t qan_smem(int Tk, int H) {      // barriers, 7 parameter rows, s_x, s_qt + the cross-attention buffers
    return sizeof(float) * (4 + 7 * D + (size_t)(SLAB + 2) * (D + 8) + 30 * (D + 8)) + xattn_tail_smem(Tk, H);
}

// One nn.Linear on fp16 (hi, lo) operand pairs; output as full fp32 and/or as a pair.
static int linear(idb_handle* h, const __half* a_b, const __half* a_s, int lda, const __half* w_b, const __half* w_s, int ldw,
                  const float* bias, const float* res, float* C, __half* C_b, __half* C_s, int ldc, int M, int N, int K, int epi,
                  cudaStream_t st, int ksplit = 1, float* zero = nullptr) {
    GemmArgs g;
    g.ksplit = ksplit; g.zero = zero; g.zero_ld = D; g.zero_cols = D;
    g.A_hi = a_b; g.A_lo = a_s; g.lda = lda; g.W_hi = w_b; g.W_lo = w_s; g.ldw = ldw; g.bias = bias; g.res = res; g.ldr = D;
    g.C = C; g.C_hi = C_b; g.C_lo = C_s; g.ldc = ldc; g.M = M; g.N = N; g.K = K; g.epi = epi;
    g.pdl = h->pdl;   // weights are step-invariant: their tiles may be fetched before the dependency wait
    return idb_gemm_ex(h, g, st);
}

// Decoder body on the bound workspaces.  Activation triples (full, big, small): d.h/h_b/h_s hold the
// embedded tokens on entry; on exit d.h (+ split) holds the decoder output (last norm3 applied).
static int denoiser_layers(idb_handle* h, cudaStream_t st) {
    Denoiser& d = h->den;
    const int B = d.B, T = d.T, M = d.M, Tm = d.Tm, F = d.cfg.d_ff, H = d.cfg.n_heads, N = d.cfg.n_queries;
    const dim3 slab_grid(B, (T + SLAB - 1) / SLAB);
    const int ln_blocks = (M * 32 + 255) / 256;
    const DenoiserLayer* pending = nullptr;   // layer whose norm3 has not been applied to d.z yet (unfused feed-forward path)
    const bool pdl = h->pdl != 0;
    const bool fused = h->gemm_backend == 1 && h->fused_mlp && idb_mlp_tcgen05_supported(D, F);
    int rc;
    for (auto& L : d.layers) {
        // ---- first sub-block -> x1 = (d.h2, h2_b, h2_s)
        if (L.qan) {
            QanArgs qa = {};
            qa.zin = pending ? d.z : d.h; qa.prew = pending ? pending->ln3w : nullptr; qa.preb = pending ? pending->ln3b : nullptr;
            qa.qpack = L.qt_pack; qa.wk = L.wk; qa.lnw = L.ln1w; qa.lnb = L.ln1b; qa.mpack = reinterpret_cast<const uint8_t*>(L.mem_pack);
            qa.bo2 = L.b_oc; qa.ln2w = L.ln2w; qa.ln2b = L.ln2b; qa.out = d.h2; qa.out_b = d.h2_b; qa.out_s = d.h2_s;
            qa.T = T; qa.N = N; qa.B = B; qa.Tk = Tm; qa.H = H;
            if (fused && h->fused_mlp >= 3 && !pending && qan_smem(Tm, H) <= (size_t)(tc::mlp::RING + tc::mlp::S_BYTES)) {
                // the whole layer in one cluster kernel (attention phase + feed-forward phase on sample-aligned row tiles)
                const int nslabs = (T + SLAB - 1) / SLAB, G = tc::mlp::CLUSTER / nslabs;
                CUtensorMap mp[6];
                if ((rc = idb_mlp_make_maps(h, d.h2_b, d.h2_s, L.w1_b, L.w1_s, L.w2_b, L.w2_s, M, mp))) return rc;
                idb_launch(pdl, k_layer_qan_fused, dim3(tc::mlp::CLUSTER, (B + G - 1) / G), ANT, (size_t)tc::mlp::SMEM_BYTES, st, qa,
                           mp[0], mp[1], mp[2], mp[3], mp[4], mp[5], (const float*)L.b1, (const float*)L.b2, (const float*)d.h2, d.h,
                           (const float*)L.ln3w, (const float*)L.ln3b, d.h_b, d.h_s, M, G, nslabs);
                LAUNCH_CHECK(h);
                continue;
            }
            // QaN block + LN1 + cross-attention + LN2 in one kernel: (z | h) -> (d.h2, pairs)
            if (pending) idb_launch(pdl, k_qan_xattn_ln<true, true>, slab_grid, ANT, qan_smem(Tm, H), st, qa);
            else idb_launch(pdl, k_qan_xattn_ln<true, false>, slab_grid, ANT, qan_smem(Tm, H), st, qa);
            LAUNCH_CHECK(h);
        } else {
            if (pending) {
                idb_launch(pdl, k_ln, ln_blocks, 256, 0, st, d.z, pending->ln3w, pending->ln3b, d.h, d.h_b, d.h_s, M);
                LAUNCH_CHECK(h);
            }
            const int NQ = 2 * D + H * D;
            if ((rc = linear(h, d.h_b, d.h_s, D, L.w_qkvf_b, L.w_qkvf_s, D, L.b_qkvf, nullptr, d.qkv, nullptr, nullptr, NQ, M, NQ, D,
                             EPI_BIAS, st))) return rc;
            AttnArgs aa = {};
            aa.q = d.qkv; aa.ldq = NQ; aa.k = d.qkv + D; aa.ldk = NQ; aa.v = d.qkv + 2 * D; aa.ldv = NQ; aa.res = d.h; aa.bo = L.bo_f;
            aa.lnw = L.ln1w; aa.lnb = L.ln1b; aa.out = d.qc; aa.T = T; aa.H = H;
            XattnArgs xa = {};
            xa.x1 = d.qc; xa.mpack = reinterpret_cast<const uint8_t*>(L.mem_pack); xa.bo = L.b_oc;
            xa.lnw = L.ln2w; xa.lnb = L.ln2b; xa.out = d.h2; xa.out_b = d.h2_b; xa.out_s = d.h2_s; xa.T = T; xa.B = B; xa.Tk = Tm; xa.H = H;
            if (fused && h->fused_mlp >= 3 && attn_smem(T, H) <= (size_t)(tc::mlp::RING + tc::mlp::S_BYTES) &&
                xattn_smem(Tm, H) <= (size_t)(tc::mlp::RING + tc::mlp::S_BYTES)) {
                // self-attention + cross-attention + feed-forward of the layer in one cluster kernel
                const int nslabs = (T + SLAB - 1) / SLAB, G = tc::mlp::CLUSTER / nslabs;
                CUtensorMap mp[6];
                if ((rc = idb_mlp_make_maps(h, d.h2_b, d.h2_s, L.w1_b, L.w1_s, L.w2_b, L.w2_s, M, mp))) return rc;
                idb_launch(pdl, k_layer_std_fused, dim3(tc::mlp::CLUSTER, (B + G - 1) / G), ANT, (size_t)tc::mlp::SMEM_BYTES, st, aa, xa,
                           mp[0], mp[1], mp[2], mp[3], mp[4], mp[5], (const float*)L.b1, (const float*)L.b2, (const float*)d.h2, d.h,
                           (const float*)L.ln3w, (const float*)L.ln3b, d.h_b, d.h_s, M, G, nslabs);
                LAUNCH_CHECK(h);
                continue;
            }
            if (h->fuse_attn) {
                // self-attention + LN1 and cross-attention + LN2 in one launch: h -> (d.qc) -> (d.h2, pairs)
                const size_t smem = attn_smem(T, H) > xattn_smem(Tm, H) ? attn_smem(T, H) : xattn_smem(Tm, H);
                idb_launch(pdl, k_attn_xattn_ln, slab_grid, ANT, smem, st, aa, xa);
                LAUNCH_CHECK(h);
            } else {
                idb_launch(pdl, k_attn_ln, slab_grid, ANT, attn_smem(T, H), st, aa);
                LAUNCH_CHECK(h);
                // cross attention on the LN1 rows (d.qc) -> (d.h2, pairs)
                idb_launch(pdl, k_xattn_ln, slab_grid, ANT, xattn_smem(Tm, H), st, xa);
                LAUNCH_CHECK(h);
            }
        }
        // ---- feed forward on x2 = d.h2: ff = gelu(x2 W1^T + b1) kept as pairs only; z = ff W2^T + b2 + x2  (pre-norm3)
        if (fused) {
            // both GEMMs, GELU, the residual AND the layer's norm3 in one cluster kernel: the hidden activations never
            // leave the SM and the next layer starts from normalised rows (fp32 + fp16 pairs)
            if (h->fused_mlp >= 2) {
                if ((rc = idb_mlp_tcgen05(h, d.h2_b, d.h2_s, L.w1_b, L.w1_s, L.b1, L.w2_b, L.w2_s, L.b2, d.h2, D, d.h, D, M, h->pdl, st,
                                          L.ln3w, L.ln3b, d.h_b, d.h_s)))
                    return rc;
                continue;
            }
            if ((rc = idb_mlp_tcgen05(h, d.h2_b, d.h2_s, L.w1_b, L.w1_s, L.b1, L.w2_b, L.w2_s, L.b2, d.h2, D, d.z, D, M, h->pdl, st)))
                return rc;
        } else {
            // ff1 also clears d.z (dead here) so that ff2 can run split-K = 2 and fill 120 SMs instead of 60
            if ((rc = linear(h, d.h2_b, d.h2_s, D, L.w1_b, L.w1_s, D, L.b1, nullptr, nullptr, d.ff_b, d.ff_s, F, M, F, D, EPI_BIAS | EPI_GELU, st,
                             1, d.z)))
                return rc;
            if ((rc = linear(h, d.ff_b, d.ff_s, F, L.w2_b, L.w2_s, F, L.b2, d.h2, d.z, nullptr, nullptr, D, M, D, F, EPI_BIAS | EPI_RES, st, 2)))
                return rc;
        }
        // QaN layers return tgt + (x - tgt) (model/sublayers.py:338-339); that differs from x by
        // <= 1 ulp of max(|x|,|tgt|) and is not reproduced (DESIGN.md "Deviations").
        pending = &L;
    }
    if (pending) {
        idb_launch(pdl, k_ln, ln_blocks, 256, 0, st, d.z, pending->ln3w, pending->ln3b, d.h, d.h_b, d.h_s, M);
        LAUNCH_CHECK(h);
    }
    return IDB_OK;
}

static constexpr int STEP_IO_PARTS = 4;

static StepIO step_io_base(idb_handle* h) {
    Denoiser& d = h->den;
    const idb_denoiser_config& c = d.cfg;
    StepIO a = {};
    a.i_host = -1;
    a.lin = d.lin; a.zero_pose = d.zero_pose;
    a.tbl = h->diff.tbl; a.step_cur = d.step_cur; a.ticket = d.ticket; a.n_steps = h->diff.n;
    a.xtok_b = d.xtok_b; a.xtok_s = d.xtok_s; a.tab = d.temb_tab; a.pe = d.pe; a.add = d.addend; a.pe_rows = d.pe_rows;
    a.T = d.T; a.C = c.c_body + c.c_obj + c.c_extra; a.Cp = (a.C + 7) & ~7;
    a.Clin = c.c_body + (c.variant == 0 ? c.c_obj : 7);
    a.variant = c.variant; a.c_body = c.c_body; a.n_points = c.n_points;
    return a;
}

template <int MODE>
static int launch_step_io(idb_handle* h, const StepIO& a, cudaStream_t st) {
    const int ncp = (a.Cp + STEP_IO_PARTS - 1) / STEP_IO_PARTS;
    const size_t smem = sizeof(float) * ((size_t)ncp * (a.T + 1) + (size_t)a.T * 8);
    idb_launch(h->pdl != 0, k_step_io<MODE>, dim3(h->den.B, STEP_IO_PARTS), 256, smem, st, a);
    LAUNCH_CHECK(h);
    return IDB_OK;
}

// x (B,1,C,T) -> token pairs + embedding addend.  tstep: device timesteps (B), or null = the sampler's
// current step (tbl[step_cur].t).
int idb_denoiser_tokens(idb_handle* h, const float* x, const long long* tstep, cudaStream_t st) {
    if (!h->den.B) return idb_fail(h, IDB_ERR_STATE, "idb_denoiser_bind first");
    if (!tstep && !h->diff.tbl) return idb_fail(h, IDB_ERR_STATE, "idb_diffusion_init first");
    StepIO a = step_io_base(h);
    a.x_in = x; a.tstep = tstep;
    return launch_step_io<4>(h, a, st);
}

// decoder on the prepared tokens: input embedding, 8 layers, output heads -> d.lin [B*T][Clin]
int idb_denoiser_body(idb_handle* h, cudaStream_t st) {
    Denoiser& d = h->den;
    const idb_denoiser_config& c = d.cfg;
    const int M = d.M, C = c.c_body + c.c_obj + c.c_extra, Cp = (C + 7) & ~7;
    const int Clin = c.c_body + (c.variant == 0 ? c.c_obj : 7);
    int rc;
    // input embedding (model/diffusion_smpl.py:227-232): h = xtok W_in^T + (b_in + temb + pe)
    if ((rc = linear(h, d.xtok_b, d.xtok_s, Cp, d.w_in_b, d.w_in_s, Cp, nullptr, d.addend, d.h, d.h_b, d.h_s, D, M, D, Cp, EPI_RES, st)))
        return rc;
    if ((rc = denoiser_layers(h, st))) return rc;
    // output heads (model/diffusion_smpl.py:234-237)
    return linear(h, d.h_b, d.h_s, D, d.w_out_b, d.w_out_s, D, d.b_out, nullptr, d.lin, nullptr, nullptr, Clin, M, Clin, D, EPI_BIAS, st);
}

// d.lin -> x0 (B,1,C,T) with the optional inpainting blend
int idb_denoiser_heads(idb_handle* h, const float* gt, const unsigned char* mask, float* out, cudaStream_t st) {
    StepIO a = step_io_base(h);
    a.gt = gt; a.mask = mask; a.x0_out = out;
    return launch_step_io<1>(h, a, st);
}

// posterior sample from a given x0 (after the correction hook, or the stand-alone finish call)
int idb_step_finish(idb_handle* h, const float* x0, const float* xt, const float* noise, int tape_mode, float* x_next, int emit_next,
                    cudaStream_t st, int i_host) {
    StepIO a = step_io_base(h);
    a.i_host = i_host;
    a.x0_in = x0; a.xt = xt; a.noise = noise; a.tape_mode = tape_mode; a.x_next = x_next; a.emit_next = emit_next;
    return launch_step_io<2>(h, a, st);
}

// heads + posterior sample + next step's tokens in one kernel (the tail of a plain sampling step)
int idb_step_tail(idb_handle* h, const float* gt, const unsigned char* mask, float* x0_out, const float* xt, const float* noise,
                  int tape_mode, float* x_next, int emit_next, cudaStream_t st, int i_host) {
    StepIO a = step_io_base(h);
    a.i_host = i_host;
    a.gt = gt; a.mask = mask; a.x0_out = x0_out;
    a.xt = xt; a.noise = noise; a.tape_mode = tape_mode; a.x_next = x_next; a.emit_next = emit_next;
    return launch_step_io<3>(h, a, st);
}

// x (B,1,C,T) -> x0 prediction (B,1,C,T); optional inpainting blend
int idb_denoiser_run(idb_handle* h, const float* x, const long long* tstep, const float* gt, const unsigned char* mask,
                     float* out, cudaStream_t st) {
    int rc;
    if ((rc = idb_denoiser_tokens(h, x, tstep, st))) return rc;
    if ((rc = idb_denoiser_body(h, st))) return rc;
    return idb_denoiser_heads(h, gt, mask, out, st);
}

int idb_denoiser_prepare_kernels(idb_handle* h) {
    // opt in to > 48 KB dynamic shared memory once (T <= 36, Tm <= 16 supported: the self-attention slab kernel keeps all folded values of a sample, 4*T*256 floats, in shared memory)
    CUDA_TRY(h, cudaFuncSetAttribute(k_qan_xattn_ln<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qan_smem(16, 4)));
    CUDA_TRY(h, cudaFuncSetAttribute(k_qan_xattn_ln<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qan_smem(16, 4)));
    CUDA_TRY(h, cudaFuncSetAttribute(k_layer_qan_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::mlp::SMEM_BYTES));
    CUDA_TRY(h, cudaFuncSetAttribute(k_layer_std_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::mlp::SMEM_BYTES));
    CUDA_TRY(h, cudaFuncSetAttribute(k_qan_xattn_ln<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)qan_enc_smem()));
    CUDA_TRY(h, cudaFuncSetAttribute(k_xattn_ln, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)xattn_smem(16, 4)));
    CUDA_TRY(h, cudaFuncSetAttribute(k_attn_ln, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)attn_smem(36, 4)));
    CUDA_TRY(h, cudaFuncSetAttribute(k_attn_xattn_ln, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     (int)(attn_smem(36, 4) > xattn_smem(16, 4) ? attn_smem(36, 4) : xattn_smem(16, 4))));
    return IDB_OK;
}

// ---------------------------------------------------------------------------------------------
// Conditioning encoder (SURVEY 8f rank 1, the part of MDM._get_embeddings after the point-cloud encoder,
// model/diffusion_smpl.py:217-221): cond = encoder(PositionalEmbedding(bodyEmbedding(past body) +
// objEmbedding(past obj) + pc_embedding)); for the skeleton model (model/diffusion_skeleton.py:194-215) the
// point-cloud term is shapeEmbedding(zero_pose_obj).  Runs once per batch before idb_denoiser_bind; the layers reuse the
// decoder's kernels (folded-QKV GEMM + k_attn_ln, the QaN kernel without its cross-attention half, the fused
// feed-forward kernel or, for d_ff != 1024, two GEMMs), rows m = b*Tp + t.  Only the token kernels differ per variant.
namespace {

// past (B,1,C,Tp) -> token pairs [B*Tp][Cp] (zero padded) + addend[b*Tp+t][:] = (pc[b] + b_body + b_obj) + pe[t]
__global__ void k_cond_tokens(const float* __restrict__ past, const float* __restrict__ pc, const float* __restrict__ b_in,
                              const float* __restrict__ pe, __half* __restrict__ xtok_b, __half* __restrict__ xtok_s,
                              float* __restrict__ add, int C, int Cp, int Tp) {
    const int b = blockIdx.x;
    for (int i = threadIdx.x; i < Tp * Cp; i += blockDim.x) {
        const int t = i / Cp, c = i % Cp;
        const size_t o = ((size_t)b * Tp + t) * Cp + c;
        split_f16(c < C ? past[((size_t)b * C + c) * Tp + t] : 0.f, xtok_b[o], xtok_s[o]);
    }
    for (int i = threadIdx.x; i < Tp * (D / 4); i += blockDim.x) {
        const int t = i / (D / 4), c4 = i % (D / 4);
        const float4 p = reinterpret_cast<const float4*>(pc + (size_t)b * D)[c4], bi = reinterpret_cast<const float4*>(b_in)[c4];
        const float4 q = reinterpret_cast<const float4*>(pe + (size_t)t * D)[c4];
        reinterpret_cast<float4*>(add + ((size_t)b * Tp + t) * D)[c4] =
            make_float4((p.x + bi.x) + q.x, (p.y + bi.y) + q.y, (p.z + bi.z) + q.z, (p.w + bi.w) + q.w);
    }
}

// LayerNorm of token rows m = b*Tp + t, written in the reference's sequence-first layout out[(t*B + b)][:]
__global__ void k_ln_seq_first(const float* __restrict__ a, const float* __restrict__ w, const float* __restrict__ bb,
                               float* __restrict__ out, int B, int Tp) {
    const int m = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    pdl_trigger();
    pdl_wait();
    if (m >= B * Tp) return;
    const int b = m / Tp, t = m - b * Tp;
    if (w) {
        warp_ln_row(a + (size_t)m * D, w, bb, out + ((size_t)t * B + b) * D, lane);
    } else {
        const float4* src = reinterpret_cast<const float4*>(a + (size_t)m * D);
        float4* dst = reinterpret_cast<float4*>(out + ((size_t)t * B + b) * D);
        dst[lane] = src[lane]; dst[lane + 32] = src[lane + 32];
    }
}

// skeleton variant (model/diffusion_skeleton.py:194-215): past (B,1,C,Tp) with C = 3 n_joints + 3 n_points + 7 -> token pairs
// [B*Tp][Cp] (zero padded; W_in has zero rows for the 7 pose channels, so the whole past slice is fed as it is) and
// addend[b*Tp+t][:] = (shape[b] + b_body + b_obj) + pe[t], shape[b] = shapeEmbedding(zero_pose_obj[b]) = Ws zp[b] + bs
// (K = 3 n_points fp32 terms per output, ascending k).  grid B, block D, dynamic shared memory K floats.
__global__ void __launch_bounds__(D)
k_skel_cond_tokens(const float* __restrict__ past, const float* __restrict__ zp, const float* __restrict__ wsT, const float* __restrict__ bs,
                   const float* __restrict__ b_in, const float* __restrict__ pe, __half* __restrict__ xtok_b, __half* __restrict__ xtok_s,
                   float* __restrict__ add, int C, int Cp, int Tp, int K) {
    extern __shared__ float s_zp[];
    const int b = blockIdx.x, n = threadIdx.x;
    for (int k = n; k < K; k += D) s_zp[k] = zp[(size_t)b * K + k];
    for (int i = n; i < Tp * Cp; i += D) {
        const int t = i / Cp, c = i % Cp;
        const size_t o = ((size_t)b * Tp + t) * Cp + c;
        split_f16(c < C ? past[((size_t)b * C + c) * Tp + t] : 0.f, xtok_b[o], xtok_s[o]);
    }
    __syncthreads();
    float s = 0.f;
    for (int k = 0; k < K; k++) s = fmaf(wsT[(size_t)k * D + n], s_zp[k], s);
    const float base = (s + bs[n]) + b_in[n];
    for (int t = 0; t < Tp; t++) add[((size_t)b * Tp + t) * D + n] = base + pe[(size_t)t * D + n];
}

}  // namespace

// encoder workspace for M = B*Tp rows (token pairs Cp wide), grown on demand
static int encoder_workspace(idb_handle* h, int M, int Cp) {
    Denoiser& d = h->den;
    const int F = d.cfg.d_ff, H = d.cfg.n_heads;
    if (M <= d.enc_cap) return IDB_OK;
    for (void* p : d.enc_owned) cudaFree(p);
    d.enc_owned.clear();
    d.enc_cap = 0;
    auto A = [&](float** p, size_t n) { if (cudaMalloc((void**)p, n * sizeof(float)) != cudaSuccess) return 1; d.enc_owned.push_back(*p); return 0; };
    auto AH = [&](__half** p, size_t n) { if (cudaMalloc((void**)p, n * sizeof(__half)) != cudaSuccess) return 1; d.enc_owned.push_back(*p); return 0; };
    int rc = 0;
    rc |= A(&d.e_add, (size_t)M * D); rc |= A(&d.e_h, (size_t)M * D); rc |= A(&d.e_h2, (size_t)M * D); rc |= A(&d.e_z, (size_t)M * D);
    rc |= A(&d.e_qkv, (size_t)M * (2 * D + H * D));
    rc |= AH(&d.e_xtok_b, (size_t)M * Cp); rc |= AH(&d.e_xtok_s, (size_t)M * Cp);
    rc |= AH(&d.e_h_b, (size_t)M * D); rc |= AH(&d.e_h_s, (size_t)M * D); rc |= AH(&d.e_h2_b, (size_t)M * D); rc |= AH(&d.e_h2_s, (size_t)M * D);
    rc |= AH(&d.e_ff_b, (size_t)M * F); rc |= AH(&d.e_ff_s, (size_t)M * F);
    if (rc) return idb_fail(h, IDB_ERR_CUDA, "out of device memory (encoder workspace)");
    d.enc_cap = M;
    return IDB_OK;
}

// Shared by both conditioning entry points, on the prepared token pairs (e_xtok, Cp wide) and addend (e_add): input embedding
// GEMM, the encoder layer stack, the last norm into the sequence-first (Tp,B,D) output.
static int encoder_stack(idb_handle* h, int B, int Tp, int Cp, float* cond_out, cudaStream_t st) {
    Denoiser& d = h->den;
    const idb_denoiser_config& c = d.cfg;
    const int M = B * Tp, F = c.d_ff, H = c.n_heads, N = c.n_queries;
    const bool fused = h->gemm_backend == 1 && h->fused_mlp && idb_mlp_tcgen05_supported(D, F);
    const bool pdl = h->pdl != 0;
    int rc;
    if ((rc = linear(h, d.e_xtok_b, d.e_xtok_s, Cp, d.w_in_b, d.w_in_s, Cp, nullptr, d.e_add, d.e_h, d.e_h_b, d.e_h_s, D, M, D, Cp, EPI_RES, st)))
        return rc;
    const dim3 slab_grid(B, (Tp + SLAB - 1) / SLAB);
    const int ln_blocks = (M * 32 + 255) / 256;
    const DenoiserLayer* pending = nullptr;      // layer whose final norm (norm2) has not been applied to e_z yet
    for (auto& L : d.enc_layers) {
        if (L.qan) {
            QanArgs qa = {};
            qa.zin = pending ? d.e_z : d.e_h; qa.prew = pending ? pending->ln3w : nullptr; qa.preb = pending ? pending->ln3b : nullptr;
            qa.qpack = L.qt_pack; qa.wk = L.wk; qa.lnw = L.ln1w; qa.lnb = L.ln1b;
            qa.out = d.e_h2; qa.out_b = d.e_h2_b; qa.out_s = d.e_h2_s; qa.T = Tp; qa.N = N; qa.B = B; qa.Tk = 0; qa.H = H;
            idb_launch(pdl, k_qan_xattn_ln<false>, slab_grid, ANT, qan_enc_smem(), st, qa);
            LAUNCH_CHECK(h);
        } else {
            if (pending) {
                idb_launch(pdl, k_ln, ln_blocks, 256, 0, st, d.e_z, pending->ln3w, pending->ln3b, d.e_h, d.e_h_b, d.e_h_s, M);
                LAUNCH_CHECK(h);
            }
            const int NQ = 2 * D + H * D;
            if ((rc = linear(h, d.e_h_b, d.e_h_s, D, L.w_qkvf_b, L.w_qkvf_s, D, L.b_qkvf, nullptr, d.e_qkv, nullptr, nullptr, NQ, M, NQ, D,
                             EPI_BIAS, st))) return rc;
            AttnArgs aa = {};
            aa.q = d.e_qkv; aa.ldq = NQ; aa.k = d.e_qkv + D; aa.ldk = NQ; aa.v = d.e_qkv + 2 * D; aa.ldv = NQ; aa.res = d.e_h; aa.bo = L.bo_f;
            aa.lnw = L.ln1w; aa.lnb = L.ln1b; aa.out = d.e_h2; aa.out_b = d.e_h2_b; aa.out_s = d.e_h2_s; aa.T = Tp; aa.H = H;
            idb_launch(pdl, k_attn_ln, slab_grid, ANT, attn_smem(Tp, H), st, aa);
            LAUNCH_CHECK(h);
        }
        if (fused) {
            if (h->fused_mlp >= 2) {
                if ((rc = idb_mlp_tcgen05(h, d.e_h2_b, d.e_h2_s, L.w1_b, L.w1_s, L.b1, L.w2_b, L.w2_s, L.b2, d.e_h2, D, d.e_h, D, M, h->pdl,
                                          st, L.ln3w, L.ln3b, d.e_h_b, d.e_h_s)))
                    return rc;
                continue;
            }
            if ((rc = idb_mlp_tcgen05(h, d.e_h2_b, d.e_h2_s, L.w1_b, L.w1_s, L.b1, L.w2_b, L.w2_s, L.b2, d.e_h2, D, d.e_z, D, M, h->pdl, st)))
                return rc;
        } else {
            // two GEMMs (also the only path for d_ff != 1024, e.g. the skeleton model's 256)
            if ((rc = linear(h, d.e_h2_b, d.e_h2_s, D, L.w1_b, L.w1_s, D, L.b1, nullptr, nullptr, d.e_ff_b, d.e_ff_s, F, M, F, D,
                             EPI_BIAS | EPI_GELU, st))) return rc;
            if ((rc = linear(h, d.e_ff_b, d.e_ff_s, F, L.w2_b, L.w2_s, F, L.b2, d.e_h2, d.e_z, nullptr, nullptr, D, M, D, F, EPI_BIAS | EPI_RES, st)))
                return rc;
        }
        pending = &L;
    }
    // last norm (or, when the fused feed-forward kernel already applied it, a plain copy) into the (Tp,B,D) layout
    idb_launch(pdl, k_ln_seq_first, ln_blocks, 256, 0, st, pending ? d.e_z : d.e_h, pending ? pending->ln3w : (const float*)nullptr,
               pending ? pending->ln3b : (const float*)nullptr, cond_out, B, Tp);
    LAUNCH_CHECK(h);
    return IDB_OK;
}

extern "C" int idb_encode_condition(idb_handle* h, int B, int Tp, const float* past, const float* pc_embedding, float* cond_out,
                                    void* stream) {
    IDB_ENTER(h);
    if (!h || !past || !pc_embedding || !cond_out || B <= 0 || Tp <= 0) return IDB_ERR_ARG;
    Denoiser& d = h->den;
    if (!d.committed) return idb_fail(h, IDB_ERR_STATE, "idb_denoiser_commit first");
    if (d.enc_layers.empty()) return idb_fail(h, IDB_ERR_STATE, "the conditioning encoder's weights (encoder.layers.*) were not loaded");
    if (Tp > 36) return idb_fail(h, IDB_ERR_ARG, "supported past window: <= 36 frames");
    const idb_denoiser_config& c = d.cfg;
    const int M = B * Tp, C = c.c_body + c.c_obj, Cp = (C + 7) & ~7;
    if (c.variant != 0) return idb_fail(h, IDB_ERR_ARG, "idb_encode_condition: SMPL model only (skeleton: idb_encode_condition_skeleton)");
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = encoder_workspace(h, M, Cp))) return rc;
    k_cond_tokens<<<B, 256, 0, st>>>(past, pc_embedding, d.b_in, d.pe, d.e_xtok_b, d.e_xtok_s, d.e_add, C, Cp, Tp);
    LAUNCH_CHECK(h);
    return encoder_stack(h, B, Tp, Cp, cond_out, st);
}

extern "C" int idb_encode_condition_skeleton(idb_handle* h, int B, int Tp, const float* past, const float* zero_pose_obj, float* cond_out,
                                             void* stream) {
    IDB_ENTER(h);
    if (!h || !past || !zero_pose_obj || !cond_out || B <= 0 || Tp <= 0) return IDB_ERR_ARG;
    Denoiser& d = h->den;
    if (!d.committed) return idb_fail(h, IDB_ERR_STATE, "idb_denoiser_commit first");
    const idb_denoiser_config& c = d.cfg;
    if (c.variant != 1) return idb_fail(h, IDB_ERR_ARG, "idb_encode_condition_skeleton: skeleton model only (SMPL: idb_encode_condition)");
    if (d.enc_layers.empty() || !d.w_shapeT)
        return idb_fail(h, IDB_ERR_STATE, "the conditioning encoder's weights (encoder.layers.*, shapeEmbedding.*) were not loaded");
    if (Tp > 36 || Tp > d.pe_rows) return idb_fail(h, IDB_ERR_ARG, "supported past window: <= 36 frames");
    const int M = B * Tp, C = c.c_body + c.c_obj + c.c_extra, Cp = (C + 7) & ~7, K = c.c_obj;
    cudaStream_t st = (cudaStream_t)stream;
    int rc;
    if ((rc = encoder_workspace(h, M, Cp))) return rc;
    k_skel_cond_tokens<<<B, D, K * sizeof(float), st>>>(past, zero_pose_obj, d.w_shapeT, d.b_shape, d.b_in, d.pe, d.e_xtok_b, d.e_xtok_s,
                                                        d.e_add, C, Cp, Tp, K);
    LAUNCH_CHECK(h);
    return encoder_stack(h, B, Tp, Cp, cond_out, st);
}

extern "C" int idb_denoiser_forward(idb_handle* h, const float* x, const int64_t* timesteps, float* out, void* stream) {
    IDB_ENTER(h);
    if (!h || !x || !timesteps || !out) return IDB_ERR_ARG;
    return idb_denoiser_run(h, x, (const long long*)timesteps, nullptr, nullptr, out, (cudaStream_t)stream);
}
