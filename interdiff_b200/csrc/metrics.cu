// Evaluation metrics on the device (SURVEY 8f rank 3): the reference's `metrics` (eval_smpl_short.py:24-81) -
// global / pelvis-aligned MPJPE, body and object translation error, object rotation error (quaternion L1, sign
// ambiguity resolved by the minimum) and the penetration ratio of the posed object points against the body mesh.
// The penetration term reuses the hot path's kernels (vertex normals, cluster-pruned signed nearest neighbour);
// everything else is one reduction kernel per batch.  All reductions run in a fixed order (bit-reproducible).
// The skeleton model's metrics (eval_skeleton.py:46-68, train_diffusion_skeleton.py:65-87) are one kernel of their own.
#include "common.cuh"
#include "body.cuh"

namespace {

// pytorch3d 0.7.2 axis_angle_to_quaternion: (w, x, y, z), small-angle series below 1e-6
__device__ __forceinline__ void mt_aa_to_quat(const float* aa, float* q) {
    const float ang = sqrtf(aa[0] * aa[0] + aa[1] * aa[1] + aa[2] * aa[2]);
    const float half = ang * 0.5f;
    const float s = fabsf(ang) < 1e-6f ? 0.5f - (ang * ang) / 48.0f : sinf(half) / ang;
    q[0] = cosf(half); q[1] = aa[0] * s; q[2] = aa[1] * s; q[3] = aa[2] * s;
}

// posed object points of frame f = t*B + b:  out[f][p] = R(aa) pts[b][p] + trans   (eval_smpl_short.py:36-37)
__global__ void k_metric_objpts(const float* __restrict__ obj_pred, const float* __restrict__ pts, float* __restrict__ out, int B, int P) {
    __shared__ float R[12];
    const int f = blockIdx.y, b = f % B;
    if (threadIdx.x == 0) {
        const float* o = obj_pred + (size_t)f * 6;
        float q[4];
        mt_aa_to_quat(o, q);
        const float r = q[0], i = q[1], j = q[2], k = q[3];
        const float two_s = 2.0f / (r * r + i * i + j * j + k * k);
        R[0] = 1 - two_s * (j * j + k * k); R[1] = two_s * (i * j - k * r); R[2] = two_s * (i * k + j * r);
        R[3] = two_s * (i * j + k * r); R[4] = 1 - two_s * (i * i + k * k); R[5] = two_s * (j * k - i * r);
        R[6] = two_s * (i * k - j * r); R[7] = two_s * (j * k + i * r); R[8] = 1 - two_s * (i * i + j * j);
        R[9] = o[3]; R[10] = o[4]; R[11] = o[5];
    }
    __syncthreads();
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const float x = pts[((size_t)b * P + p) * 3], y = pts[((size_t)b * P + p) * 3 + 1], z = pts[((size_t)b * P + p) * 3 + 2];
    float* o = out + ((size_t)f * P + p) * 3;
    o[0] = (x * R[0] + y * R[1] + z * R[2]) + R[9];
    o[1] = (x * R[3] + y * R[4] + z * R[5]) + R[10];
    o[2] = (x * R[6] + y * R[7] + z * R[8]) + R[11];
}

// one block per sample b: per-frame terms by warps (lanes over joints / points), then a sequential mean over frames.
// out[k][b], k = global_mpjpe, local_mpjpe, body_translation, obj_translation, obj_rot_error, penetrate
__global__ void __launch_bounds__(256)
k_metric_reduce(const float* __restrict__ obj_pred, const float* __restrict__ jtr, const float* __restrict__ body,
                const float* __restrict__ obj_gt, const float* __restrict__ jtr_gt, const float* __restrict__ body_gt,
                const float* __restrict__ o2h, float* __restrict__ out, int T, int B, int J, int P, int Db) {
    extern __shared__ float sm[];          // [6][T] per-frame terms
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int t = warp; t < T; t += 8) {
        const size_t f = (size_t)t * B + b;
        const float* a = jtr + f * J * 3;
        const float* g = jtr_gt + f * J * 3;
        float sg = 0.f, sl = 0.f;
        for (int j = lane; j < J; j += 32) {
            const float dx = a[j * 3] - g[j * 3], dy = a[j * 3 + 1] - g[j * 3 + 1], dz = a[j * 3 + 2] - g[j * 3 + 2];
            sg += sqrtf(dx * dx + dy * dy + dz * dz);
            // (a_j - a_0) - (g_j - g_0): evaluated like the reference (subtract the pelvis from each side first)
            const float lx = (a[j * 3] - a[0]) - (g[j * 3] - g[0]), ly = (a[j * 3 + 1] - a[1]) - (g[j * 3 + 1] - g[1]),
                        lz = (a[j * 3 + 2] - a[2]) - (g[j * 3 + 2] - g[2]);
            sl += sqrtf(lx * lx + ly * ly + lz * lz);
        }
        sg = warp_sum(sg); sl = warp_sum(sl);
        int neg = 0;
        const float* d = o2h + f * P;
        for (int p = lane; p < P; p += 32) neg += d[p] < 0.f ? 1 : 0;
#pragma unroll
        for (int o = 16; o; o >>= 1) neg += __shfl_xor_sync(0xffffffffu, neg, o);
        if (lane == 0) {
            sm[0 * T + t] = sg / (float)J;
            sm[1 * T + t] = sl / (float)J;
            const float* bt = body + f * Db + Db - 3;
            const float* bg = body_gt + f * Db + Db - 3;
            const float tx = bt[0] - bg[0], ty = bt[1] - bg[1], tz = bt[2] - bg[2];
            sm[2 * T + t] = sqrtf(tx * tx + ty * ty + tz * tz);
            const float* op = obj_pred + f * 6;
            const float* og = obj_gt + f * 6;
            const float ox = op[3] - og[3], oy = op[4] - og[4], oz = op[5] - og[5];
            sm[3 * T + t] = sqrtf(ox * ox + oy * oy + oz * oz);
            float q[4], qg[4];
            mt_aa_to_quat(op, q);
            mt_aa_to_quat(og, qg);
            float e1 = 0.f, e2 = 0.f;
            for (int k = 0; k < 4; k++) { e1 += fabsf(q[k] - qg[k]); e2 += fabsf(q[k] + qg[k]); }
            sm[4 * T + t] = fminf(e1, e2);
            sm[5 * T + t] = (float)neg / (float)P;
        }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        float s = 0.f;
        for (int t = 0; t < T; t++) s += sm[threadIdx.x * T + t];
        out[(size_t)threadIdx.x * B + b] = s / (float)T;
    }
}

}  // namespace

extern "C" int idb_metrics(idb_handle* h, int T, int B, int J, int P, int Db, const float* obj_pred, const float* body_jtr,
                           const float* body, const float* obj_gt, const float* body_jtr_gt, const float* body_gt, const float* verts,
                           const float* obj_points, float* out, void* stream) {
    IDB_ENTER(h);
    if (!h || !obj_pred || !body_jtr || !body || !obj_gt || !body_jtr_gt || !body_gt || !verts || !obj_points || !out) return IDB_ERR_ARG;
    if (T <= 0 || B <= 0 || J <= 0 || P <= 0 || Db < 3) return IDB_ERR_ARG;
    if (!h->body || !h->body->faces) return idb_fail(h, IDB_ERR_STATE, "idb_body_init with faces first");
    const int V = h->body->V, F = T * B;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t need = sizeof(float) * ((size_t)F * P * 3 + (size_t)F * V * 3 + (size_t)F * P);
    if (need > h->metrics_bytes) {
        if (h->metrics_ws) { CUDA_TRY(h, cudaStreamSynchronize(st)); cudaFree(h->metrics_ws); h->metrics_ws = nullptr; }
        CUDA_TRY(h, cudaMalloc(&h->metrics_ws, need));
        h->metrics_bytes = need;
    }
    float* objp = reinterpret_cast<float*>(h->metrics_ws);
    float* normals = objp + (size_t)F * P * 3;
    float* o2h = normals + (size_t)F * V * 3;
    k_metric_objpts<<<dim3((P + 255) / 256, F), 256, 0, st>>>(obj_pred, obj_points, objp, B, P);
    LAUNCH_CHECK(h);
    int rc;
    if ((rc = idb_vertex_normals(h, F, verts, normals, st))) return rc;
    if ((rc = idb_signed_nn(h, F, P, V, objp, verts, normals, o2h, nullptr, nullptr, st))) return rc;
    k_metric_reduce<<<B, 256, sizeof(float) * 6 * T, st>>>(obj_pred, body_jtr, body, obj_gt, body_jtr_gt, body_gt, o2h, out, T, B, J, P, Db);
    LAUNCH_CHECK(h);
    return IDB_OK;
}

// ---- skeleton model metrics (eval_skeleton.py:46-68 calc_metric_single, train_diffusion_skeleton.py:65-87 calc_metric) -----
namespace {
// One block per sample b, read straight from the sample layout (B,1,C,T), C = 3 J + 3 P + 7 = [joints | keypoints | trans(3),
// quat xyzw(4)]: per-frame terms by warps (lanes over joints / keypoints) for the future frames t >= past_len, then a sequential
// mean over those frames.  out[k][b], k = mpjpe_h, mpjpe_o, translation_error, rotation_error (sign-min of the quaternion L1
// distance, eval_skeleton.py:59-62), rotation_error_l2 (the same with the L2 norm, train_diffusion_skeleton.py:78-81).
__global__ void __launch_bounds__(256)
k_skeleton_metrics(const float* __restrict__ pred, const float* __restrict__ gt, float* __restrict__ out, int B, int T, int P0, int J, int Np) {
    extern __shared__ float sm[];          // [5][nF] per-frame terms
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int C = 3 * (J + Np) + 7, nF = T - P0;
    const float* pp = pred + (size_t)b * C * T;
    const float* gg = gt + (size_t)b * C * T;
    auto dist3 = [&](int c0, int t) {
        const float dx = pp[(size_t)c0 * T + t] - gg[(size_t)c0 * T + t], dy = pp[(size_t)(c0 + 1) * T + t] - gg[(size_t)(c0 + 1) * T + t],
                    dz = pp[(size_t)(c0 + 2) * T + t] - gg[(size_t)(c0 + 2) * T + t];
        return sqrtf(dx * dx + dy * dy + dz * dz);
    };
    for (int f = warp; f < nF; f += 8) {
        const int t = P0 + f;
        float sh = 0.f, so = 0.f;
        for (int j = lane; j < J; j += 32) sh += dist3(3 * j, t);
        for (int p = lane; p < Np; p += 32) so += dist3(3 * (J + p), t);
        sh = warp_sum(sh); so = warp_sum(so);
        if (lane == 0) {
            const int c0 = 3 * (J + Np);
            sm[0 * nF + f] = sh / (float)J;
            sm[1 * nF + f] = so / (float)Np;
            sm[2 * nF + f] = dist3(c0, t);
            float e1 = 0.f, e2 = 0.f, s1 = 0.f, s2 = 0.f;
            for (int k = 0; k < 4; k++) {
                const float p = pp[(size_t)(c0 + 3 + k) * T + t], g = gg[(size_t)(c0 + 3 + k) * T + t];
                const float dm = p - g, dp = p + g;
                e1 += fabsf(dm); e2 += fabsf(dp); s1 += dm * dm; s2 += dp * dp;
            }
            sm[3 * nF + f] = fminf(e1, e2);
            sm[4 * nF + f] = fminf(sqrtf(s1), sqrtf(s2));
        }
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        float s = 0.f;
        for (int f = 0; f < nF; f++) s += sm[threadIdx.x * nF + f];
        out[(size_t)threadIdx.x * B + b] = s / (float)nF;
    }
}
}  // namespace

extern "C" int idb_skeleton_metrics(idb_handle* h, int B, int T, int past_len, int n_joints, int n_points, const float* pred, const float* gt,
                                    float* out, void* stream) {
    IDB_ENTER(h);
    if (!h || !pred || !gt || !out || B <= 0 || T <= 0 || n_joints <= 0 || n_points <= 0) return IDB_ERR_ARG;
    if (past_len < 0 || past_len >= T) return idb_fail(h, IDB_ERR_ARG, "past_len must leave at least one future frame");
    const int nF = T - past_len;
    if (nF > 2048) return idb_fail(h, IDB_ERR_ARG, "at most 2048 future frames");
    k_skeleton_metrics<<<B, 256, sizeof(float) * 5 * nF, (cudaStream_t)stream>>>(pred, gt, out, B, T, past_len, n_joints, n_points);
    LAUNCH_CHECK(h);
    return IDB_OK;
}

// ---- post-processing of a sampled window (SURVEY 8f rank 3): smooth + best-of-N reduction -------------------------------
namespace {
// x (T, inner): every predicted future frame is shifted by the second-difference jump at the past / future seam
// (eval_smpl_short.py:217-223: x[-F:] = x[-F:] + (2 x[-F-1] - x[-F-2] - x[-F]); the right-hand side uses the OLD x[-F]).
__global__ void k_smooth(float* __restrict__ x, int T, int Fut, size_t inner) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= inner) return;
    const int s = T - Fut;                                 // first future frame
    const float d = (2.0f * x[(size_t)(s - 1) * inner + i] - x[(size_t)(s - 2) * inner + i]) - x[(size_t)s * inner + i];
    for (int t = s; t < T; t++) x[(size_t)t * inner + i] = x[(size_t)t * inner + i] + d;
}
__global__ void k_min_inplace(float* __restrict__ acc, const float* __restrict__ cur, size_t n) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) acc[i] = fminf(acc[i], cur[i]);
}
}  // namespace

extern "C" int idb_smooth(idb_handle* h, int T, int future_len, long long inner, float* x, void* stream) {
    IDB_ENTER(h);
    if (!h || !x || inner <= 0) return IDB_ERR_ARG;
    if (future_len < 1 || T - future_len < 2) return idb_fail(h, IDB_ERR_ARG, "smooth needs at least two past frames and one future frame");
    k_smooth<<<(unsigned)((inner + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, T, future_len, (size_t)inner);
    LAUNCH_CHECK(h);
    return IDB_OK;
}

/* acc[i] = min(acc[i], cur[i]) : the element-wise minimum over the diverse samples of a batch (eval_smpl_short.py:268-296) */
extern "C" int idb_metric_min(idb_handle* h, long long n, float* acc, const float* cur, void* stream) {
    IDB_ENTER(h);
    if (!h || !acc || !cur || n <= 0) return IDB_ERR_ARG;
    k_min_inplace<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(acc, cur, (size_t)n);
    LAUNCH_CHECK(h);
    return IDB_OK;
}
