// cov_pose.cu — ModelPose fused forward+backward (reference src/model.py:98-127).
//
// One pass over the cloud: each thread streams groups of four points (three LDG.128, 48 B),
// evaluates m and dm/dy in registers, writes the four observations with one STG.128 and keeps
// seven running sums (sum m, F = sum dm/dy, T = sum dm/dy x y).  Warp shuffles + one shared-memory
// step reduce them per block into a row of fp32 partials; a second tiny kernel adds the rows in
// fp64 in a fixed order (deterministic, no atomics).  HBM-bound: 16 B/point.
#include "cov_common.cuh"
#include "../../include/coverage_b200.h"

namespace {

struct PoseSums {
    float m, fx, fy, fz, tx, ty, tz;
};

__device__ __forceinline__ void pose_point(float x, float y, float z, float wgt, const float4* row, const CovConst& C,
                                           float& obs, PoseSums& S) {
    CovEval ev;
    float m = cov_vis<true>(x, y, z, row[0], row[1], row[2], row[3], C, &ev);
    float gx, gy, gz;
    cov_vis_grad(m, ev, row[0], row[1], row[2], C, gx, gy, gz);
    m = m > 0.f ? m : 0.f;  // also drops the NaN of the measure-zero h2 == -eps case
    m *= wgt; gx *= wgt; gy *= wgt; gz *= wgt;
    const float yx = x - row[5].x, yy = y - row[5].y, yz = z - row[5].z;  // lever arm about the camera centre
    obs = m;
    S.m += m;
    S.fx += gx; S.fy += gy; S.fz += gz;
    S.tx += gy * yz - gz * yy;   // (g x y)_x
    S.ty += gz * yx - gx * yz;
    S.tz += gx * yy - gy * yx;
}

template <bool HAS_W, bool HAS_OBS>
__global__ void __launch_bounds__(COV_THREADS)
cov_pose_kernel(const float* __restrict__ xyz, int64_t n, const float* __restrict__ weight,
                const float* __restrict__ trans, const float* __restrict__ quat, const float* __restrict__ K9,
                CovConst C, float* __restrict__ obs, float* __restrict__ partials) {
    __shared__ float4 row[COV_ROW_F4];
    __shared__ float red[COV_THREADS / 32][8];
    if (threadIdx.x == 0) cov_pose_row(trans, quat, K9, C, row);
    __syncthreads();

    PoseSums S = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    const int64_t ngroups = n >> 2;  // full groups of four points
    const int64_t stride = (int64_t)gridDim.x * COV_THREADS;
    const float4* __restrict__ xyz4 = reinterpret_cast<const float4*>(xyz);
    for (int64_t g = (int64_t)blockIdx.x * COV_THREADS + threadIdx.x; g < ngroups; g += stride) {
        const float4 a = __ldg(xyz4 + g * 3), b = __ldg(xyz4 + g * 3 + 1), c = __ldg(xyz4 + g * 3 + 2);
        float4 wv = make_float4(1.f, 1.f, 1.f, 1.f);
        if (HAS_W) wv = __ldg(reinterpret_cast<const float4*>(weight) + g);
        float4 o;
        pose_point(a.x, a.y, a.z, wv.x, row, C, o.x, S);
        pose_point(a.w, b.x, b.y, wv.y, row, C, o.y, S);
        pose_point(b.z, b.w, c.x, wv.z, row, C, o.z, S);
        pose_point(c.y, c.z, c.w, wv.w, row, C, o.w, S);
        if (HAS_OBS) reinterpret_cast<float4*>(obs)[g] = o;
    }
    // ragged tail (n % 4 points), handled by the first threads of block 0
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const int64_t j = (ngroups << 2) + threadIdx.x;
        float o;
        pose_point(xyz[j * 3], xyz[j * 3 + 1], xyz[j * 3 + 2], HAS_W ? weight[j] : 1.f, row, C, o, S);
        if (HAS_OBS) obs[j] = o;
    }
    float v[7] = {S.m, S.fx, S.fy, S.fz, S.tx, S.ty, S.tz};
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        const float r = cov_warp_sum(v[k]);
        if (lane == 0) red[warp][k] = r;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        float r = 0.f;
        if (threadIdx.x < 7)
            for (int wp = 0; wp < COV_THREADS / 32; ++wp) r += red[wp][threadIdx.x];
        partials[blockIdx.x * 8 + threadIdx.x] = r;
    }
}

// acc[k] = sum over blocks of partials[b][k], fp64, fixed order.
__global__ void cov_pose_reduce_kernel(const float* __restrict__ partials, int nblocks, double* __restrict__ acc) {
    const int k = threadIdx.x & 7, part = threadIdx.x >> 3;  // 8 columns x 32 row-strides
    double s = 0.0;
    for (int b = part; b < nblocks; b += 32) s += (double)partials[b * 8 + k];
    __shared__ double sh[32][8];
    sh[part][k] = s;
    __syncthreads();
    if (threadIdx.x < 8) {
        double t = 0.0;
        for (int p = 0; p < 32; ++p) t += sh[p][threadIdx.x];
        acc[threadIdx.x] = t;
    }
}

// d(sum)/dt = -F ;  d(sum)/dq~ = 2 ((0,T) (x) q) / |q~|   (tangent to the unit sphere, so the
// (I - q q^T) projection of F.normalize's backward is the identity on it).
__device__ __forceinline__ void pose_epilogue_row(const double* __restrict__ acc, const float* __restrict__ quat,
                                                  float* __restrict__ out) {
    double w = quat[0], x = quat[1], y = quat[2], z = quat[3];
    double n = sqrt(w * w + x * x + y * y + z * z);
    n = n > 1e-12 ? n : 1e-12;
    w /= n; x /= n; y /= n; z /= n;
    const double tx = acc[4], ty = acc[5], tz = acc[6];
    out[0] = (float)acc[0];
    out[1] = (float)(-acc[1]);
    out[2] = (float)(-acc[2]);
    out[3] = (float)(-acc[3]);
    // (0,T) (x) (w,x,y,z)
    out[4] = (float)(2.0 * (-tx * x - ty * y - tz * z) / n);
    out[5] = (float)(2.0 * (tx * w + ty * z - tz * y) / n);
    out[6] = (float)(2.0 * (ty * w - tx * z + tz * x) / n);
    out[7] = (float)(2.0 * (tz * w + tx * y - ty * x) / n);
}

__global__ void cov_pose_epilogue_kernel(const double* __restrict__ acc, const float* __restrict__ quat,
                                         float* __restrict__ out) {
    if (threadIdx.x != 0) return;
    pose_epilogue_row(acc, quat, out);
}

// ---- K candidate poses on one cloud (cov_pose_batch_fused) ---------------------------------------------------------
// For every pose k the 8 sums cov_pose_fused computes for pose k alone, in one pass over the cloud per chunk of
// kBatchChunk poses.  A warp owns one box of 128 consecutive points (4 per lane, the three LDG.128 of cov_pose_kernel) and
// walks a slice of the chunk's poses.  Per (box, pose): the four pose_point calls (unchanged, so every pair adds exactly
// what cov_pose_fused adds for it), the fixed 9-shuffle tree cov_warp_sum8 over the warp, and one lane per component
// adds the result in fp64 to the warp's own row of that pose in shared memory.  At the end of a chunk the block adds the
// warps' rows in a fixed order and sends every non-zero (pose, component) to acc with one fp64 atomic.  So fp32 sums at
// most the 128 points of one (box, pose) in a fixed order; everything above is fp64, and only the order of the fp64
// atomics differs between runs.
//
// Exact pruning (boxes given and not dense): a warp skips a pose when  fl(box_q2lb(lo, hi, td) * kd) >= 128.
// box_q2lb bounds the COMPUTED q2 of every point of the box from below (cov_common.cuh).  cov_vis forms
// Q = fma(q2, kd, t) with t = fma(dv, dv, du * du) >= 0, and rounding is monotone, so Q >= fl(q2 kd) >= 128 (or Q is
// NaN) and ex2.approx.ftz(-Q) flushes to +0: 2^-128 is below the smallest normal float.  m = E s is then 0 or NaN, which
// pose_point's m > 0 clamp maps to 0 (the NaN s of h2 == -eps included), cov_vis_grad gives g = 0, and the pair adds
// exactly zero to every sum, for any finite point and weight.  A skipped (box, pose) would have summed to exactly zero:
// pruned and dense results differ only in the order of the fp64 additions.
constexpr int kBatchChunk = 64;     // poses per chunk (rows 96 B, per-warp fp64 sums 8 x 64 B each, in shared memory)
// resident blocks per SM: 4 fit 64 registers; the weighted kernel's four extra live weights would spill there
__host__ __device__ constexpr int batch_min_blocks(bool has_w) { return has_w ? 3 : 4; }
constexpr int kBatchWarps = COV_THREADS / 32;

// pose rows of all K poses, once per call (fp64 inside, as cov_pose_kernel builds its row), and acc zeroed
__global__ void cov_pose_batch_table_kernel(const float* __restrict__ trans, const float* __restrict__ quats, int n_poses,
                                            const float* __restrict__ K9, CovConst C, float4* __restrict__ table,
                                            double* __restrict__ acc) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_poses) return;
    cov_pose_row(trans + 3 * (size_t)k, quats + 4 * (size_t)k, K9, C, table + (size_t)k * COV_ROW_F4);
#pragma unroll
    for (int i = 0; i < COV_POSE_ACC; ++i) acc[(size_t)k * COV_POSE_ACC + i] = 0.0;
}

template <bool HAS_W>
__global__ void __launch_bounds__(COV_THREADS, batch_min_blocks(HAS_W))
cov_pose_batch_kernel(const float* __restrict__ xyz, int64_t n, const float* __restrict__ weight,
                      const float4* __restrict__ table, int n_poses, CovConst C, const float4* __restrict__ boxes,
                      int per_slice, double* __restrict__ acc, unsigned long long* __restrict__ stats) {
    __shared__ float4 srow[kBatchChunk * COV_ROW_F4];
    __shared__ double wsum[kBatchWarps][kBatchChunk * 8];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t nboxes = (n + 127) >> 7, ngroups = n >> 2;
    const int64_t gwarp = (int64_t)blockIdx.x * kBatchWarps + warp, nwarps = (int64_t)gridDim.x * kBatchWarps;
    const float4* __restrict__ xyz4 = reinterpret_cast<const float4*>(xyz);
    double* __restrict__ mine = wsum[warp];
    unsigned n_all = 0, n_eval = 0;  // (warp box, pose) pairs of this warp: all, evaluated
    for (int c0 = 0; c0 < n_poses; c0 += kBatchChunk) {
        const int kc = min(n_poses - c0, kBatchChunk);
        for (int i = tid; i < kc * COV_ROW_F4; i += COV_THREADS) srow[i] = table[(size_t)c0 * COV_ROW_F4 + i];
        for (int i = tid; i < kBatchWarps * kBatchChunk * 8; i += COV_THREADS) (&wsum[0][0])[i] = 0.0;
        __syncthreads();
        const int nslices = (kc + per_slice - 1) / per_slice;
        const int64_t items = nboxes * nslices;
        for (int64_t it = gwarp; it < items; it += nwarps) {
            const int64_t b = it / nslices;
            const int k0 = (int)(it - b * nslices) * per_slice, k1 = min(k0 + per_slice, kc);
            const int64_t g = b * 32 + lane;  // this lane's group of four points
            float4 pa, pb, pc, wv = make_float4(1.f, 1.f, 1.f, 1.f);
            if (g < ngroups) {
                pa = __ldg(xyz4 + g * 3); pb = __ldg(xyz4 + g * 3 + 1); pc = __ldg(xyz4 + g * 3 + 2);
                if (HAS_W) wv = __ldg(reinterpret_cast<const float4*>(weight) + g);
            } else {  // the ragged end: points past n are 3e18 sentinels, which give m = 0 and g = 0 for every pose
                float p[12], w4[4];
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    const int64_t j = g * 4 + s;
                    const bool ok = j < n;
                    p[3 * s] = ok ? xyz[j * 3] : 3e18f;
                    p[3 * s + 1] = ok ? xyz[j * 3 + 1] : 3e18f;
                    p[3 * s + 2] = ok ? xyz[j * 3 + 2] : 3e18f;
                    w4[s] = (HAS_W && ok) ? weight[j] : 1.f;
                }
                pa = make_float4(p[0], p[1], p[2], p[3]);
                pb = make_float4(p[4], p[5], p[6], p[7]);
                pc = make_float4(p[8], p[9], p[10], p[11]);
                wv = make_float4(w4[0], w4[1], w4[2], w4[3]);
            }
            float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
            if (boxes) { lo = __ldg(boxes + 2 * b); hi = __ldg(boxes + 2 * b + 1); }
            n_all += k1 - k0;
            for (int k = k0; k < k1; ++k) {
                const float4* row = srow + k * COV_ROW_F4;
                if (boxes && __fmul_rn(box_q2lb(lo, hi, row[3]), C.kd) >= 128.f) continue;
                ++n_eval;
                PoseSums S = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                float o;
                pose_point(pa.x, pa.y, pa.z, wv.x, row, C, o, S);
                pose_point(pa.w, pb.x, pb.y, wv.y, row, C, o, S);
                pose_point(pb.z, pb.w, pc.x, wv.z, row, C, o, S);
                pose_point(pc.y, pc.z, pc.w, wv.w, row, C, o, S);
                float v[8] = {S.m, S.fx, S.fy, S.fz, S.tx, S.ty, S.tz, 0.f};
                cov_warp_sum8(v, lane);
                if ((lane & 3) == 0) mine[k * 8 + ((lane >> 2) & 7)] += (double)v[0];
            }
        }
        __syncthreads();
        for (int i = tid; i < kc * 8; i += COV_THREADS) {
            double s = 0.0;
#pragma unroll
            for (int w = 0; w < kBatchWarps; ++w) s += wsum[w][i];
            if (s != 0.0) atomicAdd(acc + (size_t)c0 * 8 + i, s);
        }
        __syncthreads();  // the next chunk overwrites the rows and the sums
    }
    if (stats && lane == 0) {
        atomicAdd(stats + 0, (unsigned long long)n_all);
        atomicAdd(stats + 1, (unsigned long long)n_eval);
    }
}

__global__ void cov_pose_batch_epilogue_kernel(const double* __restrict__ acc, const float* __restrict__ quats, int n_poses,
                                               float* __restrict__ out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_poses) return;
    pose_epilogue_row(acc + (size_t)k * COV_POSE_ACC, quats + 4 * (size_t)k, out + (size_t)k * 8);
}

size_t batch_table_bytes(int n_poses) {
    return ((size_t)(n_poses < 1 ? 1 : n_poses) * COV_ROW_F4 * sizeof(float4) + 255) & ~(size_t)255;
}

int pose_grid(int64_t n) {
    const int64_t groups = (n >> 2) + 1;
    int64_t blocks = (groups + COV_THREADS - 1) / COV_THREADS;
    const int64_t cap = (int64_t)cov_sm_count_cached() * 4;
    if (blocks > cap) blocks = cap;
    if (blocks > COV_MAX_GRID) blocks = COV_MAX_GRID;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

}  // namespace

extern "C" size_t cov_pose_workspace_bytes(int64_t n) {
    (void)n;
    return (size_t)COV_MAX_GRID * 8 * sizeof(float);
}

extern "C" int cov_pose_fused(const float* xyz, int64_t n, const float* weight, const float* trans, const float* quat,
                              const float* K, const cov_camera* cam, float* obs, double* acc, void* ws, size_t ws_bytes,
                              void* stream) {
    if (n < 0 || (n > 0 && !xyz) || !trans || !quat || !K || !cam || !acc || !ws) {
        cov_set_error("cov_pose_fused: null pointer or negative n");
        return COV_ERR_ARG;
    }
    if (ws_bytes < cov_pose_workspace_bytes(n)) {
        cov_set_error("cov_pose_fused: workspace %zu < %zu bytes", ws_bytes, cov_pose_workspace_bytes(n));
        return COV_ERR_WORKSPACE;
    }
    if (((uintptr_t)xyz | (uintptr_t)obs | (uintptr_t)weight | (uintptr_t)ws) & 15) {
        cov_set_error("cov_pose_fused: xyz/obs/weight/workspace must be 16-byte aligned");
        return COV_ERR_ALIGN;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    const int grid = pose_grid(n);
    float* partials = (float*)ws;
    if (weight) {
        if (obs) cov_pose_kernel<true, true><<<grid, COV_THREADS, 0, s>>>(xyz, n, weight, trans, quat, K, C, obs, partials);
        else cov_pose_kernel<true, false><<<grid, COV_THREADS, 0, s>>>(xyz, n, weight, trans, quat, K, C, obs, partials);
    } else {
        if (obs) cov_pose_kernel<false, true><<<grid, COV_THREADS, 0, s>>>(xyz, n, weight, trans, quat, K, C, obs, partials);
        else cov_pose_kernel<false, false><<<grid, COV_THREADS, 0, s>>>(xyz, n, weight, trans, quat, K, C, obs, partials);
    }
    cov_pose_reduce_kernel<<<1, 256, 0, s>>>(partials, grid, acc);
    return cov_check_launch("cov_pose_fused");
}

extern "C" int cov_pose_epilogue(const double* acc, const float* trans, const float* quat, float* out, void* stream) {
    (void)trans;
    if (!acc || !quat || !out) {
        cov_set_error("cov_pose_epilogue: null pointer");
        return COV_ERR_ARG;
    }
    cov_pose_epilogue_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(acc, quat, out);
    return cov_check_launch("cov_pose_epilogue");
}

extern "C" size_t cov_pose_batch_workspace_bytes(int64_t n, int n_poses, const cov_traj_opts* opts) {
    (void)n; (void)opts;  // the pose table only: no per-point scratch on either path
    return batch_table_bytes(n_poses);
}

extern "C" int cov_pose_batch_fused(const float* xyz, int64_t n, const float* weight, const float* trans,
                                    const float* quats, int n_poses, const float* K, const cov_camera* cam,
                                    const float* boxes_dev, double* acc, const cov_traj_opts* opts, void* ws,
                                    size_t ws_bytes, void* stream) {
    if (n < 0 || (n > 0 && !xyz) || !trans || !quats || n_poses < 1 || !K || !cam || !acc || !ws) {
        cov_set_error("cov_pose_batch_fused: null pointer, negative n or no poses (n=%lld, n_poses=%d)", (long long)n,
                      n_poses);
        return COV_ERR_ARG;
    }
    if (ws_bytes < cov_pose_batch_workspace_bytes(n, n_poses, opts)) {
        cov_set_error("cov_pose_batch_fused: workspace %zu < %zu bytes", ws_bytes,
                      cov_pose_batch_workspace_bytes(n, n_poses, opts));
        return COV_ERR_WORKSPACE;
    }
    if (((uintptr_t)xyz | (uintptr_t)weight | (uintptr_t)ws | (uintptr_t)boxes_dev) & 15) {
        cov_set_error("cov_pose_batch_fused: xyz/weight/workspace/boxes must be 16-byte aligned");
        return COV_ERR_ALIGN;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    float4* table = reinterpret_cast<float4*>(ws);
    cov_pose_batch_table_kernel<<<(n_poses + 127) / 128, 128, 0, s>>>(trans, quats, n_poses, K, C, table, acc);
    const int64_t nboxes = (n + 127) / 128;
    if (nboxes > 0) {
        // slices of a chunk's poses: on a cloud with fewer boxes than resident warps, enough (box, slice) items for two
        // per warp; on a large cloud one slice (every warp walks all the chunk's poses for its box)
        const int64_t blocks_max = (int64_t)cov_sm_count_cached() * batch_min_blocks(weight != nullptr);
        const int kc = n_poses < kBatchChunk ? n_poses : kBatchChunk;
        int64_t want = (2 * blocks_max * kBatchWarps + nboxes - 1) / nboxes;
        const int nslices = (int)(want < 1 ? 1 : (want > kc ? kc : want));
        const int per_slice = (kc + nslices - 1) / nslices;
        const int64_t items = nboxes * ((kc + per_slice - 1) / per_slice);
        int64_t blocks = (items + kBatchWarps - 1) / kBatchWarps;
        if (blocks > blocks_max) blocks = blocks_max;
        const float4* boxes = (opts && opts->dense) ? nullptr : reinterpret_cast<const float4*>(boxes_dev);
        unsigned long long* stats = opts ? opts->stats_dev : nullptr;
        if (weight)
            cov_pose_batch_kernel<true><<<(int)blocks, COV_THREADS, 0, s>>>(xyz, n, weight, table, n_poses, C, boxes,
                                                                            per_slice, acc, stats);
        else
            cov_pose_batch_kernel<false><<<(int)blocks, COV_THREADS, 0, s>>>(xyz, n, weight, table, n_poses, C, boxes,
                                                                             per_slice, acc, stats);
    }
    return cov_check_launch("cov_pose_batch_fused");
}

extern "C" int cov_pose_batch_epilogue(const double* acc, const float* quats, int n_poses, float* out, void* stream) {
    if (!acc || !quats || !out || n_poses < 1) {
        cov_set_error("cov_pose_batch_epilogue: null pointer or no poses (n_poses=%d)", n_poses);
        return COV_ERR_ARG;
    }
    cov_pose_batch_epilogue_kernel<<<(n_poses + 127) / 128, 128, 0, (cudaStream_t)stream>>>(acc, quats, n_poses, out);
    return cov_check_launch("cov_pose_batch_epilogue");
}
