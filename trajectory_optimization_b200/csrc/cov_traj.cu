// cov_traj.cu — ModelTraj visibility term, fused forward+backward (reference src/model.py:200-246).
//
// Data layout: the cloud stays in HBM as row-major (N,3) fp32; the W pose rows (constants of cov_common.cuh) live
// in shared memory as 6 float4 each and are read with broadcast LDS.128; per-point state lives in registers.
//
// Two passes per objective evaluation (the min/max normalisation of src/model.py:226-227 needs the extrema first):
//   pass A  cov_traj_minmax   per pose min_j m and max_j m
//   pass B  cov_traj_fused    rewards_j = sigmoid(sum_w logit(clip(p_jw))) + the gradient accumulators
//
// Each pass exists in two forms that give bit-identical normalisers and rewards:
//
// DENSE (cov_traj_opts.dense, and every cloud below 65 536 points): every (point, pose) pair is evaluated, on packed
//   fp32 pairs — one point against TWO poses per instruction stream (cov_vis2p, FFMA2); bound by the FP32 and MUFU pipes.
//   pass A: thread-local fmin/fmax over the thread's points, one integer REDUX per warp (m >= 0, so the float order
//           is the uint order), one shared atomic per warp and 32 poses, one global atomic per block and pose.
//   pass B, per tile of 256*PPT points:
//     phase 1  every pair: m, one conservative vote per pose pair; when it passes: the exact gate (m - a >= b/2  <=>
//              p >= 0.5), warp ballots of the gate into a pose-major bit matrix in shared memory (non-zero words only),
//              gated lanes add their log-odds to the point's running sum in pose order.
//     phase 2  the bit matrix is walked pose-major: a lane owns (pose, row segment), pops its set bits, re-evaluates
//              m and dm/dx for that pair and accumulates the 8 weighted sums in registers — fixed order within a block.
//
// PRUNED (default): cull -> list -> evaluate, on boxes of 128 consecutive points (cov_tile_boxes; tight when the
//   cloud is Morton-ordered by cov_spatial_sort, valid for any order).  A pair whose distance Gaussian alone bounds m
//   below what can matter is never evaluated:  m <= 2^-(kd q2)(1+1.3e-5)  and  q2 >= box bound > qcap  =>  m < bound.
//     pass A: bound = a lower bound of max_j m from a strided sample of the cloud (seed launch), valid once the
//             minimum is known to be exactly 0 (skipped points have m >= 0);
//     pass B: bound = the conservative gate threshold (a + b/2)(1 - 2^-20): a pair below it is neither gated nor
//             the arg-max, adds logit(1/2) = 0 to the log-odds sum and nothing to the gradient.
//   cov_traj_prepare_kernel (A) / cov_traj_table_kernel (B)   pose table; A also evaluates a strided sample of the
//                        cloud (lower bounds of the maxima, which minima are exactly 0); B zeroes the accumulators
//   cov_cull_kernel      one warp per group of 8 tiles of 1024 points: the group's box, then each tile's box, then each
//                        128-point box against every pose -> a pose bit mask per listed box (a pose is listed for a
//                        box when its tile's box and its own box pass the test), and the ascending work list of the
//                        boxes with a non-empty mask, positions from a decoupled look-back scan over the blocks'
//                        counts (deterministic; no second kernel); in pass B the same blocks pre-fill the rewards with
//                        1/2 (what every unlisted point gets, exactly)
//   *_tiles_kernel       persistent WARPS (for_each_item): a warp draws listed boxes (128-point items) from a ticket
//                        counter; the next item's points and pose mask arrive by TMA bulk copy in the warp's other
//                        stage (double-buffered, one mbarrier per stage) while it works on the current one.  Every
//                        pose of the mask is evaluated (pass A first runs its per-point pre-filter).  Pass B's backward
//                        re-evaluates: the warp walks the poses it gated and recomputes m and dm/dx for its own points,
//                        with every lane busy.
//   Boxes that are not listed are never read: their rewards are the pre-filled 1/2 (exact), their sum is 0.5 * count.
//
// CANDIDATE SWEEPS (many trajectories, one cloud; pose tables of up to 2048 trajectory-major poses per launch):
//   cov_sweep_tiles_kernel        forward only: per-trajectory sum_j r_j
//   cov_sweep_fused_tiles_kernel  per trajectory, pass B's accumulators (its forward and its backward, shared with the
//                                 pass B kernel through tiles_pose_iter and tiles_pose_backward)
//
// LONG TRAJECTORIES (more poses than one box mask holds): pass B per pose chunk, the fused log-odds carried between the
//   chunks in fp32 (cov_traj_logodds_tiles_kernel<CARRY>), one finalise pass over the cloud, then the backward per chunk
//   over the kept work lists (cov_traj_long_backward_kernel).
//
// Block accumulators are added to the caller's fp64 accumulator rows with fp64 atomics (the order of those additions is
// the only thing that differs between runs: ~1e-16 relative).  The arg-max / arg-min tie sets of the normalisation
// backward are rare (one point per pose unless the minimum underflowed to 0, in which case their gradient is exactly
// negligible and skipped) and go straight to the fp64 accumulator as well.
#include <algorithm>
#include <cstdlib>
#include <map>
#include <mutex>

#include "cov_common.cuh"
#include "../../include/coverage_b200.h"

namespace {

constexpr int kWarps = COV_THREADS / 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kMaskWords = 64;   // pose bit mask of a box: covers cov_traj_max_poses() <= 2048
constexpr int kBoxPts = COV_BOX_POINTS;  // points per precomputed bounding box

__host__ __device__ constexpr int tile_points(int ppt) { return COV_THREADS * ppt; }
__host__ __device__ constexpr int bit_words(int ppt) { return kWarps * ppt; }         // ballot words per pose
__host__ __device__ constexpr int bit_stride(int ppt) { return bit_words(ppt) + 4; }  // dense rows: padded, 16-byte aligned
__host__ __device__ constexpr int tile_boxes(int ppt) { return tile_points(ppt) / kBoxPts; }
__host__ __device__ inline int mask_stride_words(int W) { return (((W + 31) >> 5) + 3) & ~3; }  // 16-byte multiple

size_t minmax_smem_bytes(int W) {  // pose pairs (COV_PAIR_F4 float4 each) + block minima and maxima
    return (size_t)((W + 1) / 2) * (COV_PAIR_F4 * sizeof(float4) + 4 * sizeof(unsigned));
}
// fused pass: pose table, then (128-byte aligned) the tile stage(s), G_j, gate bits, accumulators, gated-pose list
__host__ __device__ inline int fused_stage_offset_floats(int W) {  // W rounded up to whole pose pairs (dense kernel)
    return (int)((((size_t)((W + 1) & ~1) * COV_ROW_F4 * 16 + 127) & ~(size_t)127) / 4);
}
size_t fused_smem_bytes(int W, int ppt) {  // dense pass B: pose table | tile points | G_j | gate bits | block accumulators
    return (size_t)fused_stage_offset_floats(W) * 4 + (size_t)tile_points(ppt) * 12 + (size_t)tile_points(ppt) * 4 +
           (size_t)W * bit_stride(ppt) * sizeof(unsigned) + (size_t)W * 8 * sizeof(float);
}

// Unweighted dm/dy and dm/dy x y of one (point, pose) into a tie-set accumulator (7 doubles: F, T, count).  Rare (one
// point per pose and step), so the two entry points below are real calls; they take the pose INDEX (or its row in the
// global table) and find the constants themselves — passing loaded rows would keep them live across the callers' hot
// loops.
__device__ __forceinline__ void tie_accumulate(float x, float y, float z, const float4& v0, const float4& v1,
                                               const float4& v2, const float4& v3, const float4& v5, const CovConst& C,
                                               double* dst) {
    CovEval ev;
    const float m = cov_vis<true>(x, y, z, v0, v1, v2, v3, C, &ev);
    float gx, gy, gz;
    cov_vis_grad(m, ev, v0, v1, v2, C, gx, gy, gz);
    const float yx = x - v5.x, yy = y - v5.y, yz = z - v5.z;
    atomicAdd(dst + 0, (double)gx);
    atomicAdd(dst + 1, (double)gy);
    atomicAdd(dst + 2, (double)gz);
    atomicAdd(dst + 3, (double)(gy * yz - gz * yy));
    atomicAdd(dst + 4, (double)(gz * yx - gx * yz));
    atomicAdd(dst + 5, (double)(gx * yy - gy * yx));
    atomicAdd(dst + 6, 1.0);
}

// The dense pass B keeps its table in pose PAIRS at the start of dynamic shared memory (COV_PAIR_F4, cov_common.cuh).
__device__ __noinline__ void tie_accumulate_pair(float x, float y, float z, int w, CovConst C, double* acc, int slot) {
    extern __shared__ float4 smem4[];
    const float4* pair = smem4 + (size_t)(w >> 1) * COV_PAIR_F4;
    const int h = w & 1;
    tie_accumulate(x, y, z, cov_pair_row(pair, h, 0), cov_pair_row(pair, h, 1), cov_pair_row(pair, h, 2),
                   cov_pair_row(pair, h, 3), pair[10 + h], C, acc + slot);
}

// The pruned pass B, whose pose table stays in global memory (read through L1, a handful of rows per tile).
__device__ __noinline__ void tie_accumulate_g(float x, float y, float z, const float4* __restrict__ row, CovConst C,
                                              double* dst) {
    tie_accumulate(x, y, z, __ldg(row), __ldg(row + 1), __ldg(row + 2), __ldg(row + 3), __ldg(row + 5), C, dst);
}

// ---- pruning helpers ------------------------------------------------------------------------------------------
// Order-preserving float <-> uint map (so one integer REDUX gives a float min or max of either sign).
__device__ __forceinline__ unsigned f2ord(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
    return __uint_as_float((u & 0x80000000u) ? (u ^ 0x80000000u) : ~u);
}

// (box_q2lb, the box bound the pruned kernels test against, is in cov_common.cuh)
// Pass-A cap on q2 from the extrema seen so far (as uints): +inf (evaluate everything) unless the minimum is known
// to be exactly 0.  NaN propagates and every test against it evaluates.
__device__ __forceinline__ float minmax_qcap(unsigned mn, unsigned mx, float inv_kd) {
    float cap = __uint_as_float(0x7f800000u);
    if (mn == 0u && mx != 0u) cap = (1e-4f - __log2f(__uint_as_float(mx))) * inv_kd * 1.000001f;
    return cap;
}

// =============================================== pass A, dense ===============================================
// Every (point, pose) pair.  The evaluation runs on packed fp32 pairs (FFMA2): a thread evaluates each of its points
// against TWO poses at a time, the pose rows interleaved pairwise in shared memory (COV_PAIR_F4) so that one LDS.128
// brings two packed constants; the points are kept as broadcast pairs in registers.
template <int PPT, int MINB>
__global__ void __launch_bounds__(COV_THREADS, MINB)
cov_traj_minmax_kernel(const float* __restrict__ xyz, int64_t n, const float* __restrict__ poses,
                       const float* __restrict__ quats, int W, const float* __restrict__ K9, CovConst C,
                       unsigned* __restrict__ gmin, unsigned* __restrict__ gmax) {
    extern __shared__ float4 smem4[];
    float4* ptab = smem4;
    const int NP = (W + 1) >> 1;  // pose pairs; an odd W repeats its last pose in the spare slot
    unsigned* smin = reinterpret_cast<unsigned*>(ptab + (size_t)NP * COV_PAIR_F4);
    unsigned* smax = smin + 2 * NP;
    const int tid = threadIdx.x, lane = tid & 31;
    for (int w = tid; w < 2 * NP; w += COV_THREADS) {
        const int ws = w < W ? w : W - 1;
        float4 row[COV_ROW_F4];
        cov_pose_row(poses + 3 * ws, quats + 4 * ws, K9, C, row);
        cov_pair_store(ptab + (size_t)(w >> 1) * COV_PAIR_F4, w & 1, row);
        smin[w] = 0x7f800000u;
        smax[w] = 0u;
    }
    __syncthreads();
    const CovConst2 C2 = cov_make_const2(C);
    constexpr int T = tile_points(PPT);
    const int64_t ntiles = (n + T - 1) / T;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        f2_t X[PPT], Y[PPT], Z[PPT];
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            int64_t j = tile * T + s * COV_THREADS + tid;
            j = j < n ? j : n - 1;  // a duplicate cannot change a min or a max
            const float x = __ldg(xyz + j * 3), y = __ldg(xyz + j * 3 + 1), z = __ldg(xyz + j * 3 + 2);
            X[s] = f2_pack(x, x);
            Y[s] = f2_pack(y, y);
            Z[s] = f2_pack(z, z);
        }
        for (int p0 = 0; p0 < NP; p0 += 16) {
            // lane 2i (2i+1) keeps the warp-wide min/max of pose A (B) of pair p0+i; one shared atomic per 32 poses
            unsigned keep_mn = 0x7f800000u, keep_mx = 0u;
            const int pn = (NP - p0 < 16) ? (NP - p0) : 16;
            for (int i = 0; i < pn; ++i) {
                const float4* q = ptab + (size_t)(p0 + i) * COV_PAIR_F4;
                const float4 q0 = q[0], q1 = q[1], q2 = q[2], q3 = q[3], q4 = q[4], q5 = q[5], q6 = q[6], q7 = q[7];
                float mnA, mxA, mnB, mxB;
                f2_unpack(cov_vis2p(X[0], Y[0], Z[0], q0, q1, q2, q3, q4, q5, q6, q7, C2), mnA, mnB);
                mxA = mnA;
                mxB = mnB;
#pragma unroll
                for (int s = 1; s < PPT; ++s) {
                    float a, b;
                    f2_unpack(cov_vis2p(X[s], Y[s], Z[s], q0, q1, q2, q3, q4, q5, q6, q7, C2), a, b);
                    mnA = fminf(mnA, a); mxA = fmaxf(mxA, a);
                    mnB = fminf(mnB, b); mxB = fmaxf(mxB, b);
                }
                const unsigned umnA = __reduce_min_sync(kFull, __float_as_uint(mnA));
                const unsigned umxA = __reduce_max_sync(kFull, __float_as_uint(mxA));
                const unsigned umnB = __reduce_min_sync(kFull, __float_as_uint(mnB));
                const unsigned umxB = __reduce_max_sync(kFull, __float_as_uint(mxB));
                if (lane == 2 * i) {
                    keep_mn = umnA;
                    keep_mx = umxA;
                } else if (lane == 2 * i + 1) {
                    keep_mn = umnB;
                    keep_mx = umxB;
                }
            }
            if (lane < 2 * pn) {
                atomicMin(smin + 2 * p0 + lane, keep_mn);
                atomicMax(smax + 2 * p0 + lane, keep_mx);
            }
        }
    }
    __syncthreads();
    for (int w = tid; w < W; w += COV_THREADS) {
        atomicMin(gmin + w, smin[w]);
        atomicMax(gmax + w, smax[w]);
    }
}

__global__ void cov_minmax_init_kernel(unsigned* gmin, unsigned* gmax, int W) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w < W) {
        gmin[w] = 0x7f800000u;
        gmax[w] = 0u;
    }
}

// ============================================ pruned passes: set-up ============================================
// Control words of one pruned call, at the head of the workspace (zeroed once per call: by a memset node in pass A,
// by cov_traj_table_kernel in pass B):
//   ctrl[0] work-list length (listed boxes)   ctrl[1] some pose has min_j m > 0   ctrl[2] block ticket of the
//   evaluation kernel   ctrl[3] its item ticket
//   ctrl[4..5] (box, pose) pairs of the poses the cull listed per tile, all 8 boxes of a tile (u64; work counter [6])
//   ctrl[6..7] the same over the boxes inside the cloud (u64; work counter [7])
//   ctrl[8..9] boxes of listed tiles that no pose reaches at box level (u64)
//   enc[0..W)  ~bits(min_j m)   enc[W..2W) bits(max_j m)   pass A's extrema in an encoding whose neutral element is 0:
//              m >= +0, so the unsigned order of the bits is the float order; both are kept with atomicMax
//   desc[c]    look-back descriptor of cull chunk c (status in the top two bits)
constexpr int kCtrlInts = 16;
constexpr unsigned long long kDescAgg = 1ull << 62, kDescPrefix = 2ull << 62, kDescValue = (1ull << 62) - 1;
constexpr int kChunkTiles = 64;  // tiles per cull block iteration (8 warps x 8 tiles) = one look-back descriptor

__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Pass A, first launch: pose table + seed.  Grid = (sample blocks) x (chunks of 32 poses).  The first 32 threads of a
// block build the chunk's pose rows in shared memory (fp64 inside; blocks of the first grid column also store them to
// the global table the later kernels copy), then every thread evaluates ONE point of a strided sample of the cloud
// against the 32 poses (dense), so that the cull starts from a good lower bound of each maximum and knows which
// minima are exactly 0.  Per pose one REDUX pair per warp, the 8 warps meet in shared memory, 64 global atomics per
// block into the zero-initialised encoded extrema.
__global__ void __launch_bounds__(COV_THREADS)
cov_traj_prepare_kernel(const float* __restrict__ xyz, int64_t nsamples, int64_t stride, const float* __restrict__ poses,
                        const float* __restrict__ quats, int W, const float* __restrict__ K9, CovConst C,
                        float4* __restrict__ table, unsigned* __restrict__ enc) {
    __shared__ float4 rows[32 * COV_ROW_F4];
    __shared__ unsigned smn[32], smx[32];
    const int tid = threadIdx.x, lane = tid & 31;
    const int w0 = blockIdx.y * 32;
    const int wn = (W - w0 < 32) ? (W - w0) : 32;
    if (tid < wn) {
        cov_pose_row(poses + 3 * (w0 + tid), quats + 4 * (w0 + tid), K9, C, rows + tid * COV_ROW_F4);
        if (blockIdx.x == 0) {
#pragma unroll
            for (int i = 0; i < COV_ROW_F4; ++i) table[(size_t)(w0 + tid) * COV_ROW_F4 + i] = rows[tid * COV_ROW_F4 + i];
        }
        smn[tid] = 0x7f800000u;
        smx[tid] = 0u;
    }
    __syncthreads();
    int64_t j = (int64_t)blockIdx.x * COV_THREADS + tid;
    j = (j < nsamples ? j : nsamples - 1) * stride;  // a duplicate cannot change a min or a max
    const float x = __ldg(xyz + j * 3), y = __ldg(xyz + j * 3 + 1), z = __ldg(xyz + j * 3 + 2);
    unsigned keep_mn = 0x7f800000u, keep_mx = 0u;
    for (int i = 0; i < wn; ++i) {
        const float4* r = rows + i * COV_ROW_F4;
        const float m = cov_vis<false>(x, y, z, r[0], r[1], r[2], r[3], C, nullptr);
        const unsigned umn = __reduce_min_sync(kFull, __float_as_uint(m));
        const unsigned umx = __reduce_max_sync(kFull, __float_as_uint(m));
        if (lane == i) {
            keep_mn = umn;
            keep_mx = umx;
        }
    }
    if (lane < wn) {
        atomicMin(smn + lane, keep_mn);
        atomicMax(smx + lane, keep_mx);
    }
    __syncthreads();
    if (tid < wn) {
        atomicMax(enc + w0 + tid, ~smn[tid]);
        atomicMax(enc + W + w0 + tid, smx[tid]);
    }
}

// Pass B, first launch: block 0 zeroes the control words, the look-back descriptors and the caller's accumulator rows
// (acc[W * STRIDE] starts at `sum_base` = 0.5 * n: what the unlisted points add to the reward sum) and sets ctrl[1] when
// some pose has min_j m > 0; every block builds 64 rows of the pose table with the normalisation constants:
// v3.w = qthr, v4 = (b/2, b, 1/b, a), v5.w = thr.
// SUM_DEV: the sum starts at *sum_base_dev instead (sum_j sigmoid(prior_j), cov_prior_reward_sum).
// LONG (cov_traj_fused_long): the W poses are the chunk [w0, w0 + W) of a call over w_all poses; `poses`, `quats`, `table`
// and `acc` point at the chunk's first pose, `minmax` is the call's [w_all minima | w_all maxima].  Only the chunk's
// accumulator rows are zeroed, and the reward-sum slot acc[(w_all - w0) * STRIDE] is set by the chunk with w0 = 0 alone.
template <bool SUM_DEV, bool LONG = false>
__global__ void __launch_bounds__(64)
cov_traj_table_kernel(const float* __restrict__ poses, const float* __restrict__ quats, int W,
                      const float* __restrict__ K9, CovConst C, const float* __restrict__ minmax,
                      float4* __restrict__ table, int* __restrict__ ctrl, int ctrl_words, double* __restrict__ acc,
                      double sum_base, const double* __restrict__ sum_base_dev, int w0 = 0, int w_all = 0) {
    const int tid = threadIdx.x;
    if (blockIdx.x == 0) {
        int amin = 0;
        for (int w = tid; w < W; w += blockDim.x) amin |= (LONG ? minmax[w0 + w] : minmax[w]) > 0.f;
        amin = __syncthreads_or(amin);
        for (int i = tid; i < ctrl_words; i += blockDim.x) ctrl[i] = (i == 1) ? amin : 0;
        if (acc) {
            for (int i = tid; i < W * COV_ACC_STRIDE; i += blockDim.x) acc[i] = 0.0;
            if (tid == 0 && (!LONG || w0 == 0)) acc[(size_t)(LONG ? w_all : W) * COV_ACC_STRIDE] = SUM_DEV ? *sum_base_dev : sum_base;
        }
    }
    const int w = blockIdx.x * blockDim.x + tid;
    if (w >= W) return;
    float4 row[COV_ROW_F4];
    cov_pose_row(poses + 3 * w, quats + 4 * w, K9, C, row);
    const float a = LONG ? minmax[w0 + w] : minmax[w];
    float thr;
    cov_norm_row(row, a, LONG ? minmax[w_all + w0 + w] : minmax[W + w], thr);
    row[5].w = thr;
    // q2 above qthr cannot reach thr (thr <= 0 or NaN, or a > 0 — arg-min points carry gradient: never prune)
    row[3].w = (thr > 0.f && !(a > 0.f)) ? (float)((1e-4 - log2((double)thr)) / (double)C.kd * 1.000001)
                                         : __uint_as_float(0x7f800000u);
#pragma unroll
    for (int i = 0; i < COV_ROW_F4; ++i) table[(size_t)w * COV_ROW_F4 + i] = row[i];
}

// Bounding boxes of runs of kBoxPts consecutive points: boxes[2b] = (lo, 0), boxes[2b+1] = (hi, 0); boxes past the
// end of the cloud are empty (+inf, -inf).  One warp per box.
__global__ void __launch_bounds__(256) cov_tile_boxes_kernel(const float* __restrict__ xyz, int64_t n, int64_t nboxes,
                                                             float4* __restrict__ boxes) {
    const float inf = __uint_as_float(0x7f800000u);
    const int lane = threadIdx.x & 31;
    for (int64_t b = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); b < nboxes; b += (int64_t)gridDim.x * 8) {
        float lx = inf, ly = inf, lz = inf, hx = -inf, hy = -inf, hz = -inf;
#pragma unroll
        for (int s = 0; s < kBoxPts / 32; ++s) {
            const int64_t j = b * kBoxPts + s * 32 + lane;
            if (j < n) {
                const float x = __ldg(xyz + j * 3), y = __ldg(xyz + j * 3 + 1), z = __ldg(xyz + j * 3 + 2);
                lx = fminf(lx, x); ly = fminf(ly, y); lz = fminf(lz, z);
                hx = fmaxf(hx, x); hy = fmaxf(hy, y); hz = fmaxf(hz, z);
            }
        }
        const unsigned ulx = __reduce_min_sync(kFull, f2ord(lx)), uly = __reduce_min_sync(kFull, f2ord(ly));
        const unsigned ulz = __reduce_min_sync(kFull, f2ord(lz)), uhx = __reduce_max_sync(kFull, f2ord(hx));
        const unsigned uhy = __reduce_max_sync(kFull, f2ord(hy)), uhz = __reduce_max_sync(kFull, f2ord(hz));
        if (lane == 0) {
            boxes[2 * b] = make_float4(ord2f(ulx), ord2f(uly), ord2f(ulz), 0.f);
            boxes[2 * b + 1] = make_float4(ord2f(uhx), ord2f(uhy), ord2f(uhz), 0.f);
        }
    }
}

// Cull + work list.  The work list holds the indices of the LISTED BOXES (128 points each) in ascending order, and
// mask[b][c] bit i <=> pose 32c+i is to be evaluated on box b (masks are indexed by box and written for listed boxes
// only).  The predicate is two-level: a pose is listed for a 1024-point tile when the tile's box passes the test, and
// evaluated on a box of that tile when the box's own box passes it too (`!(box_q2lb(lo, hi, v3) > cap)`, a NaN cap
// evaluates).  One warp per GROUP of 8 consecutive tiles (64 boxes): every pose is tested against the group's box
// first (one lane per pose); for each pose that passes, lane l tests tile l & 7 (one ballot gives the 8 tiles' bits) and
// its own two boxes, in-group boxes l and 32 + l (tiles l >> 3 and 4 + (l >> 3)), so a lane ends a pose word holding
// that word of its two boxes' masks and stores it once the box is known to be listed.  Pass A passes `enc` (after the
// prepare launch) and the cap is derived here; pass B reads qthr from the table.
// A block iteration covers a CHUNK of 64 consecutive tiles; the block first culls ALL its chunks (warps independent, no
// barrier), then appends each chunk's listed boxes to the work list in ascending order: the chunk's offset is the
// exclusive prefix sum of the chunks' counts, obtained with a decoupled look-back over per-chunk descriptors (publish
// the own aggregates, then sum predecessors until one carries an inclusive prefix).  The list is a pure function of the
// boxes and the caps (deterministic).  Grid <= resident capacity, and every block publishes its aggregates before it
// waits for anybody's, so every predecessor a block waits for has been (or is being) published.  `fill_dst` (pass B):
// the same blocks write 1/2 to every reward (HAS_PRIOR: sigmoid(prior_i), with pass B's expression).
// Counts for the work counters (ctrl[4..9], u64 each): (box, pose) pairs of the poses listed per tile, over all 8 boxes
// of the tile and over the boxes inside the cloud, and the boxes of listed tiles that no pose reaches.
constexpr int kCullMaxIter = 32;  // chunks per block at most (the host sizes the grid accordingly)
constexpr int kTileBoxes = 8;     // 128-point boxes per 1024-point tile of the pruned passes

// One warp's group of 8 tiles as the cull sees it from lane l: its boxes l and 32 + l, the box of tile l & 7 and the
// group's box.  Boxes of tiles past `ntiles` are empty and never listed.
struct CullGroup {
    float4 lo[2], hi[2];  // the lane's two boxes
    float4 tlo, thi;      // the box of tile l & 7
    float4 glo, ghi;      // the group's box
    bool tile_ok;         // tile l & 7 is < ntiles
    int tile_in;          // its boxes inside the cloud (0..8)
};

__device__ __forceinline__ void box_shfl_union(float4& lo, float4& hi, int o) {
    lo.x = fminf(lo.x, __shfl_xor_sync(kFull, lo.x, o)); lo.y = fminf(lo.y, __shfl_xor_sync(kFull, lo.y, o));
    lo.z = fminf(lo.z, __shfl_xor_sync(kFull, lo.z, o)); hi.x = fmaxf(hi.x, __shfl_xor_sync(kFull, hi.x, o));
    hi.y = fmaxf(hi.y, __shfl_xor_sync(kFull, hi.y, o)); hi.z = fmaxf(hi.z, __shfl_xor_sync(kFull, hi.z, o));
}

__device__ __forceinline__ CullGroup cull_group_load(const float4* __restrict__ boxes, int64_t group, int64_t ntiles,
                                                     int64_t n, int lane) {
    const float inf = __uint_as_float(0x7f800000u);
    CullGroup g;
    float4 tlo[2], thi[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int64_t box = group * (8 * kTileBoxes) + s * 32 + lane;
        g.lo[s] = make_float4(inf, inf, inf, 0.f);
        g.hi[s] = make_float4(-inf, -inf, -inf, 0.f);
        if (box < ntiles * kTileBoxes) {
            g.lo[s] = boxes[box * 2];
            g.hi[s] = boxes[box * 2 + 1];
        }
        tlo[s] = g.lo[s];
        thi[s] = g.hi[s];
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) box_shfl_union(tlo[s], thi[s], o);  // lanes 8g..8g+7: tile g (s = 0), 4 + g (s = 1)
    }
    const int t = lane & 7, src = (t & 3) << 3;  // lane l takes tile l & 7 from lane 8 (t mod 4), slot t / 4
    float4 a_lo, a_hi, b_lo, b_hi;
    a_lo.x = __shfl_sync(kFull, tlo[0].x, src); a_lo.y = __shfl_sync(kFull, tlo[0].y, src); a_lo.z = __shfl_sync(kFull, tlo[0].z, src);
    a_hi.x = __shfl_sync(kFull, thi[0].x, src); a_hi.y = __shfl_sync(kFull, thi[0].y, src); a_hi.z = __shfl_sync(kFull, thi[0].z, src);
    b_lo.x = __shfl_sync(kFull, tlo[1].x, src); b_lo.y = __shfl_sync(kFull, tlo[1].y, src); b_lo.z = __shfl_sync(kFull, tlo[1].z, src);
    b_hi.x = __shfl_sync(kFull, thi[1].x, src); b_hi.y = __shfl_sync(kFull, thi[1].y, src); b_hi.z = __shfl_sync(kFull, thi[1].z, src);
    g.tlo = t < 4 ? a_lo : b_lo;
    g.thi = t < 4 ? a_hi : b_hi;
    g.tlo.w = g.thi.w = 0.f;
    g.glo = g.tlo;
    g.ghi = g.thi;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) box_shfl_union(g.glo, g.ghi, o);  // the 8 tiles
    const int64_t tile = group * 8 + t;
    g.tile_ok = tile < ntiles;
    const int64_t rest = n - tile * (kTileBoxes * kBoxPts);
    g.tile_in = rest <= 0 ? 0 : (rest >= kTileBoxes * kBoxPts ? kTileBoxes : (int)((rest + kBoxPts - 1) / kBoxPts));
    return g;
}

template <bool HAS_PRIOR>
__global__ void __launch_bounds__(256, 5)
cov_cull_kernel(const float4* __restrict__ boxes, int64_t n, int64_t ntiles, const float4* __restrict__ table,
                int W, const unsigned* __restrict__ enc, float inv_kd, unsigned* __restrict__ amask_g, int mask_stride,
                int* __restrict__ worklist, int* __restrict__ ctrl, unsigned long long* __restrict__ desc,
                float* __restrict__ fill_dst, int64_t fill_n, const float* __restrict__ fill_prior) {
    extern __shared__ float4 v3s[];
    __shared__ unsigned long long listed_s[kCullMaxIter][8];  // per own chunk and warp: which of its 64 boxes are listed
    __shared__ int chunk_base[kCullMaxIter];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int w = tid; w < W; w += blockDim.x) {
        float4 v3 = table[(size_t)w * COV_ROW_F4 + 3];
        if (enc) v3.w = minmax_qcap(~enc[w], enc[W + w], inv_kd);
        v3s[w] = v3;
    }
    if (fill_dst) {  // fire-and-forget stores: they drain while the blocks cull
        const int64_t stride = (int64_t)gridDim.x * blockDim.x * 4;
        for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + tid) * 4; i < fill_n; i += stride) {
            if (HAS_PRIOR) {
                if (i + 4 <= fill_n && ((reinterpret_cast<uintptr_t>(fill_dst + i) & 15) == 0) &&
                    ((reinterpret_cast<uintptr_t>(fill_prior + i) & 15) == 0)) {
                    __stcs(reinterpret_cast<float4*>(fill_dst + i), cov_sigmoid4(__ldcs(reinterpret_cast<const float4*>(fill_prior + i))));
                } else {
                    for (int64_t k = i; k < fill_n && k < i + 4; ++k) fill_dst[k] = cov_sigmoid(fill_prior[k]);
                }
            } else if (i + 4 <= fill_n && ((reinterpret_cast<uintptr_t>(fill_dst + i) & 15) == 0)) {
                __stcs(reinterpret_cast<float4*>(fill_dst + i), make_float4(0.5f, 0.5f, 0.5f, 0.5f));
            } else {
                for (int64_t k = i; k < fill_n && k < i + 4; ++k) fill_dst[k] = 0.5f;
            }
        }
    }
    __syncthreads();
    const int64_t nchunks = (ntiles + kChunkTiles - 1) / kChunkTiles;
    const int nwords = (W + 31) >> 5;
    unsigned pairs_all = 0, pairs_in = 0, n_empty = 0;  // per lane: at most kCullMaxIter * 8 * 2048 pairs
    int it = 0;
    for (int64_t chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x, ++it) {
        const int64_t group = chunk * 8 + warp;
        const CullGroup g = cull_group_load(boxes, group, ntiles, n, lane);
        // the mask rows of the lane's two boxes: mrow and mrow + 32 * mask_stride
        unsigned* mrow = amask_g + (size_t)(group * (8 * kTileBoxes) + lane) * mask_stride;
        int first[2] = {-1, -1};  // first non-zero word of the box's mask: the box is listed, its words are stored
        unsigned tany = 0u;       // lanes 0..7: poses listed for tile l & 7
        for (int c = 0; c < mask_stride; ++c) {
            const int w = c * 32 + lane;
            bool cand = false;
            if (c < nwords && w < W) {
                const float4 v3 = v3s[w];
                cand = !(box_q2lb(g.glo, g.ghi, v3) > v3.w);  // NaN cap: evaluate
            }
            unsigned gword = __ballot_sync(kFull, cand);
            unsigned bm[2] = {0u, 0u}, tm = 0u;
            while (gword) {
                const int b = __ffs(gword) - 1;
                gword &= gword - 1;
                const float4 v3 = v3s[c * 32 + b];
                const bool th = g.tile_ok && !(box_q2lb(g.tlo, g.thi, v3) > v3.w);  // an empty box gives +inf
                const unsigned tb = __ballot_sync(kFull, th);  // bit t (t < 8): tile t lists the pose
                tm |= (unsigned)th << b;
                if (tb == 0u) continue;
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    const bool hit = ((tb >> (s * 4 + (lane >> 3))) & 1u) && !(box_q2lb(g.lo[s], g.hi[s], v3) > v3.w);
                    bm[s] |= (unsigned)hit << b;
                }
            }
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                if (first[s] < 0 && bm[s] != 0u) first[s] = c;
                if (first[s] >= 0) mrow[s * 32 * mask_stride + c] = bm[s];
            }
            if (lane < 8) {
                pairs_all += (unsigned)kTileBoxes * __popc(tm);
                pairs_in += (unsigned)g.tile_in * __popc(tm);
                tany |= tm;
            }
        }
#pragma unroll
        for (int s = 0; s < 2; ++s)
            for (int c = 0; c < first[s]; ++c) mrow[s * 32 * mask_stride + c] = 0u;  // the words before the first non-zero one
        const unsigned tl8 = __ballot_sync(kFull, lane < 8 && tany != 0u);  // listed tiles
#pragma unroll
        for (int s = 0; s < 2; ++s) n_empty += ((tl8 >> (s * 4 + (lane >> 3))) & 1u) && first[s] < 0;
        const unsigned l0 = __ballot_sync(kFull, first[0] >= 0), l1 = __ballot_sync(kFull, first[1] >= 0);
        if (lane == 0) listed_s[it][warp] = ((unsigned long long)l1 << 32) | l0;
    }
    const int n_it = it;
    __syncthreads();
    if (warp == 0) {
        // own chunk `k` is chunk blockIdx.x + k * gridDim.x; listed_s[k][q] = the listed boxes of its warp q
        for (int k = lane; k < n_it; k += 32) {  // publish every own aggregate first
            int total = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) total += __popcll(listed_s[k][q]);
            const int64_t chunk = blockIdx.x + (int64_t)k * gridDim.x;
            if (chunk > 0) st_release_u64(desc + chunk, kDescAgg | (unsigned long long)total);
        }
        __syncwarp();
        for (int k = 0; k < n_it; ++k) {
            const int64_t chunk = blockIdx.x + (int64_t)k * gridDim.x;
            unsigned long long total = 0ull;
#pragma unroll
            for (int q = 0; q < 8; ++q) total += (unsigned long long)__popcll(listed_s[k][q]);
            unsigned long long excl = 0ull;
            if (chunk > 0) {
                int64_t look = chunk - 1;
                while (true) {  // windows of 32 predecessors, nearest first
                    const int64_t idx = look - lane;
                    unsigned long long d = kDescPrefix;  // before chunk 0: an inclusive prefix of 0
                    if (idx >= 0) d = ld_acquire_u64(desc + idx);
                    const unsigned empty = __ballot_sync(kFull, (d >> 62) == 0ull);
                    const unsigned pref = __ballot_sync(kFull, (d >> 62) == 2ull);
                    const int first_pref = pref ? (__ffs(pref) - 1) : 32;
                    const unsigned need = first_pref >= 31 ? kFull : ((2u << first_pref) - 1u);
                    if (empty & need) continue;  // a predecessor in the window has not published yet: look again
                    unsigned long long v = (lane <= first_pref) ? (d & kDescValue) : 0ull;
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
                    excl += v;
                    if (first_pref < 32) break;
                    look -= 32;
                }
            }
            if (lane == 0) {
                st_release_u64(desc + chunk, kDescPrefix | (excl + total));
                if (chunk == nchunks - 1) ctrl[0] = (int)(excl + total);
                chunk_base[k] = (int)excl;
            }
        }
    }
    __syncthreads();
    // the listed boxes of each own chunk at their list positions
    for (int k = 0; k < n_it; ++k) {
        const unsigned long long listed = listed_s[k][warp];
        if (listed == 0ull) continue;
        const int64_t chunk = blockIdx.x + (int64_t)k * gridDim.x;
        int pos = chunk_base[k];  // listed boxes of the chunk in the warps ahead of this one
        for (int q = 0; q < warp; ++q) pos += __popcll(listed_s[k][q]);
        const unsigned below = (1u << lane) - 1u;
        const unsigned l0 = (unsigned)listed, l1 = (unsigned)(listed >> 32);
        const int64_t box0 = (chunk * 8 + warp) * (8 * kTileBoxes) + lane;
        if ((l0 >> lane) & 1u) worklist[pos + __popc(l0 & below)] = (int)box0;
        if ((l1 >> lane) & 1u) worklist[pos + __popc(l0) + __popc(l1 & below)] = (int)(box0 + 32);
    }
    pairs_all = __reduce_add_sync(kFull, pairs_all);
    pairs_in = __reduce_add_sync(kFull, pairs_in);
    n_empty = __reduce_add_sync(kFull, n_empty);
    if (lane == 0) {
        if (pairs_all) atomicAdd(reinterpret_cast<unsigned long long*>(ctrl + 4), (unsigned long long)pairs_all);
        if (pairs_in) atomicAdd(reinterpret_cast<unsigned long long*>(ctrl + 6), (unsigned long long)pairs_in);
        if (n_empty) atomicAdd(reinterpret_cast<unsigned long long*>(ctrl + 8), (unsigned long long)n_empty);
    }
}

// ================================= pruned evaluation: the persistent-warp item loop =================================
// The *_tiles_kernel below run persistent WARPS over the work list.  The unit of work is one listed box of 128
// consecutive points, taken by ONE WARP from a global ticket counter: warps never wait for each other (no block barrier,
// no static assignment), so neither the uneven cost of neighbouring boxes nor a heavy box at the end of the list leaves
// lanes idle.  A warp keeps two private stages in shared memory; its lane 0 draws the next ticket and issues the TMA bulk
// copies for it (points, the box's pose mask, and in pass B the slice of the permutation — one mbarrier per stage)
// before the warp starts on the current item.  Every pose of the mask is evaluated: the cull has already tested it
// against the box.  The pose table stays in global memory (a box touches ~5 rows: L1 hits).
constexpr int kItemPts = 128;                 // points per work item = one warp's registers = one precomputed box
constexpr int kItemPpt = kItemPts / 32;
static_assert(kItemPts == kBoxPts, "a work item is one box");

// One work item as the loop body sees it: points [j0, j0 + 128) of the cloud.
struct Item {
    int64_t j0;
    bool whole;             // j0 + 128 <= n: the points (and the permutation slice) were staged
    const float* pts;       // the staged points, xyz interleaved
    const unsigned* mask;   // the box's pose mask: the poses to evaluate
    const int32_t* perm;    // the staged slice of the permutation (WITH_PERM, whole, permutation given)
};

// Draws items until the work list is exhausted; `pre_wait(it)` runs after the next item was issued and before the wait
// for the current one, `body(item)` once the current one has arrived.  Every lane of the warp calls it.
template <bool WITH_PERM, typename PreWait, typename Body>
__device__ __forceinline__ void for_each_item(const float* __restrict__ xyz, int64_t n,
                                              const unsigned* __restrict__ amask_g, int mask_stride,
                                              const int32_t* __restrict__ perm, const int* __restrict__ worklist,
                                              int n_items, int* ticket, PreWait pre_wait, Body body) {
    constexpr int kStageWords = kItemPts * 3 + kMaskWords + (WITH_PERM ? kItemPts : 0);  // points|mask|perm
    __shared__ __align__(128) float stages[kWarps][2][kStageWords];
    __shared__ __align__(8) unsigned long long mbar[kWarps][2];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long* bar = mbar[warp];
    if (lane == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_fence_init();
    }
    __syncwarp();
    // lane 0: stage item `it` (box worklist[it] and its mask row); a ragged item's points are loaded by hand
    auto issue = [&](int it, int b) {
        if (it >= n_items) return;
        const int64_t box = worklist[it];
        const int64_t j0 = box * kItemPts;
        float* st = stages[warp][b];
        const bool whole = j0 + kItemPts <= n;
        const bool with_perm = WITH_PERM && whole && perm != nullptr;
        mbar_expect_tx(&bar[b], (whole ? kItemPts * 12u : 0u) + (unsigned)mask_stride * 4u + (with_perm ? kItemPts * 4u : 0u));
        if (whole) tma_copy(st, xyz + j0 * 3, kItemPts * 12u, &bar[b]);
        tma_copy(st + kItemPts * 3, amask_g + box * mask_stride, (unsigned)mask_stride * 4u, &bar[b]);
        if (with_perm) tma_copy(st + kItemPts * 3 + kMaskWords, perm + j0, kItemPts * 4u, &bar[b]);
    };
    unsigned uses0 = 0, uses1 = 0;
    int cur = 0;
    if (lane == 0) {
        cur = atomicAdd(ticket, 1);
        issue(cur, 0);
    }
    cur = __shfl_sync(kFull, cur, 0);
    int buf = 0;
    while (cur < n_items) {
        int nxt = 0;
        if (lane == 0) {  // the other stage was last read before the __syncwarp that ended the previous item
            nxt = atomicAdd(ticket, 1);
            issue(nxt, buf ^ 1);
        }
        nxt = __shfl_sync(kFull, nxt, 0);
        pre_wait(cur);
        if (buf == 0) mbar_wait(&bar[0], uses0++ & 1u);
        else mbar_wait(&bar[1], uses1++ & 1u);
        const float* st = stages[warp][buf];
        Item item;
        item.j0 = (int64_t)worklist[cur] * kItemPts;
        item.whole = item.j0 + kItemPts <= n;
        item.pts = st;
        item.mask = reinterpret_cast<const unsigned*>(st + kItemPts * 3);
        item.perm = reinterpret_cast<const int32_t*>(st + kItemPts * 3 + kMaskWords);
        body(item);
        __syncwarp();  // every lane is done with this stage before lane 0 refills it
        cur = nxt;
        buf ^= 1;
    }
}

// The item's points into registers, point s * 32 + lane in slot s: from the stage, or by hand at the ragged end of the
// cloud, where the slots past the end get one of two fillers that are not interchangeable:
//   CLAMP   point n - 1 again (pass A: a duplicate cannot change a min or a max; a sentinel would make the min 0)
//   !CLAMP  a point 3e18 m away, valid = false (pass B, sweep: m = 0 exactly, never gated, never a tie; a duplicate
//           would be counted twice)
template <bool CLAMP>
__device__ __forceinline__ void load_item_points(const Item& item, const float* __restrict__ xyz, int64_t n, int lane,
                                                 float (&px)[kItemPpt], float (&py)[kItemPpt], float (&pz)[kItemPpt],
                                                 bool (&valid)[kItemPpt]) {
    if (item.whole) {
#pragma unroll
        for (int s = 0; s < kItemPpt; ++s) {
            valid[s] = true;
            px[s] = item.pts[(s * 32 + lane) * 3];
            py[s] = item.pts[(s * 32 + lane) * 3 + 1];
            pz[s] = item.pts[(s * 32 + lane) * 3 + 2];
        }
    } else {
#pragma unroll
        for (int s = 0; s < kItemPpt; ++s) {
            const int64_t j = item.j0 + s * 32 + lane;
            valid[s] = j < n;
            if (CLAMP) {
                const int64_t jc = valid[s] ? j : n - 1;
                px[s] = __ldg(xyz + jc * 3);
                py[s] = __ldg(xyz + jc * 3 + 1);
                pz[s] = __ldg(xyz + jc * 3 + 2);
            } else {
                px[s] = valid[s] ? __ldg(xyz + j * 3) : 3.0e18f;
                py[s] = valid[s] ? __ldg(xyz + j * 3 + 1) : 3.0e18f;
                pz[s] = valid[s] ? __ldg(xyz + j * 3 + 2) : 3.0e18f;
            }
        }
    }
}

// =============================================== pass A, pruned ===============================================
// A pose of the box's mask (the cull tested the cap ball from the seed's extrema against the box) is evaluated when the
// cap ball meets one of the box's points; the cap is re-read from the extrema at start-up (any later value is tighter
// and valid).  Extrema meet per block in shared memory, then in the zero-initialised encoded arrays; the last block
// decodes them into the caller's floats.
template <bool HAS_PRIOR>
__global__ void __launch_bounds__(COV_THREADS, 3)
cov_traj_minmax_tiles_kernel(const float* __restrict__ xyz, int64_t n, const float4* __restrict__ table, int W, CovConst C,
                             unsigned* __restrict__ enc, float* __restrict__ minmax_out,
                             const unsigned* __restrict__ amask_g, int mask_stride, const int* __restrict__ worklist,
                             int* __restrict__ ctrl, int64_t ntiles, unsigned long long* __restrict__ stats,
                             float* __restrict__ fill_dst, int64_t fill_n, const float* __restrict__ fill_prior) {
    constexpr int PPT = kItemPpt;
    extern __shared__ float4 smem4[];                      // block minima | maxima (uint) | per-pose caps
    unsigned* smin = reinterpret_cast<unsigned*>(smem4);
    unsigned* smax = smin + W;
    float* sqcap = reinterpret_cast<float*>(smax + W);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float inv_kd = 1.f / C.kd;
    for (int w = tid; w < W; w += COV_THREADS) {
        smin[w] = 0x7f800000u;
        smax[w] = 0u;
        sqcap[w] = minmax_qcap(~enc[w], enc[W + w], inv_kd);  // from the seed (any later value is tighter and valid)
    }
    __syncthreads();
    const int n_items = ctrl[0];
    const int nwords = (W + 31) >> 5;
    // Pre-fill of pass B's rewards with 1/2 under this kernel's idle memory bandwidth (cov_traj_opts.prefill_dev): the
    // warp that takes item i also writes slice i of the buffer (fire-and-forget streaming stores), in 16-byte units.
    // HAS_PRIOR: sigmoid(prior_i) instead, from streaming 16-byte loads of the prior (same index as the buffer).
    const int64_t fill_q = (fill_n + 3) / 4;                                          // float4 slots (tail handled below)
    const int64_t fill_per_item = fill_dst ? (fill_q + (n_items > 0 ? n_items : 1) - 1) / (n_items > 0 ? n_items : 1) : 0;
    auto fill_slice = [&](int64_t q0, int64_t q1) {
        if (q1 > fill_q) q1 = fill_q;
        for (int64_t q = q0 + lane; q < q1; q += 32) {
            if (HAS_PRIOR) {
                if (q * 4 + 4 <= fill_n)
                    __stcs(reinterpret_cast<float4*>(fill_dst) + q, cov_sigmoid4(__ldcs(reinterpret_cast<const float4*>(fill_prior) + q)));
                else for (int64_t k = q * 4; k < fill_n; ++k) fill_dst[k] = cov_sigmoid(fill_prior[k]);
            } else if (q * 4 + 4 <= fill_n) {
                __stcs(reinterpret_cast<float4*>(fill_dst) + q, make_float4(0.5f, 0.5f, 0.5f, 0.5f));
            } else {
                for (int64_t k = q * 4; k < fill_n; ++k) fill_dst[k] = 0.5f;
            }
        }
    };
    if (fill_dst && n_items == 0) {  // nothing listed: the warps of the grid share the whole buffer
        const int64_t gw = (int64_t)blockIdx.x * kWarps + warp, nw = (int64_t)gridDim.x * kWarps;
        const int64_t per = (fill_q + nw - 1) / nw;
        fill_slice(gw * per, (gw + 1) * per);
    }
    unsigned n_pre = 0, n_full = 0;
    auto fill_item = [&](int it) {
        if (fill_dst) fill_slice((int64_t)it * fill_per_item, (int64_t)(it + 1) * fill_per_item);
    };
    for_each_item<false>(xyz, n, amask_g, mask_stride, nullptr, worklist, n_items, ctrl + 3, fill_item,
                         [&](const Item& item) {
        float px[PPT], py[PPT], pz[PPT];
        bool valid[PPT];
        load_item_points<true>(item, xyz, n, lane, px, py, pz, valid);
        if (item.j0 >= n) return;  // a listed box past the end of the cloud (an empty box under an infinite cap)
        for (int c = 0; c < nwords; ++c) {
            unsigned word = item.mask[c];
            while (word) {
                const int w = c * 32 + __ffs(word) - 1;
                word &= word - 1;
                const float4* row = table + (size_t)w * COV_ROW_F4;
                const float4 v3 = __ldg(row + 3);
                const float cap = sqcap[w];
                ++n_pre;
                float qmin = cov_q2(px[0], py[0], pz[0], v3);
#pragma unroll
                for (int s = 1; s < PPT; ++s) qmin = fminf(qmin, cov_q2(px[s], py[s], pz[s], v3));
                if (!__any_sync(kFull, !(qmin > cap))) continue;
                ++n_full;
                const float4 v0 = __ldg(row), v1 = __ldg(row + 1), v2 = __ldg(row + 2);
                float m[PPT];
#pragma unroll
                for (int s = 0; s < PPT; ++s) m[s] = cov_vis<false>(px[s], py[s], pz[s], v0, v1, v2, v3, C, nullptr);
                float mn = m[0], mx = m[0];
#pragma unroll
                for (int s = 1; s < PPT; ++s) {
                    mn = fminf(mn, m[s]);
                    mx = fmaxf(mx, m[s]);
                }
                const unsigned umn = __reduce_min_sync(kFull, __float_as_uint(mn));
                const unsigned umx = __reduce_max_sync(kFull, __float_as_uint(mx));
                if (lane == 0) {
                    atomicMin(smin + w, umn);
                    atomicMax(smax + w, umx);
                }
            }
        }
    });
    __syncthreads();
    for (int w = tid; w < W; w += COV_THREADS) {
        if (smax[w] != 0u || smin[w] != 0x7f800000u) {
            atomicMax(enc + w, ~smin[w]);
            atomicMax(enc + W + w, smax[w]);
        }
    }
    if (stats && lane == 0) {
        if (tid == 0 && blockIdx.x == 0) {
            atomicAdd(stats + 2, (unsigned long long)ntiles * kWarps * W);
            atomicAdd(stats + 7, *reinterpret_cast<const unsigned long long*>(ctrl + 6));  // counted by the cull
        }
        atomicAdd(stats + 3, (unsigned long long)n_full);
        atomicAdd(stats + 5, (unsigned long long)n_pre);
    }
    // the last block to arrive decodes the extrema into the caller's floats (minima, then maxima)
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(ctrl + 2, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (s_last) {
        __threadfence();
        unsigned* out = reinterpret_cast<unsigned*>(minmax_out);
        for (int w = tid; w < W; w += COV_THREADS) {
            out[w] = ~__ldcg(enc + w);
            out[W + w] = __ldcg(enc + W + w);
        }
    }
}

// =================================================== pass B ===================================================
// Gate bit matrix of the dense kernel.  Row w holds kWarps groups of PPT ballot words (group g = the words of warp g;
// word k of a row covers points [32k, 32k+32) of the tile, since a warp owns 32*PPT consecutive points).  Rows are
// padded by 4 words (conflict-free when lanes walk different rows at the same word).
template <int PPT>
__device__ __forceinline__ unsigned* bit_row_group(unsigned* bits, int w, int group) {
    return bits + (size_t)w * bit_stride(PPT) + group * PPT;
}

__device__ __forceinline__ float4 lds_f4(unsigned saddr) {
    float4 v;
    asm("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}

// Phase 1 of the dense pass B for one pose PAIR: every point of the thread against both poses on packed fp32 pairs
// (cov_vis2p), then ONE conservative warp vote for the pair and — only when some lane may pass for either pose — the
// exact gate, the ballots and the log-odds per pose.  Non-zero ballot words go to the gate bit matrix (which is all zero
// otherwise: zeroed at kernel start, and the gradient walk clears what it consumed).  The spare slot of an odd W repeats
// the last pose and is skipped after the vote.  Returns whether this warp gated a pair (warp-uniform).
template <int PPT, bool AMIN>
__device__ __forceinline__ bool dense_pair_iter(int pair, int W, unsigned ptab_s, unsigned* __restrict__ bits, int warp,
                                                const f2_t (&X)[PPT], const f2_t (&Y)[PPT], const f2_t (&Z)[PPT],
                                                float (&L)[PPT], const CovConst& C, const CovConst2& C2,
                                                double* __restrict__ acc, int lane) {
    const unsigned base = ptab_s + (unsigned)pair * (COV_PAIR_F4 * 16u);
    const float4 q0 = lds_f4(base), q1 = lds_f4(base + 16u), q2 = lds_f4(base + 32u), q3 = lds_f4(base + 48u),
                 q4 = lds_f4(base + 64u), q5 = lds_f4(base + 80u), q6 = lds_f4(base + 96u), q7 = lds_f4(base + 112u);
    float m[2][PPT];
#pragma unroll
    for (int s = 0; s < PPT; ++s) f2_unpack(cov_vis2p(X[s], Y[s], Z[s], q0, q1, q2, q3, q4, q5, q6, q7, C2), m[0][s], m[1][s]);
    float mxa = m[0][0], mxb = m[1][0];
#pragma unroll
    for (int s = 1; s < PPT; ++s) {
        mxa = fmaxf(mxa, m[0][s]);
        mxb = fmaxf(mxb, m[1][s]);
    }
    // conservative gate thresholds (v3.w of the two poses): one vote for the pair; a few % of the iterations pass
    bool hot = __any_sync(kFull, (mxa >= q7.z) | (mxb >= q7.w));
    if (AMIN) hot = true;  // arg-min points carry gradient: every pair is looked at (block-uniform)
    if (!hot) return false;
    unsigned anyb = 0u;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        const int w = 2 * pair + h;
        if (w >= W) break;  // the spare slot of an odd pose count
        const float4 v4 = lds_f4(base + (8u + h) * 16u);
        unsigned bal[PPT];
        unsigned any_h = 0u;
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            const float d = __fsub_rn(m[h][s], v4.w);
            const bool act = d >= v4.x;  // exactly p >= 0.5
            bal[s] = __ballot_sync(kFull, act);
            any_h |= bal[s];
            if (act) {
                L[s] += cov_logodds(d, v4, C);
                if (d == v4.y) {
                    float x, y, z, t;
                    f2_unpack(X[s], x, t); f2_unpack(Y[s], y, t); f2_unpack(Z[s], z, t);
                    tie_accumulate_pair(x, y, z, w, C, acc, w * COV_ACC_STRIDE + 8);
                }
            }
        }
        anyb |= any_h;
        if (any_h != 0u && lane == 0) {
            unsigned* brow = bit_row_group<PPT>(bits, w, warp);
            if (PPT == 4) *reinterpret_cast<uint4*>(brow) = make_uint4(bal[0], bal[1 % PPT], bal[2 % PPT], bal[3 % PPT]);
            else if (PPT == 2) *reinterpret_cast<uint2*>(brow) = make_uint2(bal[0], bal[1 % PPT]);
            else brow[0] = bal[0];
        }
        if (AMIN) {  // only compact clouds whose minimum did not underflow to 0
            if (v4.w > 0.f) {
#pragma unroll
                for (int s = 0; s < PPT; ++s)
                    if (m[h][s] == v4.w) {
                        float x, y, z, t;
                        f2_unpack(X[s], x, t); f2_unpack(Y[s], y, t); f2_unpack(Z[s], z, t);
                        tie_accumulate_pair(x, y, z, w, C, acc, w * COV_ACC_STRIDE + 15);
                    }
            }
        }
    }
    return anyb != 0u;
}

// Forward of one listed pose for a warp of the pruned kernel: m for the warp's points, log-odds of the gated ones added to
// L; returns whether the warp has a gated pair for the pose.  `row` = the pose's 6 float4 in the global table (L1 hits:
// a tile touches a handful of rows).  The conservative threshold lives in v5.w (v3.w holds qthr); the exact gate test
// runs only when some lane may pass.
template <int PPT, bool AMIN>
__device__ __forceinline__ bool tiles_pose_iter(const float4* __restrict__ row, const float4& v3, const float (&px)[PPT],
                                                const float (&py)[PPT], const float (&pz)[PPT], float (&L)[PPT],
                                                const CovConst& C, double* __restrict__ acc_row) {
    float m[PPT];
    const float4 v0 = __ldg(row), v1 = __ldg(row + 1), v2 = __ldg(row + 2);
    const float thr = __ldg(&row[5].w);
#pragma unroll
    for (int s = 0; s < PPT; ++s) m[s] = cov_vis<false>(px[s], py[s], pz[s], v0, v1, v2, v3, C, nullptr);
    float mmax = m[0];
#pragma unroll
    for (int s = 1; s < PPT; ++s) mmax = fmaxf(mmax, m[s]);
    bool any = false;
    if (__any_sync(kFull, mmax >= thr)) {  // warp-uniform: some point may pass the gate (conservative threshold)
        const float4 v4 = __ldg(row + 4);
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            const float d = __fsub_rn(m[s], v4.w);
            const bool act = d >= v4.x;  // exactly p >= 0.5
            any |= act;
            if (act) {
                L[s] += cov_logodds(d, v4, C);
                if (acc_row && d == v4.y) tie_accumulate_g(px[s], py[s], pz[s], row, C, acc_row + 8);
            }
        }
        any = __any_sync(kFull, any);
    }
    if (AMIN) {  // only compact clouds whose minimum did not underflow to 0 (block-uniform choice of the caller)
        const float a = __ldg(&row[4].w);
        if (a > 0.f) {
#pragma unroll
            for (int s = 0; s < PPT; ++s)
                if (m[s] == a) tie_accumulate_g(px[s], py[s], pz[s], row, C, acc_row + 15);
        }
    }
    return any;
}

// Backward of one gated pose for a warp of the pruned kernels (pass B, the differentiable sweep): m again for the warp's
// points (bit-identical to the forward), the gate, dm/dx, the 8 weighted sums in registers; a fixed 9-shuffle tree reduces
// them over the warp and one lane per component adds the result to the pose's fp64 accumulator row (fire-and-forget
// RED.F64).  G = the points' dr/dL (times the upstream gradient, if any).
template <int PPT>
__device__ __forceinline__ void tiles_pose_backward(const float4* __restrict__ row, const float (&px)[PPT],
                                                    const float (&py)[PPT], const float (&pz)[PPT], const float (&G)[PPT],
                                                    const CovConst& C, double* __restrict__ acc_row, int lane) {
    const float4 v0 = __ldg(row), v1 = __ldg(row + 1), v2 = __ldg(row + 2), v3 = __ldg(row + 3), v4 = __ldg(row + 4),
                 v5 = __ldg(row + 5);
    float v[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int s = 0; s < PPT; ++s) {
        CovEval ev;
        const float m = cov_vis<true>(px[s], py[s], pz[s], v0, v1, v2, v3, C, &ev);
        const float d = __fsub_rn(m, v4.w);
        if (d >= v4.x) {  // exactly p >= 0.5, as in the forward
            const float p = __fdiv_rn(d, v4.y);
            if (p <= C.hi) {  // clamp backward gate (inclusive)
                float gx, gy, gz;
                cov_vis_grad(m, ev, v0, v1, v2, C, gx, gy, gz);
                const float yx = px[s] - v5.x, yy = py[s] - v5.y, yz = pz[s] - v5.z;
                const float e = G[s] * cov_rcp(p * (1.f - p));
                const float om = e * v4.z;
                v[0] += om * gx; v[1] += om * gy; v[2] += om * gz;
                v[3] += om * (gy * yz - gz * yy);
                v[4] += om * (gz * yx - gx * yz);
                v[5] += om * (gx * yy - gy * yx);
                v[6] += e;
                v[7] += e * p;
            }
        }
    }
    cov_warp_sum8(v, lane);
    if ((lane & 3) == 0 && v[0] != 0.f) {  // one fire-and-forget fp64 RED per component
        const int comp = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
        atomicAdd(acc_row + comp, (double)v[0]);
    }
}

// Phase 2 of the dense kernel: the gated pairs of all W bit rows, each row split over 2^seg_log2 lanes.  A lane pops
// its set bits in ascending point order, recomputes m (bit-identical) and dm/dx, and accumulates in registers;
// segments are combined with xor-shuffles; one owner lane adds into accs.
template <int PPT>
__device__ __forceinline__ void fused_phase2(const float4* __restrict__ ptab, unsigned* __restrict__ bits,
                                             const float* __restrict__ pt, const float* __restrict__ Gs,
                                             float* __restrict__ accs, int W, int seg_log2, const CovConst& C, int tid) {
    constexpr int NW = bit_words(PPT);
    constexpr int RS = bit_stride(PPT);
    const int nseg = 1 << seg_log2;       // lanes that share one pose row
    const int wps = NW >> seg_log2;       // ballot words per lane
    const int ntask = W << seg_log2;
    for (int base = 0; base < ntask; base += COV_THREADS) {
        const int task = base + tid;
        const bool live = task < ntask;
        const int w = live ? (task >> seg_log2) : 0;
        const int seg = task & (nseg - 1);
        const float4* pair = ptab + (size_t)(w >> 1) * COV_PAIR_F4;
        const int hslot = w & 1;
        const float4 v0 = cov_pair_row(pair, hslot, 0), v1 = cov_pair_row(pair, hslot, 1), v2 = cov_pair_row(pair, hslot, 2),
                     v3 = cov_pair_row(pair, hslot, 3), v4 = pair[8 + hslot], v5 = pair[10 + hslot];
        unsigned* brow = bits + (size_t)w * RS;  // every word of a row belongs to exactly one lane: it is cleared once read
        int k = seg * wps;
        const int kend = live ? k + wps : k;
        unsigned word = live ? brow[k] : 0u;
        if (word != 0u) brow[k] = 0u;
        float f0 = 0.f, f1 = 0.f, f2 = 0.f, t0 = 0.f, t1 = 0.f, t2 = 0.f, se = 0.f, sep = 0.f;
        while (true) {
            while (word == 0u && k + 1 < kend) {
                word = brow[++k];
                if (word != 0u) brow[k] = 0u;
            }
            if (!__any_sync(kFull, word != 0u)) break;
            if (word != 0u) {
                const int bit = __ffs(word) - 1;
                word &= word - 1;
                const int local = k * 32 + bit;
                CovEval ev;
                const float x = pt[local * 3], y = pt[local * 3 + 1], z = pt[local * 3 + 2];
                const float m = cov_vis<true>(x, y, z, v0, v1, v2, v3, C, &ev);
                const float d = __fsub_rn(m, v4.w);
                const float p = __fdiv_rn(d, v4.y);
                if (p <= C.hi) {  // clamp backward gate (inclusive); p >= 0.5 holds for every set bit
                    float gx, gy, gz;
                    cov_vis_grad(m, ev, v0, v1, v2, C, gx, gy, gz);
                    const float yx = x - v5.x, yy = y - v5.y, yz = z - v5.z;
                    const float e = Gs[local] / (p * (1.f - p));
                    const float om = e * v4.z;
                    f0 += om * gx; f1 += om * gy; f2 += om * gz;
                    t0 += om * (gy * yz - gz * yy);
                    t1 += om * (gz * yx - gx * yz);
                    t2 += om * (gx * yy - gy * yx);
                    se += e;
                    sep += e * p;
                }
            }
        }
        for (int o = 1; o < nseg; o <<= 1) {
            f0 += __shfl_xor_sync(kFull, f0, o); f1 += __shfl_xor_sync(kFull, f1, o);
            f2 += __shfl_xor_sync(kFull, f2, o); t0 += __shfl_xor_sync(kFull, t0, o);
            t1 += __shfl_xor_sync(kFull, t1, o); t2 += __shfl_xor_sync(kFull, t2, o);
            se += __shfl_xor_sync(kFull, se, o); sep += __shfl_xor_sync(kFull, sep, o);
        }
        if (live && seg == 0) {
            float* a8 = accs + (size_t)w * 8;
            a8[0] += f0; a8[1] += f1; a8[2] += f2; a8[3] += t0;
            a8[4] += t1; a8[5] += t2; a8[6] += se; a8[7] += sep;
        }
    }
}

// A block's accumulators -> the caller's fp64 rows (fp64 atomics; the reward sum likewise).
template <typename T>
__device__ __forceinline__ void fused_block_flush(const T* accs, int W, double* __restrict__ acc, double sum_r,
                                                  double* red, int tid) {
    for (int i = tid; i < W * 8; i += COV_THREADS) {
        const T v = accs[i];
        if (v != (T)0) atomicAdd(acc + (size_t)(i >> 3) * COV_ACC_STRIDE + (i & 7), (double)v);
    }
    const double ws = cov_warp_sum(sum_r);
    if ((tid & 31) == 0) red[tid >> 5] = ws;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int i = 0; i < kWarps; ++i) t += red[i];
        if (t != 0.0) atomicAdd(acc + (size_t)W * COV_ACC_STRIDE, t);
    }
}

// ---- dense ----
// HAS_PRIOR: r_j = sigmoid(prior_j + L_j), prior indexed like `rewards` (through out_index).
// WSUM (with HAS_UP): `upstream` is the point weight w_j; the reward sum is sum_j w_j r_j and G_j = w_j r_j (1 - r_j).
template <int PPT, bool HAS_UP, bool HAS_PRIOR, bool WSUM = false>
__global__ void __launch_bounds__(COV_THREADS, 2)
cov_traj_fused_kernel(const float* __restrict__ xyz, int64_t n, const float* __restrict__ poses,
                      const float* __restrict__ quats, int W, const float* __restrict__ K9, CovConst C,
                      const float* __restrict__ minmax, const float* __restrict__ upstream,
                      const int32_t* __restrict__ out_index, float* __restrict__ rewards, double* __restrict__ acc,
                      int seg_log2, const float* __restrict__ prior) {
    constexpr int T = tile_points(PPT);
    constexpr int RS = bit_stride(PPT);
    // shared memory: pose table | the tile's points (xyz interleaved) | G_j | gate bits | block accumulators
    extern __shared__ float4 smem4[];
    float4* ptab = smem4;
    float* pt = reinterpret_cast<float*>(smem4) + fused_stage_offset_floats(W);
    float* Gs = pt + T * 3;
    unsigned* bits = reinterpret_cast<unsigned*>(Gs + T);
    float* accs = reinterpret_cast<float*>(bits + (size_t)W * RS);
    __shared__ double red[kWarps];
    __shared__ int amin_pos;  // some pose has min_j m > 0: its arg-min points carry gradient

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) amin_pos = 0;
    __syncthreads();
    const int NP = (W + 1) >> 1;  // pose pairs; an odd W repeats its last pose in the spare slot (never used)
    for (int w = tid; w < 2 * NP; w += COV_THREADS) {
        const int ws = w < W ? w : W - 1;
        float4 row[COV_ROW_F4];
        cov_pose_row(poses + 3 * ws, quats + 4 * ws, K9, C, row);
        const float a = minmax[ws];
        cov_norm_row(row, a, minmax[W + ws], row[3].w);  // conservative gate threshold (exact test in the rare path)
        cov_pair_store(ptab + (size_t)(w >> 1) * COV_PAIR_F4, w & 1, row);
        if (a > 0.f) amin_pos = 1;  // benign race: every writer stores 1
    }
    for (int i = tid; i < W * 8; i += COV_THREADS) accs[i] = 0.f;
    for (int i = tid; i < W * RS; i += COV_THREADS) bits[i] = 0u;  // phase 1 stores non-zero ballots only; phase 2 clears what it reads
    __syncthreads();

    double sum_r = 0.0;
    const int64_t ntiles = (n + T - 1) / T;
    const bool check_amin = amin_pos != 0;
    const unsigned ptab_s = smem_u32(ptab);
    const CovConst2 C2 = cov_make_const2(C);
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        f2_t X[PPT], Y[PPT], Z[PPT];   // the thread's points as broadcast pairs
        float L[PPT];
        bool valid[PPT];
        const int lbase = warp * (32 * PPT) + lane;
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            const int64_t j = tile * T + lbase + s * 32;
            valid[s] = j < n;
            // a point past the end sits 3e18 m away: m = 0 exactly, never gated, never a tie
            const float x = valid[s] ? __ldg(xyz + j * 3) : 3.0e18f;
            const float y = valid[s] ? __ldg(xyz + j * 3 + 1) : 3.0e18f;
            const float z = valid[s] ? __ldg(xyz + j * 3 + 2) : 3.0e18f;
            pt[(lbase + s * 32) * 3] = x;
            pt[(lbase + s * 32) * 3 + 1] = y;
            pt[(lbase + s * 32) * 3 + 2] = z;
            X[s] = f2_pack(x, x);
            Y[s] = f2_pack(y, y);
            Z[s] = f2_pack(z, z);
            L[s] = 0.f;
        }
        bool any_gate = false;  // warp-uniform
        if (check_amin) {  // arg-min points carry gradient: every pair must be looked at
            for (int pr = 0; pr < NP; ++pr) any_gate |= dense_pair_iter<PPT, true>(pr, W, ptab_s, bits, warp, X, Y, Z, L, C, C2, acc, lane);
        } else {
            for (int pr = 0; pr < NP; ++pr) any_gate |= dense_pair_iter<PPT, false>(pr, W, ptab_s, bits, warp, X, Y, Z, L, C, C2, acc, lane);
        }
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            float x = L[s];
            if (HAS_PRIOR && valid[s]) {
                const int64_t j = tile * T + lbase + s * 32;
                x = cov_fuse_prior(__ldg(prior + (out_index ? (int64_t)out_index[j] : j)), x);
            }
            const float r = 1.f / (1.f + expf(-x));
            float g = r * (1.f - r);
            if (valid[s]) {
                const int64_t j = tile * T + lbase + s * 32;
                const int64_t jo = out_index ? (int64_t)out_index[j] : j;
                rewards[jo] = r;
                if (WSUM) {
                    const float wj = upstream[jo];
                    sum_r += (double)wj * (double)r;
                    g *= wj;
                } else {
                    sum_r += (double)r;
                    if (HAS_UP) g *= upstream[jo];
                }
            }
            Gs[lbase + s * 32] = g;
        }
        // one barrier per tile; the gradient walk (and its closing barrier) only when somebody gated a pair
        if (__syncthreads_or(any_gate ? 1 : 0)) {
            fused_phase2<PPT>(ptab, bits, pt, Gs, accs, W, seg_log2, C, tid);
            __syncthreads();
        }
    }
    fused_block_flush(accs, W, acc, sum_r, red, tid);
}

// ---- pruned: persistent warps over the work list (for_each_item), per 128-point item ----
//   forward   walk the box's pose mask (the poses whose qthr-ball meets the box) and evaluate each; gated lanes add their
//             log-odds; the warp notes (one bit per pose) whether it had a gated pair.  Then r_j,
//             G_j = r_j (1 - r_j) per point; rewards stored.
//   backward  the warp walks its noted poses: m again for its points (bit-identical), the gate, dm/dx, the 8 weighted
//             sums in registers; a fixed 9-shuffle tree reduces them over the warp and one lane per component adds the
//             result to the caller's fp64 accumulator row (fire-and-forget RED.F64).
// On the bench cloud ~58 % of the point slots of an evaluated (warp, pose) are gated (profiles/r02_*), so the
// re-evaluation keeps most lanes busy.
// `rewards` was pre-filled with 1/2, only other values are stored; the warps add sum_j (r_j - 1/2) of the listed
// tiles to acc[W * STRIDE], which starts at 0.5 * n.
// HAS_PRIOR: the pre-fill is sigmoid(prior_j) and the sum starts at sum_j sigmoid(prior_j); a listed point reads its
// prior at the index its reward goes to (the gather HAS_UP makes for upstream_j), r_j = sigmoid(prior_j + L_j) is stored
// where L_j != 0 and r_j - sigmoid(prior_j) is added.  G_j = r_j (1 - r_j) for every point, L_j = 0 included (a gated
// pair with p exactly 1/2 adds nothing to L_j but still enters the backward).
// WSUM (point weights, with HAS_UP): `upstream` is the weight w_j, gathered like upstream_j; w_j (r_j - r0_j) is added
// (r0_j = 1/2 or sigmoid(prior_j)) to a sum that starts at sum_j w_j r0_j, and G_j = w_j r_j (1 - r_j).
constexpr int kTilesMinBlocks = 3;            // resident blocks per SM the register allocation aims at

template <bool HAS_UP, bool HAS_PRIOR, bool WSUM = false>
__global__ void __launch_bounds__(COV_THREADS, kTilesMinBlocks)
cov_traj_fused_tiles_kernel(const float* __restrict__ xyz, int64_t n, const float4* __restrict__ table, int W, CovConst C,
                            const float* __restrict__ upstream, const int32_t* __restrict__ out_index,
                            float* __restrict__ rewards, double* __restrict__ acc,
                            const unsigned* __restrict__ amask_g, int mask_stride,
                            const int* __restrict__ worklist, int* __restrict__ ctrl, int64_t ntiles,
                            unsigned long long* __restrict__ stats, const float* __restrict__ prior) {
    static_assert(HAS_UP || !WSUM, "the weight rides on the upstream gather");
    constexpr int PPT = kItemPpt;
    __shared__ unsigned wgate[kWarps][kMaskWords];   // per warp: poses with a gated pair among its points (this item)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool check_amin = ctrl[1] != 0;  // some pose has min_j m > 0
    const int n_items = ctrl[0];
    const int nwords = (W + 31) >> 5;
    unsigned* wg = wgate[warp];  // lane 0 rewrites it for the next item only after the closing __syncwarp of this one
    double sum_r = 0.0;
    unsigned n_full = 0, n_bwd = 0;
    for_each_item<true>(xyz, n, amask_g, mask_stride, out_index, worklist, n_items, ctrl + 3, [](int) {},
                        [&](const Item& item) {
        // ------------------------------ forward ------------------------------
        float px[PPT], py[PPT], pz[PPT], L[PPT];
        bool valid[PPT];
        load_item_points<false>(item, xyz, n, lane, px, py, pz, valid);
#pragma unroll
        for (int s = 0; s < PPT; ++s) L[s] = 0.f;
        bool warp_gated = false;
        for (int c = 0; c < nwords; ++c) {
            unsigned word = item.mask[c];
            unsigned gbits = 0u;
            while (word) {
                const int b = __ffs(word) - 1;
                const int w = c * 32 + b;
                word &= word - 1;
                const float4* row = table + (size_t)w * COV_ROW_F4;
                const float4 v3 = __ldg(row + 3);
                // no per-point pre-filter here: it rejected only 11 % of what the cull's box test let through and cost a fifth
                // of the evaluation it saved
                ++n_full;
                double* acc_row = acc + (size_t)w * COV_ACC_STRIDE;
                const bool g = check_amin ? tiles_pose_iter<PPT, true>(row, v3, px, py, pz, L, C, acc_row)
                                          : tiles_pose_iter<PPT, false>(row, v3, px, py, pz, L, C, acc_row);
                if (g) gbits |= 1u << b;
            }
            if (lane == 0) wg[c] = gbits;
            warp_gated |= gbits != 0u;
        }
        float G[PPT];
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            if (HAS_PRIOR) {
                if (!valid[s]) {  // past the end of the cloud: never gated, G unused
                    G[s] = 0.f;
                    continue;
                }
                const int64_t j = item.j0 + s * 32 + lane;
                const int64_t jo = out_index ? (item.whole ? (int64_t)item.perm[s * 32 + lane] : (int64_t)out_index[j]) : j;
                const float pr = __ldg(prior + jo);
                const float r0 = cov_sigmoid(pr);
                float r = r0;
                if (L[s] != 0.f) {
                    r = cov_sigmoid(cov_fuse_prior(pr, L[s]));
                    rewards[jo] = r;
                }
                G[s] = r * (1.f - r);
                if (WSUM) {
                    const float wj = upstream[jo];
                    sum_r += (double)wj * (double)(r - r0);
                    G[s] *= wj;
                    continue;
                }
                sum_r += (double)(r - r0);
                if (HAS_UP) G[s] *= upstream[jo];
                continue;
            }
            float r = 0.5f;
            G[s] = 0.25f;  // exactly what the formulas below give for L = 0
            if (L[s] != 0.f) {
                r = 1.f / (1.f + expf(-L[s]));
                G[s] = r * (1.f - r);
            }
            if (valid[s]) {
                const int64_t j = item.j0 + s * 32 + lane;
                if (!WSUM) sum_r += (double)(r - 0.5f);
                const bool store = r != 0.5f;
                int64_t jo = j;
                if (out_index && (store || HAS_UP))
                    jo = item.whole ? (int64_t)item.perm[s * 32 + lane] : (int64_t)out_index[j];  // staged with the item
                if (store) rewards[jo] = r;
                if (WSUM) {
                    const float wj = upstream[jo];
                    sum_r += (double)wj * (double)(r - 0.5f);
                    G[s] *= wj;
                } else if (HAS_UP) {
                    G[s] *= upstream[jo];
                }
            }
        }
        // ------------------------------ backward ------------------------------
        if (warp_gated) {
            __syncwarp();  // lane 0's notes are visible to the warp
            for (int c = 0; c < nwords; ++c) {
                unsigned word = wg[c];
                while (word) {
                    const int w = c * 32 + __ffs(word) - 1;
                    word &= word - 1;
                    ++n_bwd;
                    tiles_pose_backward<PPT>(table + (size_t)w * COV_ROW_F4, px, py, pz, G, C,
                                             acc + (size_t)w * COV_ACC_STRIDE, lane);
                }
            }
        }
    });
    {
        const double ws = cov_warp_sum(sum_r);
        if (lane == 0 && ws != 0.0) atomicAdd(acc + (size_t)W * COV_ACC_STRIDE, ws);
    }
    if (stats && lane == 0) {
        if (threadIdx.x == 0 && blockIdx.x == 0) {
            atomicAdd(stats + 0, (unsigned long long)ntiles * kWarps * W);
            atomicAdd(stats + 6, *reinterpret_cast<const unsigned long long*>(ctrl + 4));  // counted by the cull
        }
        atomicAdd(stats + 1, (unsigned long long)n_full);
        atomicAdd(stats + 4, (unsigned long long)n_bwd);
    }
}

// ---- candidate sweep, pruned (BASELINE config 5): forward only, per-trajectory sum_j r_j ----
// Persistent warps as in the two passes above (for_each_item).  Poses are trajectory-major (pose = traj * per_traj + i),
// so walking a box's pose mask in ascending order visits the trajectories one after the other: a warp keeps the log-odds
// sums of its points for the current trajectory, and when the trajectory changes it adds sum_j (sigmoid(L_j) - 1/2) to
// that trajectory's total (fp64 shared atomic; the block adds its totals to the output at the end).  Trajectories no
// pose of which is listed for an item contribute exactly 1/2 per point: 0.5 * n is added once.
// HAS_PRIOR: sum_j (sigmoid(prior_j + L_j) - sigmoid(prior_j)) at a flush (the item's 128 priors, in the cloud's order,
// read there), and *prior_sum = sum_j sigmoid(prior_j) in place of 0.5 * n.
// HAS_W: each point's term times its weight w_j (read next to the prior, in the cloud's order), and *prior_sum is the
// weighted base sum_j w_j r0_j (cov_weight_sums).
// PREFIX (cov_sweep_prefix_rewards): one slot per pose instead of one per trajectory.  After each pose at which the warp
// gated a pair, the item's flush value V (the same fp32 terms and warp sum) is what the sweep of the trajectory cut after
// that pose would add at its end; the difference (double)V - (double)V_prev goes to the pose's slot (V_prev = 0 at the
// trajectory's first pose).  Block 0 adds the base to slot 0 of each trajectory; the inclusive scan of a trajectory's
// slots (cov_prefix_scan_kernel) is then the truncated sweep's sum, up to the order of fp64 additions.
template <bool HAS_PRIOR, bool HAS_W = false, bool PREFIX = false>
__global__ void __launch_bounds__(COV_THREADS, 3)
cov_sweep_tiles_kernel(const float* __restrict__ xyz, int64_t n, const float4* __restrict__ table, int W, int per_traj,
                       int n_traj, CovConst C, const unsigned* __restrict__ amask_g, int mask_stride, const int* __restrict__ worklist, int* __restrict__ ctrl,
                       double* __restrict__ sum_out, const float* __restrict__ prior, const double* __restrict__ prior_sum,
                       const float* __restrict__ weight) {
    constexpr int PPT = kItemPpt;
    extern __shared__ float4 smem4[];
    double* ssum = reinterpret_cast<double*>(smem4);   // per-trajectory (PREFIX: per-pose) totals of this block
    const int tid = threadIdx.x, lane = tid & 31;
    const int nslots = PREFIX ? W : n_traj;
    for (int t = tid; t < nslots; t += COV_THREADS) ssum[t] = 0.0;
    __syncthreads();
    const int n_items = ctrl[0];
    const int nwords = (W + 31) >> 5;
    for_each_item<false>(xyz, n, amask_g, mask_stride, nullptr, worklist, n_items, ctrl + 3, [](int) {},
                         [&](const Item& item) {
        float px[PPT], py[PPT], pz[PPT], L[PPT];
        bool valid[PPT];
        load_item_points<false>(item, xyz, n, lane, px, py, pz, valid);
        int cur = -1;      // trajectory whose log-odds sums are in L
        bool touched = false;
        float vprev = 0.f;  // PREFIX: the item's value after the last gated pose of `cur`
        // the warp sum of the item's reward terms for the log-odds sums in L
        auto value = [&]() {
            float a = 0.f;
#pragma unroll
            for (int s = 0; s < PPT; ++s) {
                if (HAS_W) {
                    if (valid[s] && L[s] != 0.f) {
                        const int64_t j = item.j0 + s * 32 + lane;
                        const float wj = __ldg(weight + j);
                        if (HAS_PRIOR) {
                            const float pr = __ldg(prior + j);
                            a += wj * (cov_sigmoid(cov_fuse_prior(pr, L[s])) - cov_sigmoid(pr));
                        } else {
                            a += wj * (1.f / (1.f + expf(-L[s])) - 0.5f);
                        }
                    }
                } else if (HAS_PRIOR) {
                    if (valid[s] && L[s] != 0.f) {
                        const float pr = __ldg(prior + item.j0 + s * 32 + lane);
                        a += cov_sigmoid(cov_fuse_prior(pr, L[s])) - cov_sigmoid(pr);
                    }
                } else if (valid[s] && L[s] != 0.f) {
                    a += 1.f / (1.f + expf(-L[s])) - 0.5f;
                }
            }
            return cov_warp_sum(a);
        };
        auto flush = [&]() {
            if (cur >= 0 && touched) {
                const float a = value();
                if (lane == 0 && a != 0.f) atomicAdd(ssum + cur, (double)a);
            }
        };
        for (int c = 0; c < nwords; ++c) {
            unsigned word = item.mask[c];
            while (word) {
                const int w = c * 32 + __ffs(word) - 1;
                word &= word - 1;
                const float4* row = table + (size_t)w * COV_ROW_F4;
                const float4 v3 = __ldg(row + 3);
                const int t = w / per_traj;
                if (t != cur) {
                    if (!PREFIX) flush();
                    cur = t;
                    touched = false;
                    vprev = 0.f;
#pragma unroll
                    for (int s = 0; s < PPT; ++s) L[s] = 0.f;
                }
                const bool g = tiles_pose_iter<PPT, false>(row, v3, px, py, pz, L, C, nullptr);
                if (PREFIX) {
                    if (g) {  // warp-uniform
                        const float v = value();
                        if (lane == 0 && v != vprev) atomicAdd(ssum + w, (double)v - (double)vprev);
                        vprev = v;
                    }
                } else {
                    touched |= g;
                }
            }
        }
        if (!PREFIX) flush();
    });
    __syncthreads();
    for (int t = tid; t < nslots; t += COV_THREADS) {
        double v = ssum[t];
        if (blockIdx.x == 0 && (!PREFIX || t % per_traj == 0)) v += (HAS_PRIOR || HAS_W) ? *prior_sum : 0.5 * (double)n;
        if (v != 0.0) atomicAdd(sum_out + t, v);
    }
}

// Inclusive prefix sums of each trajectory's P slots, in place: one warp per trajectory, 32 slots at a time (a fixed
// shuffle tree, then the carry of the previous 32), so the result is a deterministic function of the slots.
__global__ void __launch_bounds__(256) cov_prefix_scan_kernel(double* __restrict__ sums, int n_traj, int per_traj) {
    const int t = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (t >= n_traj) return;
    double* row = sums + (size_t)t * per_traj;
    double carry = 0.0;
    for (int i0 = 0; i0 < per_traj; i0 += 32) {
        const int i = i0 + lane;
        double v = i < per_traj ? row[i] : 0.0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const double u = __shfl_up_sync(kFull, v, o);
            if (lane >= o) v += u;
        }
        v += carry;
        if (i < per_traj) row[i] = v;
        carry = __shfl_sync(kFull, v, 31);
    }
}

// ---- differentiable candidate sweep, pruned: per trajectory what pass B computes for it alone ----
// The walk of cov_sweep_tiles_kernel (trajectory-major poses, one trajectory's log-odds sums in L at a time) with pass B's
// bookkeeping: while it walks the poses of the current trajectory, lane 0 notes in the warp's shared mask which of them had
// a gated pair.  At each trajectory boundary and at the end of the item the warp computes r_j and G_j = dr/dL with pass B's
// expressions, adds sum_j (r_j - 1/2) to the trajectory's reward sum and runs pass B's backward (tiles_pose_backward) over
// the noted poses, then clears the notes.  Pose w of trajectory t owns row (w - t P) of block t of the accumulators,
// `acc + t * COV_SWEEP_ACC_BLOCK(P)`: the layout cov_traj_fused writes for that trajectory alone (rows, then sum_j r_j).
// The forward of a trajectory visits the same poses in the same order as pass B with W = P on the same item (same cull),
// so its L, r_j and G_j — and the re-evaluated m of the backward — are bit-identical to pass B's.
// HAS_PRIOR: at a flush r_j = sigmoid(prior_j + L_j) and r_j - sigmoid(prior_j) is added, with the item's 128 priors (in
// the cloud's order) read there; the blocks start at sum_j sigmoid(prior_j) (cov_sweep_acc_init_kernel).
// HAS_W: the item's 128 weights w_j (cloud's order) are read at a flush too; w_j (r_j - r0_j) is added and G_j is
// multiplied by w_j before the backward; the blocks start at sum_j w_j r0_j (cov_weight_sums).
template <bool HAS_PRIOR, bool HAS_W = false>
__global__ void __launch_bounds__(COV_THREADS, kTilesMinBlocks)
cov_sweep_fused_tiles_kernel(const float* __restrict__ xyz, int64_t n, const float4* __restrict__ table, int W, int per_traj,
                             CovConst C, const unsigned* __restrict__ amask_g, int mask_stride, const int* __restrict__ worklist, int* __restrict__ ctrl, int64_t ntiles,
                             double* __restrict__ acc, unsigned long long* __restrict__ stats,
                             const float* __restrict__ prior, const float* __restrict__ weight) {
    constexpr int PPT = kItemPpt;
    __shared__ unsigned wgate[kWarps][kMaskWords];   // per warp: poses of the current trajectory with a gated pair
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool check_amin = ctrl[1] != 0;  // some pose has min_j m > 0
    const int n_items = ctrl[0];
    const int nwords = (W + 31) >> 5;
    const size_t block = COV_SWEEP_ACC_BLOCK(per_traj);
    unsigned* wg = wgate[warp];
    for (int c = lane; c < kMaskWords; c += 32) wg[c] = 0u;  // afterwards every flush clears the words it walked
    __syncwarp();
    unsigned n_full = 0, n_bwd = 0;
    for_each_item<false>(xyz, n, amask_g, mask_stride, nullptr, worklist, n_items, ctrl + 3, [](int) {},
                         [&](const Item& item) {
        float px[PPT], py[PPT], pz[PPT], L[PPT];
        bool valid[PPT];
        load_item_points<false>(item, xyz, n, lane, px, py, pz, valid);
        int cur = -1;          // trajectory whose log-odds sums are in L
        bool gated = false;    // warp-uniform: some pose of `cur` had a gated pair (otherwise r_j = 1/2, nothing to add)
        auto flush = [&]() {
            if (cur < 0 || !gated) return;
            double* A = acc + (size_t)cur * block;
            float G[PPT];
            float a = 0.f;
#pragma unroll
            for (int s = 0; s < PPT; ++s) {
                if (HAS_PRIOR) {
                    const float pr = valid[s] ? __ldg(prior + item.j0 + s * 32 + lane) : 0.f;
                    const float r0 = cov_sigmoid(pr);
                    const float r = L[s] != 0.f ? cov_sigmoid(cov_fuse_prior(pr, L[s])) : r0;
                    G[s] = r * (1.f - r);
                    if (HAS_W) {
                        const float wj = valid[s] ? __ldg(weight + item.j0 + s * 32 + lane) : 0.f;
                        G[s] *= wj;
                        a += wj * (r - r0);
                    } else if (valid[s]) {
                        a += r - r0;
                    }
                    continue;
                }
                float r = 0.5f;
                G[s] = 0.25f;  // exactly what the formulas below give for L = 0
                if (L[s] != 0.f) {
                    r = 1.f / (1.f + expf(-L[s]));
                    G[s] = r * (1.f - r);
                }
                if (HAS_W) {
                    const float wj = valid[s] ? __ldg(weight + item.j0 + s * 32 + lane) : 0.f;
                    G[s] *= wj;
                    a += wj * (r - 0.5f);
                } else if (valid[s]) {
                    a += r - 0.5f;
                }
            }
            a = cov_warp_sum(a);
            if (lane == 0 && a != 0.f) atomicAdd(A + (size_t)per_traj * COV_ACC_STRIDE, (double)a);
            __syncwarp();  // lane 0's notes are visible to the warp
            const int p0 = cur * per_traj;
            const int c1 = (p0 + per_traj - 1) >> 5;
            for (int c = p0 >> 5; c <= c1; ++c) {  // only this trajectory's poses are noted
                unsigned word = wg[c];
                while (word) {
                    const int w = c * 32 + __ffs(word) - 1;
                    word &= word - 1;
                    ++n_bwd;
                    tiles_pose_backward<PPT>(table + (size_t)w * COV_ROW_F4, px, py, pz, G, C,
                                             A + (size_t)(w - p0) * COV_ACC_STRIDE, lane);
                }
            }
            __syncwarp();  // every lane has read the notes
            if (lane == 0)
                for (int c = p0 >> 5; c <= c1; ++c) wg[c] = 0u;
        };
        for (int c = 0; c < nwords; ++c) {
            unsigned word = item.mask[c];
            while (word) {
                const int b = __ffs(word) - 1;
                const int w = c * 32 + b;
                word &= word - 1;
                const float4* row = table + (size_t)w * COV_ROW_F4;
                const float4 v3 = __ldg(row + 3);
                ++n_full;
                const int t = w / per_traj;
                if (t != cur) {
                    flush();
                    cur = t;
                    gated = false;
#pragma unroll
                    for (int s = 0; s < PPT; ++s) L[s] = 0.f;
                }
                double* acc_row = acc + (size_t)t * block + (size_t)(w - t * per_traj) * COV_ACC_STRIDE;
                const bool g = check_amin ? tiles_pose_iter<PPT, true>(row, v3, px, py, pz, L, C, acc_row)
                                          : tiles_pose_iter<PPT, false>(row, v3, px, py, pz, L, C, acc_row);
                if (g) {
                    gated = true;
                    if (lane == 0) wg[c] |= 1u << b;
                }
            }
        }
        flush();
    });
    if (stats && lane == 0) {
        if (threadIdx.x == 0 && blockIdx.x == 0) {
            atomicAdd(stats + 0, (unsigned long long)ntiles * kWarps * W);
            atomicAdd(stats + 6, *reinterpret_cast<const unsigned long long*>(ctrl + 4));  // counted by the cull
        }
        atomicAdd(stats + 1, (unsigned long long)n_full);
        atomicAdd(stats + 4, (unsigned long long)n_bwd);
    }
}

// Every trajectory's accumulator block as pass B starts it: rows zero, the reward sum at `sum_base` (0.5 * n: what the
// points no listed pose reaches add), or at *sum_base_dev (sum_j sigmoid(prior_j)) when that is given.
__global__ void cov_sweep_acc_init_kernel(double* __restrict__ acc, int64_t count, int64_t block, double sum_base) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
        acc[i] = (i % block == block - 1) ? sum_base : 0.0;
}
__global__ void cov_sweep_acc_init_dev_kernel(double* __restrict__ acc, int64_t count, int64_t block,
                                              const double* __restrict__ sum_base_dev) {
    const double base = *sum_base_dev;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x)
        acc[i] = (i % block == block - 1) ? base : 0.0;
}

// SURVEY.md App. A.2, one pose: fold the min/max-path terms into the accumulator row A and map (F, T) to (d/dt, d/dq~).
// a, mx: the pose's normalisers; q: its raw quaternion; c0: the scale of the gradient (1/N for the mean).
__device__ __forceinline__ void traj_epilogue_pose(const double* __restrict__ A, float a, float mx,
                                                   const float* __restrict__ q, double c0, float* __restrict__ gp,
                                                   float* __restrict__ gq) {
    const double b = (double)__fsub_rn(mx, a);
    const double dLdb = -A[7] / b;
    const double dLda = -A[6] / b - dLdb;
    double F[3] = {A[0], A[1], A[2]}, Tq[3] = {A[3], A[4], A[5]};
    if (A[14] > 0.0) {
        const double c = dLdb / A[14];
        for (int k = 0; k < 3; ++k) { F[k] += c * A[8 + k]; Tq[k] += c * A[11 + k]; }
    }
    if (A[21] > 0.0) {
        const double c = dLda / A[21];
        for (int k = 0; k < 3; ++k) { F[k] += c * A[15 + k]; Tq[k] += c * A[18 + k]; }
    }
    double qw = q[0], qx = q[1], qy = q[2], qz = q[3];
    double qn = sqrt(qw * qw + qx * qx + qy * qy + qz * qz);
    qn = qn > 1e-12 ? qn : 1e-12;
    qw /= qn; qx /= qn; qy /= qn; qz /= qn;
    for (int k = 0; k < 3; ++k) gp[k] = (float)(-c0 * F[k]);
    const double s = 2.0 * c0 / qn;
    gq[0] = (float)(s * (-Tq[0] * qx - Tq[1] * qy - Tq[2] * qz));
    gq[1] = (float)(s * (Tq[0] * qw + Tq[1] * qz - Tq[2] * qy));
    gq[2] = (float)(s * (Tq[1] * qw - Tq[0] * qz + Tq[2] * qx));
    gq[3] = (float)(s * (Tq[2] * qw + Tq[0] * qy - Tq[1] * qx));
}

__global__ void cov_traj_epilogue_kernel(const double* __restrict__ acc, const float* __restrict__ minmax,
                                         const float* __restrict__ quats, int W, double n_total, int upstream_mode,
                                         float* __restrict__ out) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w == 0) out[0] = (float)(acc[(size_t)W * COV_ACC_STRIDE] / n_total);
    if (w >= W) return;
    const double c0 = upstream_mode ? 1.0 : 1.0 / n_total;
    traj_epilogue_pose(acc + (size_t)w * COV_ACC_STRIDE, minmax[w], minmax[W + w], quats + 4 * w, c0, out + 1 + 3 * w,
                       out + 1 + 3 * W + 4 * w);
}

// The sweep's epilogue: trajectory t's mean and the gradient of that mean, from block t of the accumulators.
// minmax (2, T P): all minima, then all maxima.  out = [T means | T P (d/dt) | T P (d/dq~)].
__global__ void cov_sweep_epilogue_kernel(const double* __restrict__ acc, const float* __restrict__ minmax,
                                          const float* __restrict__ quats, int n_traj, int per_traj, double n_total,
                                          float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // pose t * P + k
    const int TP = n_traj * per_traj;
    const size_t block = COV_SWEEP_ACC_BLOCK(per_traj);
    if (i < n_traj) out[i] = (float)(acc[(size_t)i * block + (size_t)per_traj * COV_ACC_STRIDE] / n_total);
    if (i >= TP) return;
    const int t = i / per_traj, k = i - t * per_traj;
    traj_epilogue_pose(acc + (size_t)t * block + (size_t)k * COV_ACC_STRIDE, minmax[i], minmax[TP + i], quats + 4 * (size_t)i,
                       1.0 / n_total, out + n_traj + 3 * (size_t)i, out + n_traj + 3 * (size_t)TP + 4 * (size_t)i);
}

// The epilogues of the point-weighted calls: the denominator is read on the device (sum_j w_j, cov_weight_sums) instead
// of n_total.  With *den == n they compute what cov_traj_epilogue_kernel (upstream_mode 0) and cov_sweep_epilogue_kernel
// compute, bit for bit.
__global__ void cov_traj_epilogue_dev_kernel(const double* __restrict__ acc, const float* __restrict__ minmax,
                                             const float* __restrict__ quats, int W, const double* __restrict__ den,
                                             float* __restrict__ out) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    const double d = *den;
    if (w == 0) out[0] = (float)(acc[(size_t)W * COV_ACC_STRIDE] / d);
    if (w >= W) return;
    traj_epilogue_pose(acc + (size_t)w * COV_ACC_STRIDE, minmax[w], minmax[W + w], quats + 4 * w, 1.0 / d, out + 1 + 3 * w,
                       out + 1 + 3 * W + 4 * w);
}

__global__ void cov_sweep_epilogue_dev_kernel(const double* __restrict__ acc, const float* __restrict__ minmax,
                                              const float* __restrict__ quats, int n_traj, int per_traj,
                                              const double* __restrict__ den, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;  // pose t * P + k
    const int TP = n_traj * per_traj;
    const size_t block = COV_SWEEP_ACC_BLOCK(per_traj);
    const double d = *den;
    if (i < n_traj) out[i] = (float)(acc[(size_t)i * block + (size_t)per_traj * COV_ACC_STRIDE] / d);
    if (i >= TP) return;
    const int t = i / per_traj, k = i - t * per_traj;
    traj_epilogue_pose(acc + (size_t)t * block + (size_t)k * COV_ACC_STRIDE, minmax[i], minmax[TP + i], quats + 4 * (size_t)i,
                       1.0 / d, out + n_traj + 3 * (size_t)i, out + n_traj + 3 * (size_t)TP + 4 * (size_t)i);
}

// ============================================== point weights ==============================================
// [sum_j w_j r0_j, sum_j w_j] in fp64, r0_j = sigmoid(prior_j) (HAS_PRIOR) or 1/2: the reward-sum base of the weighted
// calls and the denominator of their means.  Grid-stride, warp and block sums, two fp64 atomics per block into the
// zeroed output.
template <bool HAS_PRIOR>
__global__ void __launch_bounds__(256) cov_weight_sums_kernel(const float* __restrict__ weight,
                                                              const float* __restrict__ prior, int64_t n,
                                                              double* __restrict__ out) {
    __shared__ double red[2][8];
    double base = 0.0, tot = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double w = (double)__ldg(weight + i);
        base += w * (HAS_PRIOR ? (double)cov_sigmoid(__ldg(prior + i)) : 0.5);
        tot += w;
    }
    base = cov_warp_sum(base);
    tot = cov_warp_sum(tot);
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = base;
        red[1][threadIdx.x >> 5] = tot;
    }
    __syncthreads();
    if (threadIdx.x < 2) {
        double t = 0.0;
        for (int i = 0; i < 8; ++i) t += red[threadIdx.x][i];
        atomicAdd(out + threadIdx.x, t);
    }
}

// ============================================ prior log-odds (map memory) ============================================
// sum_j sigmoid(prior_j) in fp64 (the reward-sum base of the prior paths): grid-stride, warp and block sums, one fp64
// atomic per block into the zeroed output.
__global__ void __launch_bounds__(256) cov_prior_sum_kernel(const float* __restrict__ prior, int64_t n,
                                                            double* __restrict__ out) {
    __shared__ double red[8];
    double v = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        v += (double)cov_sigmoid(__ldg(prior + i));
    v = cov_warp_sum(v);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < 8; ++i) t += red[i];
        atomicAdd(out, t);
    }
}

// Fused log-odds output, pruned: pass B's forward (same work list and masks, same pose order, hence the same L_j)
// without the backward; out[jo] = out[jo] + L_j for the points with L_j != 0 (the caller pre-filled `out` with the prior,
// indexed like the rewards), the x that pass B's sigmoid takes.
// CARRY (one pose chunk of the long path, cov_traj_fused_long / cov_traj_logodds_long): L_j starts from carry[j] (cloud
// order; zeroed once per call) instead of 0 and, when the warp gated a pair, is stored back there, so that after the last
// chunk carry[j] holds the fp32 sum of every chunk's terms in ascending pose order: the L_j of one call over all poses, bit
// for bit.  A point of such an item whose sum is still 0 is stored as -0 (a marker the finalise kernel reads: the point may
// enter the backward; -0 + x = x for every term x, so the sums are unchanged).  With `acc` (the chunk's rows) the arg-max
// and arg-min tie accumulators go there as in pass B's forward; with `gate_out` lane 0 overwrites the item's mask row
// with the poses at which the warp gated a pair: the poses pass B's backward walks for it (cov_traj_long_backward_kernel).
template <bool CARRY = false>
__global__ void __launch_bounds__(COV_THREADS, kTilesMinBlocks)
cov_traj_logodds_tiles_kernel(const float* __restrict__ xyz, int64_t n, const float4* __restrict__ table, int W, CovConst C,
                              const int32_t* __restrict__ out_index, float* __restrict__ out,
                              const unsigned* __restrict__ amask_g, int mask_stride,
                              const int* __restrict__ worklist, int* __restrict__ ctrl, double* __restrict__ acc = nullptr,
                              float* __restrict__ carry = nullptr, unsigned* __restrict__ gate_out = nullptr,
                              int64_t ntiles = 0, unsigned long long* __restrict__ stats = nullptr) {
    constexpr int PPT = kItemPpt;
    const int lane = threadIdx.x & 31;
    const int n_items = ctrl[0];
    const int nwords = (W + 31) >> 5;
    if constexpr (CARRY) {
        const bool check_amin = acc && ctrl[1] != 0;  // some pose of the chunk has min_j m > 0
        unsigned n_full = 0;
        for_each_item<false>(xyz, n, amask_g, mask_stride, nullptr, worklist, n_items, ctrl + 3, [](int) {},
                             [&](const Item& item) {
            float px[PPT], py[PPT], pz[PPT], L[PPT];
            bool valid[PPT];
            load_item_points<false>(item, xyz, n, lane, px, py, pz, valid);
#pragma unroll
            for (int s = 0; s < PPT; ++s) L[s] = valid[s] ? carry[item.j0 + s * 32 + lane] : 0.f;
            bool warp_gated = false;
            unsigned* grow = gate_out ? gate_out + (size_t)(item.j0 / kItemPts) * mask_stride : nullptr;
            for (int c = 0; c < nwords; ++c) {
                unsigned word = item.mask[c];
                unsigned gbits = 0u;
                while (word) {
                    const int b = __ffs(word) - 1;
                    const int w = c * 32 + b;
                    word &= word - 1;
                    const float4* row = table + (size_t)w * COV_ROW_F4;
                    const float4 v3 = __ldg(row + 3);
                    ++n_full;
                    double* acc_row = acc ? acc + (size_t)w * COV_ACC_STRIDE : nullptr;
                    const bool g = check_amin ? tiles_pose_iter<PPT, true>(row, v3, px, py, pz, L, C, acc_row)
                                              : tiles_pose_iter<PPT, false>(row, v3, px, py, pz, L, C, acc_row);
                    if (g) gbits |= 1u << b;
                }
                if (grow && lane == 0) grow[c] = gbits;
                warp_gated |= gbits != 0u;
            }
            if (warp_gated) {
#pragma unroll
                for (int s = 0; s < PPT; ++s)
                    if (valid[s]) carry[item.j0 + s * 32 + lane] = L[s] != 0.f ? L[s] : -0.f;
            }
        });
        if (stats && lane == 0) {
            if (threadIdx.x == 0 && blockIdx.x == 0) {
                atomicAdd(stats + 0, (unsigned long long)ntiles * kWarps * W);
                atomicAdd(stats + 6, *reinterpret_cast<const unsigned long long*>(ctrl + 4));  // counted by the cull
            }
            atomicAdd(stats + 1, (unsigned long long)n_full);
        }
    } else {
        for_each_item<true>(xyz, n, amask_g, mask_stride, out_index, worklist, n_items, ctrl + 3, [](int) {},
                            [&](const Item& item) {
            float px[PPT], py[PPT], pz[PPT], L[PPT];
            bool valid[PPT];
            load_item_points<false>(item, xyz, n, lane, px, py, pz, valid);
#pragma unroll
            for (int s = 0; s < PPT; ++s) L[s] = 0.f;
            for (int c = 0; c < nwords; ++c) {
                unsigned word = item.mask[c];
                while (word) {
                    const int w = c * 32 + __ffs(word) - 1;
                    word &= word - 1;
                    const float4* row = table + (size_t)w * COV_ROW_F4;
                    tiles_pose_iter<PPT, false>(row, __ldg(row + 3), px, py, pz, L, C, nullptr);
                }
            }
#pragma unroll
            for (int s = 0; s < PPT; ++s) {
                if (valid[s] && L[s] != 0.f) {
                    const int64_t j = item.j0 + s * 32 + lane;
                    const int64_t jo = out_index ? (item.whole ? (int64_t)item.perm[s * 32 + lane] : (int64_t)out_index[j]) : j;
                    out[jo] = cov_fuse_prior(out[jo], L[s]);
                }
            }
        });
    }
}

// The long path after the last chunk's forward: one grid-stride pass over the cloud order.  carry[j] = +0 (bits 0): no
// chunk gated a pair in the point's item, so r_j = r0_j and the point enters no backward: nothing to do.  Otherwise
// L_j = carry[j] (-0 for 0) gives r_j with pass B's expressions: r_j is stored in the caller's order where L_j != 0,
// sum_j (r_j - r0_j) (WSUM: w_j (r_j - r0_j)) is added to the reward-sum slot, and carry[j] becomes G_j = r_j (1 - r_j)
// (times w_j or upstream_j), the dr/dL the backward reads.  FOLD (cov_traj_logodds_long): out[jo] = cov_fuse_prior(out[jo],
// L_j) where L_j != 0, as cov_traj_logodds_tiles_kernel writes it.
template <bool FOLD, bool HAS_UP, bool HAS_PRIOR, bool WSUM>
__global__ void __launch_bounds__(256)
cov_traj_long_finalise_kernel(int64_t n, float* __restrict__ carry, const int32_t* __restrict__ out_index,
                              float* __restrict__ out, const float* __restrict__ upstream,
                              const float* __restrict__ prior, double* __restrict__ sum_slot) {
    static_assert(HAS_UP || !WSUM, "the weight rides on the upstream gather");
    double sum_r = 0.0;
    const int64_t nq = (n + 3) / 4;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        const bool whole = q * 4 + 4 <= n;
        float v[4];
        if (whole) {
            const float4 f = reinterpret_cast<const float4*>(carry)[q];
            v[0] = f.x; v[1] = f.y; v[2] = f.z; v[3] = f.w;
        } else {
            for (int k = 0; k < 4; ++k) v[k] = q * 4 + k < n ? carry[q * 4 + k] : 0.f;
        }
        if ((__float_as_uint(v[0]) | __float_as_uint(v[1]) | __float_as_uint(v[2]) | __float_as_uint(v[3])) == 0u) continue;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (__float_as_uint(v[k]) == 0u) continue;
            const float L = v[k];
            const int64_t j = q * 4 + k;
            const int64_t jo = out_index ? (int64_t)out_index[j] : j;
            if (FOLD) {
                if (L != 0.f) out[jo] = cov_fuse_prior(out[jo], L);
                continue;
            }
            float r, G;
            if (HAS_PRIOR) {
                const float pr = __ldg(prior + jo);
                const float r0 = cov_sigmoid(pr);
                r = r0;
                if (L != 0.f) {
                    r = cov_sigmoid(cov_fuse_prior(pr, L));
                    out[jo] = r;
                }
                G = r * (1.f - r);
                if (WSUM) {
                    const float wj = upstream[jo];
                    sum_r += (double)wj * (double)(r - r0);
                    G *= wj;
                } else {
                    sum_r += (double)(r - r0);
                    if (HAS_UP) G *= upstream[jo];
                }
            } else {
                r = 0.5f;
                G = 0.25f;  // exactly what the formulas below give for L = 0
                if (L != 0.f) {
                    r = 1.f / (1.f + expf(-L));
                    G = r * (1.f - r);
                    out[jo] = r;
                }
                if (WSUM) {
                    const float wj = upstream[jo];
                    sum_r += (double)wj * (double)(r - 0.5f);
                    G *= wj;
                } else {
                    sum_r += (double)(r - 0.5f);
                    if (HAS_UP) G *= upstream[jo];
                }
            }
            v[k] = G;
        }
        if (FOLD) continue;
        if (whole) reinterpret_cast<float4*>(carry)[q] = make_float4(v[0], v[1], v[2], v[3]);
        else for (int k = 0; k < 4 && q * 4 + k < n; ++k) carry[q * 4 + k] = v[k];
    }
    if (!FOLD) {
        const double ws = cov_warp_sum(sum_r);
        if ((threadIdx.x & 31) == 0 && ws != 0.0) atomicAdd(sum_slot, ws);
    }
}

// The long path's backward of one pose chunk: persistent warps over the chunk's kept work list (for_each_item), each item
// with the mask row its forward rewrote (the poses at which the warp gated a pair) and the 128 G_j of its points (cloud
// order, from the finalise kernel).  tiles_pose_backward for every pose of the mask: the (box, pose) pairs, m and terms of
// pass B's backward.  The item ticket is ctrl[2] (the forward drew ctrl[3]).
__global__ void __launch_bounds__(COV_THREADS, kTilesMinBlocks)
cov_traj_long_backward_kernel(const float* __restrict__ xyz, int64_t n, const float4* __restrict__ table, int W, CovConst C,
                              const float* __restrict__ G_dev, double* __restrict__ acc,
                              const unsigned* __restrict__ amask_g, int mask_stride, const int* __restrict__ worklist,
                              int* __restrict__ ctrl, unsigned long long* __restrict__ stats) {
    constexpr int PPT = kItemPpt;
    const int lane = threadIdx.x & 31;
    const int n_items = ctrl[0];
    const int nwords = (W + 31) >> 5;
    unsigned n_bwd = 0;
    for_each_item<false>(xyz, n, amask_g, mask_stride, nullptr, worklist, n_items, ctrl + 2, [](int) {},
                         [&](const Item& item) {
        unsigned any = 0u;
        for (int c = 0; c < nwords; ++c) any |= item.mask[c];
        if (any == 0u) return;
        float px[PPT], py[PPT], pz[PPT], G[PPT];
        bool valid[PPT];
        load_item_points<false>(item, xyz, n, lane, px, py, pz, valid);
#pragma unroll
        for (int s = 0; s < PPT; ++s) G[s] = valid[s] ? __ldg(G_dev + item.j0 + s * 32 + lane) : 0.f;
        for (int c = 0; c < nwords; ++c) {
            unsigned word = item.mask[c];
            while (word) {
                const int w = c * 32 + __ffs(word) - 1;
                word &= word - 1;
                ++n_bwd;
                tiles_pose_backward<PPT>(table + (size_t)w * COV_ROW_F4, px, py, pz, G, C, acc + (size_t)w * COV_ACC_STRIDE,
                                         lane);
            }
        }
    });
    if (stats && lane == 0) atomicAdd(stats + 4, (unsigned long long)n_bwd);
}

// Fused log-odds output, dense: every (point, pose) pair, the pose rows (with the normalisers, cov_norm_row) in shared
// memory; the same gate and log-odds terms in pose order as the dense pass B, hence the same L_j.
template <int PPT>
__global__ void __launch_bounds__(COV_THREADS, 2)
cov_traj_logodds_kernel(const float* __restrict__ xyz, int64_t n, const float* __restrict__ poses,
                        const float* __restrict__ quats, int W, const float* __restrict__ K9, CovConst C,
                        const float* __restrict__ minmax, const int32_t* __restrict__ out_index, float* __restrict__ out) {
    extern __shared__ float4 smem4[];
    const int tid = threadIdx.x;
    for (int w = tid; w < W; w += COV_THREADS) {
        float4* row = smem4 + (size_t)w * COV_ROW_F4;
        cov_pose_row(poses + 3 * w, quats + 4 * w, K9, C, row);
        cov_norm_row(row, minmax[w], minmax[W + w], row[3].w);  // conservative gate threshold in v3.w
    }
    __syncthreads();
    constexpr int T = COV_THREADS * PPT;
    const int64_t ntiles = (n + T - 1) / T;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        float px[PPT], py[PPT], pz[PPT], L[PPT];
        bool valid[PPT];
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            const int64_t j = tile * T + s * COV_THREADS + tid;
            valid[s] = j < n;
            px[s] = valid[s] ? __ldg(xyz + j * 3) : 3.0e18f;  // past the end: m = 0 exactly, never gated
            py[s] = valid[s] ? __ldg(xyz + j * 3 + 1) : 3.0e18f;
            pz[s] = valid[s] ? __ldg(xyz + j * 3 + 2) : 3.0e18f;
            L[s] = 0.f;
        }
        for (int w = 0; w < W; ++w) {
            const float4* row = smem4 + (size_t)w * COV_ROW_F4;
            const float4 v0 = row[0], v1 = row[1], v2 = row[2], v3 = row[3];
            float m[PPT];
#pragma unroll
            for (int s = 0; s < PPT; ++s) m[s] = cov_vis<false>(px[s], py[s], pz[s], v0, v1, v2, v3, C, nullptr);
            float mmax = m[0];
#pragma unroll
            for (int s = 1; s < PPT; ++s) mmax = fmaxf(mmax, m[s]);
            if (__any_sync(kFull, mmax >= v3.w)) {
                const float4 v4 = row[4];
#pragma unroll
                for (int s = 0; s < PPT; ++s) {
                    const float d = __fsub_rn(m[s], v4.w);
                    if (d >= v4.x) L[s] += cov_logodds(d, v4, C);  // exactly p >= 0.5
                }
            }
        }
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            if (valid[s] && L[s] != 0.f) {
                const int64_t j = tile * T + s * COV_THREADS + tid;
                const int64_t jo = out_index ? (int64_t)out_index[j] : j;
                out[jo] = cov_fuse_prior(out[jo], L[s]);
            }
        }
    }
}

// ==================================================== host ====================================================
constexpr size_t kSmemCap = (227 - 4) * 1024;  // opt-in shared memory per block on sm_100, minus static use
constexpr int64_t kSeedSamples = 16384;          // pruned pass A: size of the strided sample that seeds the bounds
constexpr int64_t kDenseBelow = 4 * kSeedSamples;  // clouds this small go straight to the dense kernels

// Resident blocks per SM of a kernel at a given dynamic shared-memory size, cached per (kernel, device, size): the
// opt-in shared-memory attribute is raised once per kernel and device to the cap (not per call: two host threads with
// different pose counts must not race between "set" and "launch"), the occupancy query runs once per size.
struct OccKey {
    const void* fn;
    int dev;
    size_t smem;
    bool operator<(const OccKey& o) const {
        return fn != o.fn ? fn < o.fn : dev != o.dev ? dev < o.dev : smem < o.smem;
    }
};
std::mutex g_occ_mutex;
std::map<OccKey, int> g_occ;

template <typename Kern>
int blocks_per_sm(Kern kern, int threads, size_t smem) {
    int dev = 0;
    cudaGetDevice(&dev);
    const OccKey key{reinterpret_cast<const void*>(kern), dev, smem};
    std::lock_guard<std::mutex> lock(g_occ_mutex);
    auto it = g_occ.find(key);
    if (it != g_occ.end()) return it->second;
    const OccKey attr_key{reinterpret_cast<const void*>(kern), dev, (size_t)-1};
    if (g_occ.find(attr_key) == g_occ.end()) {
        cudaFuncAttributes fa;
        size_t cap = kSmemCap;
        if (cudaFuncGetAttributes(&fa, kern) == cudaSuccess && fa.sharedSizeBytes + cap > 227 * 1024)
            cap = 227 * 1024 - fa.sharedSizeBytes;  // opt-in limit covers static + dynamic
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap) != cudaSuccess)
            cudaGetLastError();
        g_occ[attr_key] = 1;
    }
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem) != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        per_sm = 1;
    }
    g_occ[key] = per_sm;
    return per_sm;
}

// Grid of a persistent kernel: as many blocks as are resident at once, but no more than there are tiles.
template <typename Kern>
unsigned persistent_grid(Kern kern, size_t smem, int64_t ntiles) {
    const int64_t g = (int64_t)blocks_per_sm(kern, COV_THREADS, smem) * cov_sm_count_cached();
    return (unsigned)std::max<int64_t>(1, std::min<int64_t>(g, ntiles));
}
// the dense kernels: a block-stride loop over the tiles, at most COV_MAX_GRID blocks
template <typename Kern>
unsigned grid_for(Kern kern, size_t smem, int64_t ntiles) {
    return std::min(persistent_grid(kern, smem, ntiles), (unsigned)COV_MAX_GRID);
}

// points per thread of the DENSE kernels: the largest tile that still gives every SM two tiles and fits shared memory
int pick_ppt(int64_t n, int W, bool fused) {
    const int sms = cov_sm_count_cached();
    const int cand[3] = {4, 2, 1};
    for (int i = 0; i < 3; ++i) {
        const int ppt = cand[i];
        const size_t sm = fused ? fused_smem_bytes(W, ppt) : minmax_smem_bytes(W);
        if (sm > kSmemCap) continue;
        const int64_t ntiles = (n + tile_points(ppt) - 1) / tile_points(ppt);
        if (ntiles >= 2 * (int64_t)sms || ppt == 1) return ppt;
    }
    return 0;
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }
int64_t boxes_padded(int64_t n) { return ((n + 2047) / 2048) * (2048 / kBoxPts); }

// Work items the cull can list at most: every box of every 1024-point tile.
int64_t list_capacity(int64_t n) { return ((n + 1023) / 1024) * kTileBoxes; }

// Workspace of both passes (every region 256-byte aligned):
//   [control: ctrl ints | encoded extrema 2W | look-back descriptors][pose table][work list][box masks][boxes]
// The work list and the masks are sized for the worst case, every box listed: list_capacity entries, and as many mask
// rows of mask_stride_words(W), indexed by box.  The cull writes the rows of the listed boxes only.
struct TrajWorkspace {
    int* ctrl;
    unsigned* enc;
    unsigned long long* desc;
    size_t ctrl_bytes;  // the span a pruned call zeroes first
    float4* table;
    int* worklist;
    unsigned* amask;
    float4* boxes;
    size_t bytes;
};
TrajWorkspace carve_workspace(void* ws, int64_t n, int W) {
    const int64_t nt = (n + 1023) / 1024;  // tiles of the pruned passes
    const int64_t nchunks = (nt + kChunkTiles - 1) / kChunkTiles;
    const int64_t cap = list_capacity(n);
    char* p = reinterpret_cast<char*>(ws);
    size_t off = 0;
    TrajWorkspace t;
    auto take = [&](size_t bytes) { char* q = p + off; off += align256(bytes); return q; };
    const size_t enc_off = kCtrlInts * sizeof(int);
    const size_t desc_off = (enc_off + 2 * (size_t)W * sizeof(unsigned) + 7) & ~(size_t)7;
    t.ctrl_bytes = desc_off + (size_t)nchunks * sizeof(unsigned long long);
    char* c = take(t.ctrl_bytes);
    t.ctrl = reinterpret_cast<int*>(c);
    t.enc = reinterpret_cast<unsigned*>(c + enc_off);
    t.desc = reinterpret_cast<unsigned long long*>(c + desc_off);
    t.table = reinterpret_cast<float4*>(take((size_t)W * COV_ROW_F4 * sizeof(float4)));
    t.worklist = reinterpret_cast<int*>(take((size_t)cap * sizeof(int)));
    t.amask = reinterpret_cast<unsigned*>(take((size_t)cap * mask_stride_words(W) * sizeof(unsigned)));
    t.boxes = reinterpret_cast<float4*>(take((size_t)boxes_padded(n) * 2 * sizeof(float4)));
    t.bytes = off;
    return t;
}

int check_traj_args(const char* who, const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                    const float* K, const cov_camera* cam, const void* ws, size_t ws_bytes, bool pruned) {
    if (!xyz || n <= 0 || !poses || !quats || W <= 0 || !K || !cam) {
        cov_set_error("%s: null pointer, empty cloud or no poses (n=%lld, W=%d)", who, (long long)n, W);
        return COV_ERR_ARG;
    }
    // the dense kernels keep the pose table in shared memory; the pruned ones only a bit per pose in the box masks
    const int max_w = pruned ? cov_traj_max_poses_pruned() : cov_traj_max_poses();
    if (W > max_w) {
        cov_set_error("%s: %d poses exceed what one call takes on this path (max %d)", who, W, max_w);
        return COV_ERR_UNSUPPORTED;
    }
    if (n >= ((int64_t)1 << 31) * 256) {
        cov_set_error("%s: %lld points exceed the int32 tile index range", who, (long long)n);
        return COV_ERR_UNSUPPORTED;
    }
    if (!ws) {
        cov_set_error("%s: null workspace", who);
        return COV_ERR_ARG;
    }
    if (ws_bytes < cov_traj_workspace_bytes(n, W)) {
        cov_set_error("%s: workspace %zu < %zu bytes", who, ws_bytes, cov_traj_workspace_bytes(n, W));
        return COV_ERR_WORKSPACE;
    }
    if ((((uintptr_t)ws) & 255) || (((uintptr_t)xyz) & 15)) {
        cov_set_error("%s: workspace must be 256-byte aligned and the cloud 16-byte aligned", who);
        return COV_ERR_ALIGN;
    }
    return COV_OK;
}

void launch_tile_boxes(const float* xyz, int64_t n, float4* boxes, cudaStream_t s) {
    const int64_t nb = boxes_padded(n);
    const int grid = (int)std::min<int64_t>((nb + 7) / 8, (int64_t)cov_sm_count_cached() * 16);
    cov_tile_boxes_kernel<<<grid, 256, 0, s>>>(xyz, n, nb, boxes);
}

// boxes for this call: the caller's (cov_tile_boxes, once per cloud) or built into the workspace now
const float4* boxes_for_call(const float* xyz, int64_t n, const float* boxes_dev, const TrajWorkspace& t, cudaStream_t s) {
    if (boxes_dev) return reinterpret_cast<const float4*>(boxes_dev);
    launch_tile_boxes(xyz, n, t.boxes, s);
    return t.boxes;
}

// cull + work list in one launch (1024-point tiles of n points); every block must be resident (the blocks wait on one
// another's descriptors)
int launch_cull(const float4* boxes, int64_t n, const TrajWorkspace& t, int W, const unsigned* enc, float inv_kd,
                float* fill_dst, int64_t fill_n, cudaStream_t s, const float* fill_prior = nullptr) {
    const int64_t ntiles = (n + tile_points(4) - 1) / tile_points(4);
    const size_t smem = (size_t)W * sizeof(float4);
    const auto cull = fill_prior ? cov_cull_kernel<true> : cov_cull_kernel<false>;
    const int64_t nchunks = (ntiles + kChunkTiles - 1) / kChunkTiles;
    const int64_t resident = (int64_t)blocks_per_sm(cull, 256, smem) * cov_sm_count_cached();
    int64_t want = nchunks;
    if (fill_dst) want = std::max<int64_t>(want, (int64_t)cov_sm_count_cached() * 4);  // enough stores in flight for the fill
    int64_t g = std::max<int64_t>(1, std::min<int64_t>(want, resident));
    if ((nchunks + g - 1) / g > kCullMaxIter) {
        cov_set_error("cov_cull: %lld tiles exceed what one launch can list (%lld blocks x %d chunks)", (long long)ntiles,
                      (long long)g, kCullMaxIter);
        return COV_ERR_UNSUPPORTED;
    }
    const int grid = (int)g;
    cull<<<grid, 256, smem, s>>>(boxes, n, ntiles, t.table, W, enc, inv_kd, t.amask, mask_stride_words(W), t.worklist,
                                 t.ctrl, t.desc, fill_dst, fill_n, fill_prior);
    return COV_OK;
}

// ---- the long path (cov_traj_fused_long, cov_traj_logodds_long): poses in chunks, the fused log-odds carried ----
// Workspace: [boxes][carry: n floats][pose table: W rows][K chunk regions], every region 256-byte aligned.  A chunk region
// is [ctrl ints | look-back descriptors][work list][box masks of mask_stride_words(chunk) words]: pass B's control words,
// list and masks of one chunk, kept from its forward to its backward.
int long_chunk(int pose_chunk) { return pose_chunk > 0 ? pose_chunk : 32 * kMaskWords; }

TrajWorkspace carve_long_region(char* p, int64_t n, int Wc, float4* table) {
    const int64_t nt = (n + 1023) / 1024;
    const int64_t nchunks = (nt + kChunkTiles - 1) / kChunkTiles;
    const int64_t cap = list_capacity(n);
    size_t off = 0;
    auto take = [&](size_t bytes) { char* q = p + off; off += align256(bytes); return q; };
    TrajWorkspace t;
    t.ctrl_bytes = kCtrlInts * sizeof(int) + (size_t)nchunks * sizeof(unsigned long long);
    char* c = take(t.ctrl_bytes);
    t.ctrl = reinterpret_cast<int*>(c);
    t.enc = nullptr;
    t.desc = reinterpret_cast<unsigned long long*>(c + kCtrlInts * sizeof(int));
    t.table = table;
    t.worklist = reinterpret_cast<int*>(take((size_t)cap * sizeof(int)));
    t.amask = reinterpret_cast<unsigned*>(take((size_t)cap * mask_stride_words(Wc) * sizeof(unsigned)));
    t.boxes = nullptr;
    t.bytes = off;
    return t;
}

struct LongWorkspace {
    float4* boxes;
    float* carry;
    float4* table;
    char* regions;
    size_t region_bytes;
    size_t bytes;
};
LongWorkspace carve_long(void* ws, int64_t n, int W, int chunk) {
    char* p = reinterpret_cast<char*>(ws);
    size_t off = 0;
    auto take = [&](size_t bytes) { char* q = p + off; off += align256(bytes); return q; };
    LongWorkspace l;
    l.boxes = reinterpret_cast<float4*>(take((size_t)boxes_padded(n) * 2 * sizeof(float4)));
    l.carry = reinterpret_cast<float*>(take((size_t)n * sizeof(float)));
    l.table = reinterpret_cast<float4*>(take((size_t)W * COV_ROW_F4 * sizeof(float4)));
    l.region_bytes = carve_long_region(nullptr, n, std::min(chunk, W), nullptr).bytes;
    const int64_t k = (W + chunk - 1) / chunk;
    l.regions = take((size_t)k * l.region_bytes);
    l.bytes = off;
    return l;
}

}  // namespace

extern "C" int cov_traj_max_poses(void) {
    static int cached = 0;
    if (cached) return cached;
    int w = 1;
    while (w < 32 * kMaskWords && fused_smem_bytes(w + 1, 1) <= kSmemCap && minmax_smem_bytes(w + 1) <= kSmemCap &&
           (size_t)(w + 1) * sizeof(float4) <= 48 * 1024)
        ++w;
    cached = w;
    return w;
}

extern "C" int cov_traj_max_poses_pruned(void) { return 32 * kMaskWords; }

extern "C" size_t cov_traj_workspace_bytes(int64_t n, int n_poses) {
    if (n < 1) n = 1;
    if (n_poses < 1) n_poses = 1;
    return carve_workspace(nullptr, n, n_poses).bytes;
}

extern "C" int64_t cov_tile_boxes_count(int64_t n) { return n > 0 ? boxes_padded(n) : 0; }

extern "C" int cov_traj_prefill_applies(int64_t n, const cov_traj_opts* opts) {
    return (!(opts && opts->dense) && n >= kDenseBelow) ? 1 : 0;
}

extern "C" int cov_tile_boxes(const float* xyz, int64_t n, float* boxes, void* stream) {
    if (!xyz || !boxes || n <= 0) {
        cov_set_error("cov_tile_boxes: null pointer or empty cloud (n=%lld)", (long long)n);
        return COV_ERR_ARG;
    }
    if (((uintptr_t)boxes) & 15) {
        cov_set_error("cov_tile_boxes: boxes must be 16-byte aligned");
        return COV_ERR_ALIGN;
    }
    launch_tile_boxes(xyz, n, reinterpret_cast<float4*>(boxes), (cudaStream_t)stream);
    return cov_check_launch("cov_tile_boxes");
}

// The prior (16-byte aligned, indexed like the rewards buffer) of the _prior entry points: present and aligned.
static int check_prior(const char* who, const float* prior, const double* prior_sum, bool need_sum) {
    if (!prior || (need_sum && !prior_sum)) {
        cov_set_error("%s: null prior_dev or prior_sum_dev", who);
        return COV_ERR_ARG;
    }
    if (((uintptr_t)prior) & 15) {
        cov_set_error("%s: prior_dev must be 16-byte aligned", who);
        return COV_ERR_ALIGN;
    }
    return COV_OK;
}

// The weight (16-byte aligned, indexed like the prior) and the 2-double sums of the _weighted entry points.
static int check_weight(const char* who, const float* weight, const double* weight_sums, const float* prior) {
    if (!weight || !weight_sums) {
        cov_set_error("%s: null weight_dev or weight_sums_dev", who);
        return COV_ERR_ARG;
    }
    if ((((uintptr_t)weight) & 15) || (((uintptr_t)prior) & 15)) {
        cov_set_error("%s: weight_dev and prior_dev must be 16-byte aligned", who);
        return COV_ERR_ALIGN;
    }
    return COV_OK;
}

static int traj_minmax_impl(const float* xyz, int64_t n, const float* poses, const float* quats, int W, const float* K,
                            const cov_camera* cam, const float* boxes_dev, float* minmax, const float* prior,
                            const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream) {
    const bool prune = !(opts && opts->dense) && n >= kDenseBelow;
    int rc = check_traj_args("cov_traj_minmax", xyz, n, poses, quats, W, K, cam, ws, ws_bytes, prune);
    if (rc) return rc;
    if (!minmax) {
        cov_set_error("cov_traj_minmax: null minmax");
        return COV_ERR_ARG;
    }
    if (boxes_dev && (((uintptr_t)boxes_dev) & 15)) {
        cov_set_error("cov_traj_minmax: boxes must be 16-byte aligned");
        return COV_ERR_ALIGN;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    int ppt = prune ? 4 : pick_ppt(n, W, false);
    if (ppt == 4 && (n + tile_points(8) - 1) / tile_points(8) >= 4 * (int64_t)cov_sm_count_cached()) ppt = 8;
    if (ppt == 0) {
        cov_set_error("cov_traj_minmax: %d poses do not fit in shared memory", W);
        return COV_ERR_UNSUPPORTED;
    }
    const int64_t ntiles = (n + tile_points(ppt) - 1) / tile_points(ppt);
    if (!prune) {
        // (prefill_dev is not honoured here: the dense pass B writes every reward itself)
        unsigned* gmin = reinterpret_cast<unsigned*>(minmax);
        unsigned* gmax = gmin + W;
        const size_t smem = minmax_smem_bytes(W);
        cov_minmax_init_kernel<<<(W + 255) / 256, 256, 0, s>>>(gmin, gmax, W);
#define LAUNCH_DENSE(P, B)                                                                                       \
    {                                                                                                            \
        const int grid = grid_for(cov_traj_minmax_kernel<P, B>, smem, ntiles);                                   \
        cov_traj_minmax_kernel<P, B><<<grid, COV_THREADS, smem, s>>>(xyz, n, poses, quats, W, K, C, gmin, gmax); \
    }
        if (ppt == 8) LAUNCH_DENSE(8, 2)
        else if (ppt == 4) LAUNCH_DENSE(4, 2)
        else if (ppt == 2) LAUNCH_DENSE(2, 2)
        else LAUNCH_DENSE(1, 2)
#undef LAUNCH_DENSE
        return cov_check_launch("cov_traj_minmax");
    }
    // pruned: pose table + seed on a strided sample, cull + work list, evaluation of the listed boxes: 3 launches
    const TrajWorkspace t = carve_workspace(ws, n, W);
    const float4* boxes = boxes_for_call(xyz, n, boxes_dev, t, s);
    constexpr int ppt_t = 4;  // tiles of 1024 points, eight 128-point items each (as pass B)
    const int64_t ntiles_t = (n + tile_points(ppt_t) - 1) / tile_points(ppt_t);
    cudaMemsetAsync(t.ctrl, 0, t.ctrl_bytes, s);
    {
        const int64_t stride = (n + kSeedSamples - 1) / kSeedSamples;
        const int64_t nsamples = (n + stride - 1) / stride;
        const dim3 sgrid((unsigned)((nsamples + COV_THREADS - 1) / COV_THREADS), (unsigned)((W + 31) / 32));
        cov_traj_prepare_kernel<<<sgrid, COV_THREADS, 0, s>>>(xyz, nsamples, stride, poses, quats, W, K, C, t.table, t.enc);
    }
    if ((rc = launch_cull(boxes, n, t, W, t.enc, 1.f / C.kd, nullptr, 0, s)) != COV_OK) return rc;
    const size_t smem_t = (size_t)W * 12;
    float* prefill = opts ? opts->prefill_dev : nullptr;
    const auto tiles_kern = (prior && prefill) ? cov_traj_minmax_tiles_kernel<true> : cov_traj_minmax_tiles_kernel<false>;
    tiles_kern<<<persistent_grid(tiles_kern, smem_t, ntiles_t), COV_THREADS, smem_t, s>>>(
        xyz, n, t.table, W, C, t.enc, minmax, t.amask, mask_stride_words(W), t.worklist, t.ctrl, ntiles_t,
        opts ? opts->stats_dev : nullptr, prefill, n, prior);
    return cov_check_launch("cov_traj_minmax");
}

extern "C" int cov_traj_minmax(const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                               const float* K, const cov_camera* cam, const float* boxes_dev, float* minmax,
                               const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream) {
    return traj_minmax_impl(xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, nullptr, opts, ws, ws_bytes, stream);
}

extern "C" int cov_traj_minmax_prior(const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                                     const float* K, const cov_camera* cam, const float* boxes_dev, float* minmax,
                                     const float* prior, const cov_traj_opts* opts, void* ws, size_t ws_bytes,
                                     void* stream) {
    const int rc = check_prior("cov_traj_minmax_prior", prior, nullptr, false);
    if (rc) return rc;
    return traj_minmax_impl(xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, prior, opts, ws, ws_bytes, stream);
}

static int traj_fused_impl(const float* xyz, int64_t n, const float* poses, const float* quats, int W, const float* K,
                           const cov_camera* cam, const float* boxes_dev, const float* minmax, const float* upstream,
                           const int32_t* reward_index, float* rewards, double* acc, const float* prior,
                           const double* prior_sum, const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream,
                           const float* weight = nullptr, const double* weight_sums = nullptr) {
    // point weights ride on the upstream gather (WSUM); the reward sum starts at sum_j w_j r0_j instead
    const bool wsum = weight != nullptr;
    if (wsum) {
        upstream = weight;
        prior_sum = weight_sums;
    }
    const bool prune = !(opts && opts->dense) && n >= kDenseBelow;
    int rc = check_traj_args("cov_traj_fused", xyz, n, poses, quats, W, K, cam, ws, ws_bytes, prune);
    if (rc) return rc;
    if (!minmax || !rewards || !acc) {
        cov_set_error("cov_traj_fused: null minmax/rewards/acc");
        return COV_ERR_ARG;
    }
    if ((boxes_dev && (((uintptr_t)boxes_dev) & 15)) || (reward_index && (((uintptr_t)reward_index) & 15))) {
        cov_set_error("cov_traj_fused: boxes and reward_index must be 16-byte aligned");
        return COV_ERR_ALIGN;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    const TrajWorkspace t = carve_workspace(ws, n, W);
    if (!prune) {  // every pair evaluated: accumulators zeroed, one kernel
        const int ppt_d = pick_ppt(n, W, true);
        if (ppt_d == 0) {
            cov_set_error("cov_traj_fused: %d poses do not fit in shared memory", W);
            return COV_ERR_UNSUPPORTED;
        }
        cudaMemsetAsync(acc, 0, ((size_t)W * COV_ACC_STRIDE + 1) * sizeof(double), s);
        const size_t smem = fused_smem_bytes(W, ppt_d);
        const int64_t ntiles = (n + tile_points(ppt_d) - 1) / tile_points(ppt_d);
        // phase-2 parallelism: split each pose row over 2^seg_log2 lanes until there are >= 2 tasks per thread
        int seg_log2 = 0;
        while ((W << seg_log2) < 2 * COV_THREADS && (2 << seg_log2) <= bit_words(ppt_d) && seg_log2 < 5) ++seg_log2;
#define LAUNCH_F(P, UP, PR, WS)                                                                                    \
    {                                                                                                              \
        const int grid = grid_for(cov_traj_fused_kernel<P, UP, PR, WS>, smem, ntiles);                             \
        cov_traj_fused_kernel<P, UP, PR, WS><<<grid, COV_THREADS, smem, s>>>(xyz, n, poses, quats, W, K, C, minmax, \
                                                                             upstream, reward_index, rewards, acc, \
                                                                             seg_log2, prior);                     \
    }
#define LAUNCH_FP(UP, PR) \
    if (ppt_d == 4) LAUNCH_F(4, UP, PR, false) else if (ppt_d == 2) LAUNCH_F(2, UP, PR, false) else LAUNCH_F(1, UP, PR, false)
#define LAUNCH_FW(PR) \
    if (ppt_d == 4) LAUNCH_F(4, true, PR, true) else if (ppt_d == 2) LAUNCH_F(2, true, PR, true) else LAUNCH_F(1, true, PR, true)
        if (wsum) {
            if (prior) { LAUNCH_FW(true) } else { LAUNCH_FW(false) }
        } else if (upstream) {
            if (prior) { LAUNCH_FP(true, true) } else { LAUNCH_FP(true, false) }
        } else {
            if (prior) { LAUNCH_FP(false, true) } else { LAUNCH_FP(false, false) }
        }
#undef LAUNCH_FW
#undef LAUNCH_FP
#undef LAUNCH_F
        return cov_check_launch("cov_traj_fused");
    }
    // pruned: table (+ zeroing), cull + work list (+ rewards pre-fill), evaluation of the listed boxes: 3 launches
    constexpr int ppt = 4;  // tiles of 1024 points, eight 128-point boxes each
    static_assert(tile_boxes(ppt) == kTileBoxes, "the cull's tiles");
    const int64_t ntiles = (n + tile_points(ppt) - 1) / tile_points(ppt);
    const float4* boxes = boxes_for_call(xyz, n, boxes_dev, t, s);
    if (prior || wsum) {
        cov_traj_table_kernel<true><<<(W + 63) / 64, 64, 0, s>>>(poses, quats, W, K, C, minmax, t.table, t.ctrl,
                                                                 (int)(t.ctrl_bytes / sizeof(int)), acc, 0.0, prior_sum);
    } else {
        cov_traj_table_kernel<false><<<(W + 63) / 64, 64, 0, s>>>(poses, quats, W, K, C, minmax, t.table, t.ctrl,
                                                                  (int)(t.ctrl_bytes / sizeof(int)), acc, 0.5 * (double)n,
                                                                  nullptr);
    }
    const bool prefilled = opts && opts->rewards_prefilled;
    if ((rc = launch_cull(boxes, n, t, W, nullptr, 0.f, prefilled ? nullptr : rewards, n, s, prior)) != COV_OK)
        return rc;
    // persistent warps: as many blocks as are resident; every warp draws 128-point items from a ticket counter
    const auto tiles_kern =
        wsum ? (prior ? cov_traj_fused_tiles_kernel<true, true, true> : cov_traj_fused_tiles_kernel<true, false, true>)
        : upstream ? (prior ? cov_traj_fused_tiles_kernel<true, true> : cov_traj_fused_tiles_kernel<true, false>)
                   : (prior ? cov_traj_fused_tiles_kernel<false, true> : cov_traj_fused_tiles_kernel<false, false>);
    tiles_kern<<<persistent_grid(tiles_kern, 0, ntiles), COV_THREADS, 0, s>>>(
        xyz, n, t.table, W, C, upstream, reward_index, rewards, acc, t.amask, mask_stride_words(W), t.worklist,
        t.ctrl, ntiles, opts ? opts->stats_dev : nullptr, prior);
    return cov_check_launch("cov_traj_fused");
}

extern "C" int cov_traj_fused(const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                              const float* K, const cov_camera* cam, const float* boxes_dev, const float* minmax,
                              const float* upstream, const int32_t* reward_index, float* rewards, double* acc,
                              const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream) {
    return traj_fused_impl(xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, upstream, reward_index, rewards, acc,
                           nullptr, nullptr, opts, ws, ws_bytes, stream);
}

extern "C" int cov_traj_fused_prior(const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                                    const float* K, const cov_camera* cam, const float* boxes_dev, const float* minmax,
                                    const float* upstream, const int32_t* reward_index, float* rewards, double* acc,
                                    const float* prior, const double* prior_sum, const cov_traj_opts* opts, void* ws,
                                    size_t ws_bytes, void* stream) {
    const int rc = check_prior("cov_traj_fused_prior", prior, prior_sum, true);
    if (rc) return rc;
    return traj_fused_impl(xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, upstream, reward_index, rewards, acc,
                           prior, prior_sum, opts, ws, ws_bytes, stream);
}

extern "C" int cov_traj_fused_weighted(const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                                       const float* K, const cov_camera* cam, const float* boxes_dev, const float* minmax,
                                       const int32_t* reward_index, float* rewards, double* acc, const float* prior,
                                       const float* weight, const double* weight_sums, const cov_traj_opts* opts, void* ws,
                                       size_t ws_bytes, void* stream) {
    const int rc = check_weight("cov_traj_fused_weighted", weight, weight_sums, prior);
    if (rc) return rc;
    return traj_fused_impl(xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, nullptr, reward_index, rewards, acc, prior,
                           nullptr, opts, ws, ws_bytes, stream, weight, weight_sums);
}

extern "C" int cov_weight_sums(const float* weight, const float* prior, int64_t n, double* sums_out, void* stream) {
    if (!weight || !sums_out || n < 0) {
        cov_set_error("cov_weight_sums: null pointer or negative size (n=%lld)", (long long)n);
        return COV_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    cudaMemsetAsync(sums_out, 0, 2 * sizeof(double), s);
    if (n > 0) {
        const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)cov_sm_count_cached() * 8);
        if (prior) cov_weight_sums_kernel<true><<<grid, 256, 0, s>>>(weight, prior, n, sums_out);
        else cov_weight_sums_kernel<false><<<grid, 256, 0, s>>>(weight, nullptr, n, sums_out);
    }
    return cov_check_launch("cov_weight_sums");
}

extern "C" int cov_prior_reward_sum(const float* prior, int64_t n, double* sum_out, void* stream) {
    if (!prior || !sum_out || n < 0) {
        cov_set_error("cov_prior_reward_sum: null pointer or negative size (n=%lld)", (long long)n);
        return COV_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    cudaMemsetAsync(sum_out, 0, sizeof(double), s);
    if (n > 0) {
        const int grid = (int)std::min<int64_t>((n + 255) / 256, (int64_t)cov_sm_count_cached() * 8);
        cov_prior_sum_kernel<<<grid, 256, 0, s>>>(prior, n, sum_out);
    }
    return cov_check_launch("cov_prior_reward_sum");
}

extern "C" int cov_traj_logodds(const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                                const float* K, const cov_camera* cam, const float* boxes_dev, const float* minmax,
                                const int32_t* reward_index, float* logodds, const cov_traj_opts* opts, void* ws,
                                size_t ws_bytes, void* stream) {
    const bool prune = !(opts && opts->dense) && n >= kDenseBelow;
    int rc = check_traj_args("cov_traj_logodds", xyz, n, poses, quats, W, K, cam, ws, ws_bytes, prune);
    if (rc) return rc;
    if (!minmax || !logodds) {
        cov_set_error("cov_traj_logodds: null minmax/logodds");
        return COV_ERR_ARG;
    }
    if ((boxes_dev && (((uintptr_t)boxes_dev) & 15)) || (reward_index && (((uintptr_t)reward_index) & 15))) {
        cov_set_error("cov_traj_logodds: boxes and reward_index must be 16-byte aligned");
        return COV_ERR_ALIGN;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    if (!prune) {
        constexpr int ppt_d = 4;
        const size_t smem = (size_t)W * COV_ROW_F4 * sizeof(float4);
        if (smem > kSmemCap) {
            cov_set_error("cov_traj_logodds: %d poses do not fit in shared memory", W);
            return COV_ERR_UNSUPPORTED;
        }
        const int64_t ntiles = (n + COV_THREADS * ppt_d - 1) / (COV_THREADS * ppt_d);
        const int grid = grid_for(cov_traj_logodds_kernel<ppt_d>, smem, ntiles);
        cov_traj_logodds_kernel<ppt_d><<<grid, COV_THREADS, smem, s>>>(xyz, n, poses, quats, W, K, C, minmax, reward_index,
                                                                       logodds);
        return cov_check_launch("cov_traj_logodds");
    }
    // pruned: pass B's table and cull (no accumulators, no pre-fill), then its forward over the listed boxes
    constexpr int ppt = 4;
    const int64_t ntiles = (n + tile_points(ppt) - 1) / tile_points(ppt);
    const TrajWorkspace t = carve_workspace(ws, n, W);
    const float4* boxes = boxes_for_call(xyz, n, boxes_dev, t, s);
    cov_traj_table_kernel<false><<<(W + 63) / 64, 64, 0, s>>>(poses, quats, W, K, C, minmax, t.table, t.ctrl,
                                                              (int)(t.ctrl_bytes / sizeof(int)), nullptr, 0.0, nullptr);
    if ((rc = launch_cull(boxes, n, t, W, nullptr, 0.f, nullptr, 0, s)) != COV_OK) return rc;
    cov_traj_logodds_tiles_kernel<><<<persistent_grid(cov_traj_logodds_tiles_kernel<>, 0, ntiles), COV_THREADS, 0, s>>>(
        xyz, n, t.table, W, C, reward_index, logodds, t.amask, mask_stride_words(W), t.worklist, t.ctrl);
    return cov_check_launch("cov_traj_logodds");
}

extern "C" size_t cov_traj_long_workspace_bytes(int64_t n, int W, int pose_chunk) {
    if (n < 1) n = 1;
    if (W < 1) W = 1;
    const int max_chunk = 32 * kMaskWords;
    const int c0 = (pose_chunk < 1 || pose_chunk > max_chunk) ? max_chunk : pose_chunk;
    // the largest layout of any chunk >= c0, so that the size never grows with the chunk (a workspace sized for one
    // chunk serves every larger one); and at least the single-call workspace pass A runs its chunks in
    size_t bytes = cov_traj_workspace_bytes(n, std::min(W, max_chunk));
    for (int c = c0; c <= std::max(c0, std::min(W, max_chunk)); ++c) bytes = std::max(bytes, carve_long(nullptr, n, W, c).bytes);
    return bytes;
}

// The long path.  FOLD: cov_traj_logodds_long (out = the log-odds buffer; no accumulators, no backward).
static int traj_long_impl(const char* who, const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                          const float* K, const cov_camera* cam, const float* boxes_dev, const float* minmax,
                          const float* upstream, const int32_t* reward_index, float* out, double* acc, const float* prior,
                          const double* base, const float* weight, int pose_chunk, const cov_traj_opts* opts, void* ws,
                          size_t ws_bytes, void* stream, bool fold) {
    if (!xyz || n <= 0 || !poses || !quats || W <= 0 || !K || !cam || !minmax || !out || (!fold && !acc)) {
        cov_set_error("%s: null pointer, empty cloud or no poses (n=%lld, W=%d)", who, (long long)n, W);
        return COV_ERR_ARG;
    }
    if (pose_chunk < 0 || pose_chunk > 32 * kMaskWords) {
        cov_set_error("%s: pose_chunk %d outside 0 .. %d", who, pose_chunk, 32 * kMaskWords);
        return COV_ERR_ARG;
    }
    int rc = COV_OK;
    if (!fold) {  // base: NULL without prior and weight, cov_prior_reward_sum with a prior alone, cov_weight_sums with a weight
        if (weight && upstream) {
            cov_set_error("%s: weight_dev and upstream_dev are never given together", who);
            return COV_ERR_ARG;
        }
        if (weight) rc = check_weight(who, weight, base, prior);
        else if (prior) rc = check_prior(who, prior, base, true);
        else if (base) {
            cov_set_error("%s: base_dev must be NULL without prior_dev and weight_dev", who);
            rc = COV_ERR_ARG;
        }
        if (rc) return rc;
    }
    if (opts && opts->dense) {  // no dense long path: what one dense call takes, it takes
        if (W > cov_traj_max_poses()) {
            cov_set_error("%s: %d poses exceed what one call takes on this path (max %d)", who, W, cov_traj_max_poses());
            return COV_ERR_UNSUPPORTED;
        }
        if (fold)
            return cov_traj_logodds(xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, reward_index, out, opts, ws, ws_bytes,
                                    stream);
        return traj_fused_impl(xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, upstream, reward_index, out, acc, prior,
                               weight ? nullptr : base, opts, ws, ws_bytes, stream, weight, weight ? base : nullptr);
    }
    if (n >= ((int64_t)1 << 31) * 256) {
        cov_set_error("%s: %lld points exceed the int32 tile index range", who, (long long)n);
        return COV_ERR_UNSUPPORTED;
    }
    if (!ws) {
        cov_set_error("%s: null workspace", who);
        return COV_ERR_ARG;
    }
    const size_t need = cov_traj_long_workspace_bytes(n, W, pose_chunk);
    if (ws_bytes < need) {
        cov_set_error("%s: workspace %zu < cov_traj_long_workspace_bytes(n, %d, %d) = %zu", who, ws_bytes, W, pose_chunk,
                      need);
        return COV_ERR_WORKSPACE;
    }
    if ((((uintptr_t)ws) & 255) || (((uintptr_t)xyz) & 15) || (boxes_dev && (((uintptr_t)boxes_dev) & 15)) ||
        (reward_index && (((uintptr_t)reward_index) & 15))) {
        cov_set_error("%s: workspace must be 256-byte aligned, the cloud, boxes and reward_index 16-byte aligned", who);
        return COV_ERR_ALIGN;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    const int chunk = long_chunk(pose_chunk);
    const LongWorkspace l = carve_long(ws, n, W, chunk);
    const float4* boxes = boxes_dev ? reinterpret_cast<const float4*>(boxes_dev) : l.boxes;
    if (!boxes_dev) launch_tile_boxes(xyz, n, l.boxes, s);
    constexpr int ppt = 4;  // tiles of 1024 points, eight 128-point boxes each
    const int64_t ntiles = (n + tile_points(ppt) - 1) / tile_points(ppt);
    unsigned long long* stats = (opts && !fold) ? opts->stats_dev : nullptr;
    const bool prefilled = opts && opts->rewards_prefilled;
    const bool sum_dev = prior || weight;
    const int nk = (W + chunk - 1) / chunk;
    auto region = [&](int k) {
        return carve_long_region(l.regions + (size_t)k * l.region_bytes, n, std::min(chunk, W),
                                 l.table + (size_t)k * chunk * COV_ROW_F4);
    };
    cudaMemsetAsync(l.carry, 0, (size_t)n * sizeof(float), s);
    // forward, chunk by chunk: pass B's table (chunk rows of the accumulators zeroed), cull + work list (the first also
    // pre-fills the rewards), then the CARRY forward over the listed boxes
    const auto fwd = cov_traj_logodds_tiles_kernel<true>;
    for (int k = 0; k < nk; ++k) {
        const int w0 = k * chunk, Wc = std::min(chunk, W - w0);
        const TrajWorkspace t = region(k);
        double* acc_k = fold ? nullptr : acc + (size_t)w0 * COV_ACC_STRIDE;
        const int ctrl_words = (int)(t.ctrl_bytes / sizeof(int));
        if (sum_dev)
            cov_traj_table_kernel<true, true><<<(Wc + 63) / 64, 64, 0, s>>>(poses + 3 * (size_t)w0, quats + 4 * (size_t)w0,
                                                                           Wc, K, C, minmax, t.table, t.ctrl, ctrl_words,
                                                                           acc_k, 0.0, base, w0, W);
        else
            cov_traj_table_kernel<false, true><<<(Wc + 63) / 64, 64, 0, s>>>(poses + 3 * (size_t)w0, quats + 4 * (size_t)w0,
                                                                            Wc, K, C, minmax, t.table, t.ctrl, ctrl_words,
                                                                            acc_k, 0.5 * (double)n, nullptr, w0, W);
        const bool fill = k == 0 && !fold && !prefilled;
        if ((rc = launch_cull(boxes, n, t, Wc, nullptr, 0.f, fill ? out : nullptr, n, s, fill ? prior : nullptr)) != COV_OK)
            return rc;
        fwd<<<persistent_grid(fwd, 0, ntiles), COV_THREADS, 0, s>>>(xyz, n, t.table, Wc, C, nullptr, nullptr, t.amask,
                                                                     mask_stride_words(Wc), t.worklist, t.ctrl, acc_k,
                                                                     l.carry, fold ? nullptr : t.amask, ntiles, stats);
    }
    // finalise: r_j, the reward sum and G_j (FOLD: the fused log-odds) from the carried L_j
    {
        const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((n / 4 + 255) / 256, (int64_t)cov_sm_count_cached() * 8));
        double* sum_slot = fold ? nullptr : acc + (size_t)W * COV_ACC_STRIDE;
        const float* up = weight ? weight : upstream;
#define LAUNCH_FIN(FO, UP, PR, WS) \
    cov_traj_long_finalise_kernel<FO, UP, PR, WS><<<grid, 256, 0, s>>>(n, l.carry, reward_index, out, up, prior, sum_slot)
        if (fold) LAUNCH_FIN(true, false, false, false);
        else if (weight) { if (prior) LAUNCH_FIN(false, true, true, true); else LAUNCH_FIN(false, true, false, true); }
        else if (upstream) { if (prior) LAUNCH_FIN(false, true, true, false); else LAUNCH_FIN(false, true, false, false); }
        else if (prior) LAUNCH_FIN(false, false, true, false);
        else LAUNCH_FIN(false, false, false, false);
#undef LAUNCH_FIN
    }
    if (fold) return cov_check_launch(who);
    // backward, chunk by chunk, over the kept work lists and rewritten masks
    const auto bwd = cov_traj_long_backward_kernel;
    for (int k = 0; k < nk; ++k) {
        const int w0 = k * chunk, Wc = std::min(chunk, W - w0);
        const TrajWorkspace t = region(k);
        bwd<<<persistent_grid(bwd, 0, ntiles), COV_THREADS, 0, s>>>(xyz, n, t.table, Wc, C, l.carry,
                                                                     acc + (size_t)w0 * COV_ACC_STRIDE, t.amask,
                                                                     mask_stride_words(Wc), t.worklist, t.ctrl, stats);
    }
    return cov_check_launch(who);
}

extern "C" int cov_traj_fused_long(const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                                   const float* K, const cov_camera* cam, const float* boxes_dev, const float* minmax,
                                   const float* upstream, const int32_t* reward_index, float* rewards, double* acc,
                                   const float* prior, const double* base, const float* weight, int pose_chunk,
                                   const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream) {
    return traj_long_impl("cov_traj_fused_long", xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, upstream, reward_index,
                          rewards, acc, prior, base, weight, pose_chunk, opts, ws, ws_bytes, stream, false);
}

extern "C" int cov_traj_logodds_long(const float* xyz, int64_t n, const float* poses, const float* quats, int W,
                                     const float* K, const cov_camera* cam, const float* boxes_dev, const float* minmax,
                                     const int32_t* reward_index, float* logodds, int pose_chunk,
                                     const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream) {
    return traj_long_impl("cov_traj_logodds_long", xyz, n, poses, quats, W, K, cam, boxes_dev, minmax, nullptr,
                          reward_index, logodds, nullptr, nullptr, nullptr, nullptr, pose_chunk, opts, ws, ws_bytes, stream,
                          true);
}

// prefix: the per-pose slots of cov_sweep_prefix_rewards (sum_rewards holds n_traj * per_traj doubles; the caller scans)
static int sweep_rewards_impl(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                              int per_traj, const float* K, const cov_camera* cam, const float* boxes_dev,
                              const float* minmax, double* sum_rewards, const float* prior, const double* prior_sum,
                              const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream,
                              const float* weight = nullptr, bool prefix = false) {
    const char* who = prefix ? "cov_sweep_prefix_rewards" : "cov_sweep_rewards";
    if (!xyz || n <= 0 || !poses || !quats || n_traj <= 0 || per_traj <= 0 || !K || !cam || !minmax || !sum_rewards) {
        cov_set_error("%s: bad argument", who);
        return COV_ERR_ARG;
    }
    if (opts && opts->dense)
        return cov_sweep_rewards_dense(xyz, n, poses, quats, n_traj, per_traj, K, cam, minmax, sum_rewards, prior,
                                       prior_sum, weight, stream, prefix);
    // trajectories per launch: as many as the per-box pose mask holds (32 * kMaskWords poses); the pose table stays in
    // global memory, the block keeps one fp64 total per trajectory (prefix: per pose) in shared memory
    if (per_traj > 32 * kMaskWords) {
        cov_set_error("%s: %d poses per trajectory exceed the pose mask (%d)", who, per_traj, 32 * kMaskWords);
        return COV_ERR_UNSUPPORTED;
    }
    int chunk = (32 * kMaskWords) / per_traj;
    if (chunk > n_traj) chunk = n_traj;
    const int Wc = chunk * per_traj;
    if (!ws || ws_bytes < cov_sweep_workspace_bytes(n, n_traj, per_traj) || (((uintptr_t)ws) & 255) || (((uintptr_t)xyz) & 15)) {
        cov_set_error("%s: workspace missing, misaligned or smaller than cov_sweep_workspace_bytes(n, %d, %d) = %zu", who,
                      n_traj, per_traj, cov_sweep_workspace_bytes(n, n_traj, per_traj));
        return COV_ERR_WORKSPACE;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    const TrajWorkspace t = carve_workspace(ws, n, Wc);
    const float4* boxes = boxes_for_call(xyz, n, boxes_dev, t, s);
    const int W = n_traj * per_traj;
    constexpr int ppt = 4;  // tiles of 1024 points, eight 128-point items each
    const int64_t ntiles = (n + tile_points(ppt) - 1) / tile_points(ppt);
    float* mm = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + t.bytes);  // the chunk's minima and maxima, contiguous
    for (int t0 = 0; t0 < n_traj; t0 += chunk) {
        const int nt = (n_traj - t0 < chunk) ? n_traj - t0 : chunk;
        const int w0 = t0 * per_traj, Wn = nt * per_traj;
        cudaMemcpyAsync(mm, minmax + w0, (size_t)Wn * sizeof(float), cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(mm + Wn, minmax + W + w0, (size_t)Wn * sizeof(float), cudaMemcpyDeviceToDevice, s);
        cov_traj_table_kernel<false><<<(Wn + 63) / 64, 64, 0, s>>>(poses + 3 * (size_t)w0, quats + 4 * (size_t)w0, Wn, K, C, mm,
                                                                   t.table, t.ctrl, (int)(t.ctrl_bytes / sizeof(int)), nullptr,
                                                                   0.0, nullptr);
        if (launch_cull(boxes, n, t, Wn, nullptr, 0.f, nullptr, 0, s) != COV_OK) return COV_ERR_UNSUPPORTED;
        const size_t smem = (size_t)(prefix ? Wn : nt) * sizeof(double);
        const auto kern =
            prefix ? (weight ? (prior ? cov_sweep_tiles_kernel<true, true, true> : cov_sweep_tiles_kernel<false, true, true>)
                             : (prior ? cov_sweep_tiles_kernel<true, false, true> : cov_sweep_tiles_kernel<false, false, true>))
                   : (weight ? (prior ? cov_sweep_tiles_kernel<true, true> : cov_sweep_tiles_kernel<false, true>)
                             : (prior ? cov_sweep_tiles_kernel<true> : cov_sweep_tiles_kernel<false>));
        kern<<<persistent_grid(kern, smem, ntiles), COV_THREADS, smem, s>>>(
            xyz, n, t.table, Wn, per_traj, nt, C, t.amask, mask_stride_words(Wn), t.worklist, t.ctrl,
            sum_rewards + (prefix ? w0 : t0), prior, prior_sum, weight);
    }
    return cov_check_launch(who);
}

extern "C" int cov_sweep_rewards(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                                 int per_traj, const float* K, const cov_camera* cam, const float* boxes_dev,
                                 const float* minmax, double* sum_rewards, const cov_traj_opts* opts, void* ws,
                                 size_t ws_bytes, void* stream) {
    return sweep_rewards_impl(xyz, n, poses, quats, n_traj, per_traj, K, cam, boxes_dev, minmax, sum_rewards, nullptr,
                              nullptr, opts, ws, ws_bytes, stream);
}

extern "C" int cov_sweep_rewards_prior(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                                       int per_traj, const float* K, const cov_camera* cam, const float* boxes_dev,
                                       const float* minmax, double* sum_rewards, const float* prior,
                                       const double* prior_sum, const cov_traj_opts* opts, void* ws, size_t ws_bytes,
                                       void* stream) {
    const int rc = check_prior("cov_sweep_rewards_prior", prior, prior_sum, true);
    if (rc) return rc;
    return sweep_rewards_impl(xyz, n, poses, quats, n_traj, per_traj, K, cam, boxes_dev, minmax, sum_rewards, prior,
                              prior_sum, opts, ws, ws_bytes, stream);
}

extern "C" int cov_sweep_rewards_weighted(const float* xyz, int64_t n, const float* poses, const float* quats,
                                          int n_traj, int per_traj, const float* K, const cov_camera* cam,
                                          const float* boxes_dev, const float* minmax, double* sum_rewards,
                                          const float* prior, const float* weight, const double* weight_sums,
                                          const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream) {
    const int rc = check_weight("cov_sweep_rewards_weighted", weight, weight_sums, prior);
    if (rc) return rc;
    // the weighted base sum_j w_j r0_j takes the place of the prior's sum
    return sweep_rewards_impl(xyz, n, poses, quats, n_traj, per_traj, K, cam, boxes_dev, minmax, sum_rewards, prior,
                              weight_sums, opts, ws, ws_bytes, stream, weight);
}

extern "C" int cov_sweep_prefix_rewards(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                                        int per_traj, const float* K, const cov_camera* cam, const float* boxes_dev,
                                        const float* minmax, const float* prior, const float* weight, const double* base,
                                        double* prefix_sums, const cov_traj_opts* opts, void* ws, size_t ws_bytes,
                                        void* stream) {
    // base: NULL (n / 2) without prior and weight, cov_prior_reward_sum with a prior alone, cov_weight_sums with a weight
    int rc = COV_OK;
    if (weight) rc = check_weight("cov_sweep_prefix_rewards", weight, base, prior);
    else if (prior) rc = check_prior("cov_sweep_prefix_rewards", prior, base, true);
    else if (base) {
        cov_set_error("cov_sweep_prefix_rewards: base_dev must be NULL without prior_dev and weight_dev");
        rc = COV_ERR_ARG;
    }
    if (rc) return rc;
    if (!prefix_sums || n_traj <= 0 || per_traj <= 0 || (int64_t)n_traj * per_traj > INT32_MAX) {
        cov_set_error("cov_sweep_prefix_rewards: bad argument (prefix_sums_dev %p, n_traj=%d, poses_per_traj=%d)",
                      (void*)prefix_sums, n_traj, per_traj);
        return COV_ERR_ARG;
    }
    cudaStream_t s = (cudaStream_t)stream;
    cudaMemsetAsync(prefix_sums, 0, (size_t)n_traj * per_traj * sizeof(double), s);
    rc = sweep_rewards_impl(xyz, n, poses, quats, n_traj, per_traj, K, cam, boxes_dev, minmax, prefix_sums, prior, base,
                            opts, ws, ws_bytes, stream, weight, true);
    if (rc) return rc;
    cov_prefix_scan_kernel<<<(unsigned)(((int64_t)n_traj * 32 + 255) / 256), 256, 0, s>>>(prefix_sums, n_traj, per_traj);
    return cov_check_launch("cov_sweep_prefix_rewards");
}

extern "C" size_t cov_sweep_workspace_bytes(int64_t n, int n_traj, int per_traj) {
    if (n < 1) n = 1;
    int W = n_traj * per_traj;
    if (W > 32 * kMaskWords) W = 32 * kMaskWords;
    if (W < 1) W = 1;
    return cov_traj_workspace_bytes(n, W) + align256(2 * (size_t)W * sizeof(float));
}

// The dense path of cov_sweep_fused: [cov_traj_fused workspace for P poses][n rewards (scratch)][2 P normalisers]
static size_t sweep_fused_dense_bytes(int64_t n, int per_traj) {
    return cov_traj_workspace_bytes(n, per_traj) + align256((size_t)n * sizeof(float)) +
           align256(2 * (size_t)per_traj * sizeof(float));
}

// the path a cov_sweep_fused call with these options takes on n points
static bool sweep_fused_prunes(int64_t n, const cov_traj_opts* opts) { return !(opts && opts->dense) && n >= kDenseBelow; }

extern "C" size_t cov_sweep_fused_workspace_bytes(int64_t n, int n_traj, int per_traj, const cov_traj_opts* opts) {
    if (n < 1) n = 1;
    if (n_traj < 1) n_traj = 1;
    per_traj = std::min(std::max(per_traj, 1), 32 * kMaskWords);
    return sweep_fused_prunes(n, opts) ? cov_sweep_workspace_bytes(n, n_traj, per_traj) : sweep_fused_dense_bytes(n, per_traj);
}

static int sweep_fused_impl(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                            int per_traj, const float* K, const cov_camera* cam, const float* boxes_dev,
                            const float* minmax, double* acc, const float* prior, const double* prior_sum,
                            const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream,
                            const float* weight = nullptr, const double* weight_sums = nullptr) {
    if (!xyz || n <= 0 || !poses || !quats || n_traj <= 0 || per_traj <= 0 || !K || !cam || !minmax || !acc || !ws) {
        cov_set_error("cov_sweep_fused: null pointer, empty cloud or no poses (n=%lld, n_traj=%d, poses_per_traj=%d)",
                      (long long)n, n_traj, per_traj);
        return COV_ERR_ARG;
    }
    const bool prune = sweep_fused_prunes(n, opts);
    const int max_p = prune ? cov_traj_max_poses_pruned() : cov_traj_max_poses();
    if (per_traj > max_p) {
        cov_set_error("cov_sweep_fused: %d poses per trajectory exceed what one call takes on this path (max %d)", per_traj,
                      max_p);
        return COV_ERR_UNSUPPORTED;
    }
    if ((int64_t)n_traj * per_traj > INT32_MAX / 8 || n >= ((int64_t)1 << 31) * 256) {
        cov_set_error("cov_sweep_fused: %d x %d poses or %lld points exceed the index range", n_traj, per_traj, (long long)n);
        return COV_ERR_UNSUPPORTED;
    }
    const size_t need = cov_sweep_fused_workspace_bytes(n, n_traj, per_traj, opts);
    if (ws_bytes < need) {
        cov_set_error("cov_sweep_fused: workspace %zu < cov_sweep_fused_workspace_bytes(n, %d, %d, opts) = %zu", ws_bytes,
                      n_traj, per_traj, need);
        return COV_ERR_WORKSPACE;
    }
    if ((((uintptr_t)ws) & 255) || (((uintptr_t)xyz) & 15) || (boxes_dev && (((uintptr_t)boxes_dev) & 15))) {
        cov_set_error("cov_sweep_fused: workspace must be 256-byte aligned, the cloud and boxes 16-byte aligned");
        return COV_ERR_ALIGN;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const size_t block = COV_SWEEP_ACC_BLOCK(per_traj);
    const int TP = n_traj * per_traj;
    if (!prune) {  // the reference path: the dense cov_traj_fused once per trajectory, into that trajectory's block
                   // (the dense kernels count no work: stats_dev is left as it is)
        const size_t tws = cov_traj_workspace_bytes(n, per_traj);
        float* rewards = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + tws);
        float* mm = reinterpret_cast<float*>(reinterpret_cast<char*>(rewards) + align256((size_t)n * sizeof(float)));
        cov_traj_opts dense{};
        dense.dense = 1;
        for (int t = 0; t < n_traj; ++t) {
            const size_t w0 = (size_t)t * per_traj;
            cudaMemcpyAsync(mm, minmax + w0, (size_t)per_traj * sizeof(float), cudaMemcpyDeviceToDevice, s);
            cudaMemcpyAsync(mm + per_traj, minmax + TP + w0, (size_t)per_traj * sizeof(float), cudaMemcpyDeviceToDevice, s);
            const int rc = traj_fused_impl(xyz, n, poses + 3 * w0, quats + 4 * w0, per_traj, K, cam, nullptr, mm, nullptr,
                                           nullptr, rewards, acc + (size_t)t * block, prior, prior_sum, &dense, ws, tws,
                                           stream, weight, weight_sums);
            if (rc) return rc;
        }
        return COV_OK;
    }
    // pruned: the chunking of cov_sweep_rewards (as many trajectories per launch as the box pose mask holds); per chunk
    // pose table, cull + work list, evaluation of the listed boxes
    const int chunk = std::min((32 * kMaskWords) / per_traj, n_traj);
    const CovConst C = cov_make_const(cam);
    const TrajWorkspace t = carve_workspace(ws, n, chunk * per_traj);
    const float4* boxes = boxes_for_call(xyz, n, boxes_dev, t, s);
    constexpr int ppt = 4;  // tiles of 1024 points, eight 128-point items each
    const int64_t ntiles = (n + tile_points(ppt) - 1) / tile_points(ppt);
    float* mm = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + t.bytes);  // the chunk's minima and maxima, contiguous
    {
        const int64_t count = (int64_t)n_traj * (int64_t)block;
        const int grid = (int)std::min<int64_t>((count + 255) / 256, (int64_t)cov_sm_count_cached() * 8);
        if (weight) cov_sweep_acc_init_dev_kernel<<<grid, 256, 0, s>>>(acc, count, (int64_t)block, weight_sums);
        else if (prior) cov_sweep_acc_init_dev_kernel<<<grid, 256, 0, s>>>(acc, count, (int64_t)block, prior_sum);
        else cov_sweep_acc_init_kernel<<<grid, 256, 0, s>>>(acc, count, (int64_t)block, 0.5 * (double)n);
    }
    unsigned long long* stats = opts ? opts->stats_dev : nullptr;
    for (int t0 = 0; t0 < n_traj; t0 += chunk) {
        const int nt = std::min(n_traj - t0, chunk);
        const int w0 = t0 * per_traj, Wn = nt * per_traj;
        cudaMemcpyAsync(mm, minmax + w0, (size_t)Wn * sizeof(float), cudaMemcpyDeviceToDevice, s);
        cudaMemcpyAsync(mm + Wn, minmax + TP + w0, (size_t)Wn * sizeof(float), cudaMemcpyDeviceToDevice, s);
        cov_traj_table_kernel<false><<<(Wn + 63) / 64, 64, 0, s>>>(poses + 3 * (size_t)w0, quats + 4 * (size_t)w0, Wn, K, C,
                                                                   mm, t.table, t.ctrl, (int)(t.ctrl_bytes / sizeof(int)),
                                                                   nullptr, 0.0, nullptr);
        int rc = launch_cull(boxes, n, t, Wn, nullptr, 0.f, nullptr, 0, s);
        if (rc != COV_OK) return rc;
        const auto kern = weight ? (prior ? cov_sweep_fused_tiles_kernel<true, true> : cov_sweep_fused_tiles_kernel<false, true>)
                                 : (prior ? cov_sweep_fused_tiles_kernel<true> : cov_sweep_fused_tiles_kernel<false>);
        kern<<<persistent_grid(kern, 0, ntiles), COV_THREADS, 0, s>>>(
            xyz, n, t.table, Wn, per_traj, C, t.amask, mask_stride_words(Wn), t.worklist, t.ctrl, ntiles,
            acc + (size_t)t0 * block, stats, prior, weight);
    }
    return cov_check_launch("cov_sweep_fused");
}

extern "C" int cov_sweep_fused(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                               int per_traj, const float* K, const cov_camera* cam, const float* boxes_dev,
                               const float* minmax, double* acc, const cov_traj_opts* opts, void* ws, size_t ws_bytes,
                               void* stream) {
    return sweep_fused_impl(xyz, n, poses, quats, n_traj, per_traj, K, cam, boxes_dev, minmax, acc, nullptr, nullptr, opts,
                            ws, ws_bytes, stream);
}

extern "C" int cov_sweep_fused_prior(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                                     int per_traj, const float* K, const cov_camera* cam, const float* boxes_dev,
                                     const float* minmax, double* acc, const float* prior, const double* prior_sum,
                                     const cov_traj_opts* opts, void* ws, size_t ws_bytes, void* stream) {
    const int rc = check_prior("cov_sweep_fused_prior", prior, prior_sum, true);
    if (rc) return rc;
    return sweep_fused_impl(xyz, n, poses, quats, n_traj, per_traj, K, cam, boxes_dev, minmax, acc, prior, prior_sum, opts,
                            ws, ws_bytes, stream);
}

extern "C" int cov_sweep_fused_weighted(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                                        int per_traj, const float* K, const cov_camera* cam, const float* boxes_dev,
                                        const float* minmax, double* acc, const float* prior, const float* weight,
                                        const double* weight_sums, const cov_traj_opts* opts, void* ws, size_t ws_bytes,
                                        void* stream) {
    const int rc = check_weight("cov_sweep_fused_weighted", weight, weight_sums, prior);
    if (rc) return rc;
    return sweep_fused_impl(xyz, n, poses, quats, n_traj, per_traj, K, cam, boxes_dev, minmax, acc, prior, nullptr, opts,
                            ws, ws_bytes, stream, weight, weight_sums);
}

extern "C" int cov_sweep_epilogue(const double* acc, const float* minmax, const float* quats, int n_traj, int per_traj,
                                  int64_t n_total, float* out, void* stream) {
    if (!acc || !minmax || !quats || !out || n_traj <= 0 || per_traj <= 0 || n_total <= 0 ||
        (int64_t)n_traj * per_traj > INT32_MAX / 8) {
        cov_set_error("cov_sweep_epilogue: bad argument (n_traj=%d, poses_per_traj=%d, n_total=%lld)", n_traj, per_traj,
                      (long long)n_total);
        return COV_ERR_ARG;
    }
    const int TP = n_traj * per_traj;
    cov_sweep_epilogue_kernel<<<(TP + 127) / 128, 128, 0, (cudaStream_t)stream>>>(acc, minmax, quats, n_traj, per_traj,
                                                                                 (double)n_total, out);
    return cov_check_launch("cov_sweep_epilogue");
}

extern "C" int cov_traj_epilogue(const double* acc, const float* minmax, const float* quats, int W, int64_t n_total,
                                 int upstream_mode, float* out, void* stream) {
    if (!acc || !minmax || !quats || !out || W <= 0 || n_total <= 0) {
        cov_set_error("cov_traj_epilogue: bad argument");
        return COV_ERR_ARG;
    }
    cov_traj_epilogue_kernel<<<(W + 127) / 128, 128, 0, (cudaStream_t)stream>>>(acc, minmax, quats, W, (double)n_total,
                                                                               upstream_mode, out);
    return cov_check_launch("cov_traj_epilogue");
}

extern "C" int cov_traj_epilogue_dev(const double* acc, const float* minmax, const float* quats, int W,
                                     const double* den_dev, float* out, void* stream) {
    if (!acc || !minmax || !quats || !den_dev || !out || W <= 0) {
        cov_set_error("cov_traj_epilogue_dev: bad argument");
        return COV_ERR_ARG;
    }
    cov_traj_epilogue_dev_kernel<<<(W + 127) / 128, 128, 0, (cudaStream_t)stream>>>(acc, minmax, quats, W, den_dev, out);
    return cov_check_launch("cov_traj_epilogue_dev");
}

extern "C" int cov_sweep_epilogue_dev(const double* acc, const float* minmax, const float* quats, int n_traj, int per_traj,
                                      const double* den_dev, float* out, void* stream) {
    if (!acc || !minmax || !quats || !den_dev || !out || n_traj <= 0 || per_traj <= 0 ||
        (int64_t)n_traj * per_traj > INT32_MAX / 8) {
        cov_set_error("cov_sweep_epilogue_dev: bad argument (n_traj=%d, poses_per_traj=%d)", n_traj, per_traj);
        return COV_ERR_ARG;
    }
    const int TP = n_traj * per_traj;
    cov_sweep_epilogue_dev_kernel<<<(TP + 127) / 128, 128, 0, (cudaStream_t)stream>>>(acc, minmax, quats, n_traj, per_traj,
                                                                                     den_dev, out);
    return cov_check_launch("cov_sweep_epilogue_dev");
}
