// cov_sweep.cu — forward-only evaluation of many candidate trajectories against one cloud
// (BASELINE config 5; semantics of ModelTraj.forward, src/model.py:217-237, per trajectory).
//
// Trajectories are processed in chunks whose pose rows fit in shared memory; inside a chunk the
// block streams its point tiles once and, per trajectory, adds the gated log-odds of its poses in
// pose order, applies the sigmoid and reduces sum_j (r_j - 1/2) with warp shuffles (most points
// have r_j = 1/2 exactly, so the offset keeps the fp32 partial sums short).  Nothing per-point is
// written: the N x n_traj reward matrix (205 GB at config 5) never exists.
#include "cov_common.cuh"
#include "../../include/coverage_b200.h"

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kSweepPpt = 4;
constexpr size_t kSweepSmemBudget = 100 * 1024;  // two blocks per SM

size_t sweep_smem_bytes(int n_traj, int ppt_poses, bool prefix = false) {  // prefix: one fp64 slot per pose
    return (size_t)n_traj * ppt_poses * COV_ROW_F4 * sizeof(float4) + (size_t)n_traj * (prefix ? ppt_poses : 1) * sizeof(double);
}

// HAS_PRIOR: sum_j (sigmoid(prior_j + L_j) - sigmoid(prior_j)) per trajectory (the prior indexed like xyz), and
// *prior_sum = sum_j sigmoid(prior_j) in place of 0.5 * n.
// HAS_W: each point's term times its weight w_j (indexed like xyz), and *prior_sum is the weighted base
// sum_j w_j r0_j (cov_weight_sums).
// PREFIX (cov_sweep_prefix_rewards): one slot per pose.  After each pose at which the warp gated a pair, the fp64
// difference of the warp's successive fp32 reward sums goes to that pose's slot: each of those sums is what this kernel
// computes at the end of the trajectory cut after the pose.  Block 0 adds the base to slot 0 of each trajectory.
template <int PPT, bool HAS_PRIOR, bool HAS_W = false, bool PREFIX = false>
__global__ void __launch_bounds__(COV_THREADS, 2)
cov_sweep_kernel(const float* __restrict__ xyz, int64_t n, const float* __restrict__ poses,
                 const float* __restrict__ quats, int n_traj, int per_traj, const float* __restrict__ K9, CovConst C,
                 const float* __restrict__ mins, const float* __restrict__ maxs, double* __restrict__ sum_out,
                 const float* __restrict__ prior, const double* __restrict__ prior_sum, const float* __restrict__ weight) {
    extern __shared__ float4 smem4[];
    float4* ptab = smem4;
    const int W = n_traj * per_traj;
    double* ssum = reinterpret_cast<double*>(ptab + (size_t)W * COV_ROW_F4);
    const int tid = threadIdx.x, lane = tid & 31;
    for (int w = tid; w < W; w += COV_THREADS) {
        float4* row = ptab + (size_t)w * COV_ROW_F4;
        cov_pose_row(poses + 3 * w, quats + 4 * w, K9, C, row);
        cov_norm_row(row, mins[w], maxs[w], row[3].w);  // conservative gate threshold in v3.w
    }
    const int nslots = PREFIX ? W : n_traj;
    for (int t = tid; t < nslots; t += COV_THREADS) ssum[t] = 0.0;
    __syncthreads();
    constexpr int T = COV_THREADS * PPT;
    const int64_t ntiles = (n + T - 1) / T;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        float px[PPT], py[PPT], pz[PPT], pr[PPT], r0[PPT], wt[PPT];
        bool valid[PPT];
#pragma unroll
        for (int s = 0; s < PPT; ++s) {
            int64_t j = tile * T + s * COV_THREADS + tid;
            valid[s] = j < n;
            j = valid[s] ? j : n - 1;
            px[s] = valid[s] ? __ldg(xyz + j * 3) : 3.0e18f;  // past the end: m = 0 exactly, never gated
            py[s] = valid[s] ? __ldg(xyz + j * 3 + 1) : 3.0e18f;
            pz[s] = valid[s] ? __ldg(xyz + j * 3 + 2) : 3.0e18f;
            if (HAS_PRIOR) {
                pr[s] = __ldg(prior + j);
                r0[s] = cov_sigmoid(pr[s]);
            }
            if (HAS_W) wt[s] = __ldg(weight + j);
        }
        for (int t = 0; t < n_traj; ++t) {
            float L[PPT];
#pragma unroll
            for (int s = 0; s < PPT; ++s) L[s] = 0.f;
            // done(the warp sum of the reward terms for the log-odds sums in L), unless every one of them is 0
            auto reward_sum = [&](auto done) {
                float acc = 0.f;
                bool any_nz = false;
#pragma unroll
                for (int s = 0; s < PPT; ++s) any_nz |= (valid[s] && L[s] != 0.f);
                if (__any_sync(kFull, any_nz)) {
#pragma unroll
                    for (int s = 0; s < PPT; ++s) {
                        if (HAS_W) {
                            if (valid[s] && L[s] != 0.f) {
                                const float r = HAS_PRIOR ? cov_sigmoid(cov_fuse_prior(pr[s], L[s])) : 1.f / (1.f + expf(-L[s]));
                                acc += wt[s] * (r - (HAS_PRIOR ? r0[s] : 0.5f));
                            }
                        } else if (HAS_PRIOR) {
                            if (valid[s] && L[s] != 0.f) acc += cov_sigmoid(cov_fuse_prior(pr[s], L[s])) - r0[s];
                        } else if (valid[s] && L[s] != 0.f) {
                            acc += 1.f / (1.f + expf(-L[s])) - 0.5f;
                        }
                    }
                    done(cov_warp_sum(acc));
                }
            };
            float vprev = 0.f;  // PREFIX: the warp sum after the last pose at which the warp gated a pair
            for (int i = 0; i < per_traj; ++i) {
                const float4* row = ptab + (size_t)(t * per_traj + i) * COV_ROW_F4;
                const float4 v0 = row[0], v1 = row[1], v2 = row[2], v3 = row[3];
                float m[PPT];
#pragma unroll
                for (int s = 0; s < PPT; ++s) m[s] = cov_vis<false>(px[s], py[s], pz[s], v0, v1, v2, v3, C, nullptr);
                float mmax = m[0];
#pragma unroll
                for (int s = 1; s < PPT; ++s) mmax = fmaxf(mmax, m[s]);
                if (__any_sync(kFull, mmax >= v3.w)) {
                    const float4 v4 = row[4];
                    bool gated = false;
#pragma unroll
                    for (int s = 0; s < PPT; ++s) {
                        const float d = __fsub_rn(m[s], v4.w);
                        if (d >= v4.x) {  // exactly p >= 0.5
                            L[s] += cov_logodds(d, v4, C);
                            gated = true;
                        }
                    }
                    if (PREFIX && __any_sync(kFull, gated)) {
                        float v = 0.f;
                        reward_sum([&](float a) { v = a; });
                        if (lane == 0 && v != vprev) atomicAdd(ssum + t * per_traj + i, (double)v - (double)vprev);
                        vprev = v;
                    }
                }
            }
            if (!PREFIX)
                reward_sum([&](float acc) {
                    if (lane == 0 && acc != 0.f) atomicAdd(ssum + t, (double)acc);
                });
        }
    }
    __syncthreads();
    for (int t = tid; t < nslots; t += COV_THREADS) {
        double v = ssum[t];
        if (blockIdx.x == 0 && (!PREFIX || t % per_traj == 0)) v += (HAS_PRIOR || HAS_W) ? *prior_sum : 0.5 * (double)n;
        if (v != 0.0) atomicAdd(sum_out + t, v);
    }
}

}  // namespace

// Dense sweep (cov_traj_opts.dense); the pruned pipeline and the C entry points are in cov_traj.cu.  prefix: the per-pose
// slots of cov_sweep_prefix_rewards (n_traj * per_traj doubles) in place of the per-trajectory sums.
int cov_sweep_rewards_dense(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                            int per_traj, const float* K, const cov_camera* cam, const float* minmax,
                            double* sum_rewards, const float* prior, const double* prior_sum, const float* weight,
                            void* stream, bool prefix) {
    const char* who = prefix ? "cov_sweep_prefix_rewards" : "cov_sweep_rewards";
    if (!xyz || n <= 0 || !poses || !quats || n_traj <= 0 || per_traj <= 0 || !K || !cam || !minmax || !sum_rewards) {
        cov_set_error("%s: bad argument", who);
        return COV_ERR_ARG;
    }
    if (sweep_smem_bytes(1, per_traj, prefix) > 227 * 1024 - 256) {
        cov_set_error("%s: %d poses per trajectory do not fit in shared memory", who, per_traj);
        return COV_ERR_UNSUPPORTED;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    int chunk = 1;
    while (chunk < n_traj && sweep_smem_bytes(chunk + 1, per_traj, prefix) <= kSweepSmemBudget) ++chunk;
    const int W = n_traj * per_traj;
    constexpr int T = COV_THREADS * kSweepPpt;
    const int64_t ntiles = (n + T - 1) / T;
    const size_t smem_max = sweep_smem_bytes(chunk, per_traj, prefix);
    const auto kern =
        prefix ? (weight ? (prior ? cov_sweep_kernel<kSweepPpt, true, true, true> : cov_sweep_kernel<kSweepPpt, false, true, true>)
                         : (prior ? cov_sweep_kernel<kSweepPpt, true, false, true> : cov_sweep_kernel<kSweepPpt, false, false, true>))
               : (weight ? (prior ? cov_sweep_kernel<kSweepPpt, true, true> : cov_sweep_kernel<kSweepPpt, false, true>)
                         : (prior ? cov_sweep_kernel<kSweepPpt, true> : cov_sweep_kernel<kSweepPpt, false>));
    // always the same value: two host threads with different trajectory counts cannot race between set and launch
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024 - 256);
    int per_sm = 1;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, COV_THREADS, smem_max) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    int64_t grid = (int64_t)per_sm * cov_sm_count_cached();
    if (grid > ntiles) grid = ntiles;
    if (grid > COV_MAX_GRID) grid = COV_MAX_GRID;
    for (int t0 = 0; t0 < n_traj; t0 += chunk) {
        const int nt = (n_traj - t0 < chunk) ? n_traj - t0 : chunk;
        const int w0 = t0 * per_traj;
        kern<<<(unsigned)grid, COV_THREADS, sweep_smem_bytes(nt, per_traj, prefix), s>>>(
            xyz, n, poses + 3 * (size_t)w0, quats + 4 * (size_t)w0, nt, per_traj, K, C, minmax + w0, minmax + W + w0,
            sum_rewards + (prefix ? w0 : t0), prior, prior_sum, weight);
    }
    return cov_check_launch(who);
}
