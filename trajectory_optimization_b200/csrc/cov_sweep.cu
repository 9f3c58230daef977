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

size_t sweep_smem_bytes(int n_traj, int ppt_poses) {
    return (size_t)n_traj * ppt_poses * COV_ROW_F4 * sizeof(float4) + (size_t)n_traj * sizeof(double);
}

// HAS_PRIOR: sum_j (sigmoid(prior_j + L_j) - sigmoid(prior_j)) per trajectory (the prior indexed like xyz), and
// *prior_sum = sum_j sigmoid(prior_j) in place of 0.5 * n.
// HAS_W: each point's term times its weight w_j (indexed like xyz), and *prior_sum is the weighted base
// sum_j w_j r0_j (cov_weight_sums).
template <int PPT, bool HAS_PRIOR, bool HAS_W = false>
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
    for (int t = tid; t < n_traj; t += COV_THREADS) ssum[t] = 0.0;
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
#pragma unroll
                    for (int s = 0; s < PPT; ++s) {
                        const float d = __fsub_rn(m[s], v4.w);
                        if (d >= v4.x) L[s] += cov_logodds(d, v4, C);  // exactly p >= 0.5
                    }
                }
            }
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
                acc = cov_warp_sum(acc);
                if (lane == 0 && acc != 0.f) atomicAdd(ssum + t, (double)acc);
            }
        }
    }
    __syncthreads();
    for (int t = tid; t < n_traj; t += COV_THREADS) {
        double v = ssum[t];
        if (blockIdx.x == 0) v += (HAS_PRIOR || HAS_W) ? *prior_sum : 0.5 * (double)n;
        if (v != 0.0) atomicAdd(sum_out + t, v);
    }
}

}  // namespace

// Dense sweep (cov_traj_opts.dense); the pruned pipeline and the C entry point are in cov_traj.cu.
int cov_sweep_rewards_dense(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj,
                            int per_traj, const float* K, const cov_camera* cam, const float* minmax,
                            double* sum_rewards, const float* prior, const double* prior_sum, const float* weight,
                            void* stream) {
    if (!xyz || n <= 0 || !poses || !quats || n_traj <= 0 || per_traj <= 0 || !K || !cam || !minmax || !sum_rewards) {
        cov_set_error("cov_sweep_rewards: bad argument");
        return COV_ERR_ARG;
    }
    if (sweep_smem_bytes(1, per_traj) > 227 * 1024 - 256) {
        cov_set_error("cov_sweep_rewards: %d poses per trajectory do not fit in shared memory", per_traj);
        return COV_ERR_UNSUPPORTED;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const CovConst C = cov_make_const(cam);
    int chunk = 1;
    while (chunk < n_traj && sweep_smem_bytes(chunk + 1, per_traj) <= kSweepSmemBudget) ++chunk;
    const int W = n_traj * per_traj;
    constexpr int T = COV_THREADS * kSweepPpt;
    const int64_t ntiles = (n + T - 1) / T;
    const size_t smem_max = sweep_smem_bytes(chunk, per_traj);
    const auto kern = weight ? (prior ? cov_sweep_kernel<kSweepPpt, true, true> : cov_sweep_kernel<kSweepPpt, false, true>)
                             : (prior ? cov_sweep_kernel<kSweepPpt, true> : cov_sweep_kernel<kSweepPpt, false>);
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
        kern<<<(unsigned)grid, COV_THREADS, sweep_smem_bytes(nt, per_traj), s>>>(
            xyz, n, poses + 3 * (size_t)w0, quats + 4 * (size_t)w0, nt, per_traj, K, C, minmax + w0, minmax + W + w0,
            sum_rewards + t0, prior, prior_sum, weight);
    }
    return cov_check_launch("cov_sweep_rewards");
}
