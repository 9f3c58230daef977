/*
 * coverage_b200.h — C ABI of libcovb200.so: the B200 (sm_100a) implementation of the
 * differentiable visibility/coverage hot path of ctu-vras/trajectory_optimization.
 *
 * Conventions (all entry points):
 *   - plain C: pointers, sizes and scalars only; no C++/torch types cross the boundary;
 *   - `const float* x_dev` / `*_dev` arguments are DEVICE pointers, everything else is by value;
 *   - the caller owns every buffer (outputs, accumulators, workspace); the library never
 *     allocates or frees device memory, never synchronises the device and launches only on
 *     the stream passed as `stream` (a cudaStream_t cast to void*; NULL = legacy default);
 *   - return value 0 = success, negative = COV_ERR_*; cov_last_error() returns a
 *     thread-local message for the most recent failure on the calling thread;
 *   - re-entrant: no process-wide switches or counters; the only mutable state in the library is the thread-local
 *     error string and a mutex-protected cache of per-kernel occupancy figures (pure function of kernel, device, size);
 *   - quaternions are (w, x, y, z), unnormalised (the kernels apply F.normalize, eps 1e-12);
 *     point clouds are row-major (N,3) fp32, 16-byte aligned (COV_ERR_ALIGN otherwise).
 *
 * "ref:" lines cite the reference interface each entry point replaces
 * (paths relative to the reference repository root).
 */
#ifndef COVERAGE_B200_H
#define COVERAGE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define COV_OK 0
#define COV_ERR_ARG (-1)         /* null pointer / negative size / bad enum            */
#define COV_ERR_UNSUPPORTED (-2) /* pose count exceeds what fits in shared memory      */
#define COV_ERR_WORKSPACE (-3)   /* workspace too small                                */
#define COV_ERR_CUDA (-4)        /* a CUDA runtime call or launch failed               */
#define COV_ERR_ALIGN (-5)       /* a device pointer is not 16-byte aligned            */

/* Layout of the per-pose accumulator rows produced by cov_traj_fused (doubles). */
#define COV_ACC_STRIDE 22 /* [0..2] F, [3..5] T, [6] sum e, [7] sum e*p, [8..13] argmax F,T, [14] #argmax, \
                             [15..20] argmin F,T, [21] #argmin                                              */
#define COV_POSE_ACC 8    /* cov_pose_fused: [0] sum m, [1..3] F, [4..6] T, [7] unused                      */

/* Camera / mask constants shared by every coverage entry point.
 * ref: src/model.py:13-47 (get_dist_mask, get_fov_mask), src/model.py:93-94 (eps, pc_clip_limits). */
typedef struct cov_camera {
    float img_width;  /* pairs with u = h0/(h2+eps)  (1232 in src/tools.py:321) */
    float img_height; /* pairs with v = h1/(h2+eps)  (1616)                     */
    float min_dist;   /* Gaussian distance mask: mu = (min+max)/2, sigma = (max-min)/2 */
    float max_dist;
    float eps;        /* 1e-6 in the reference */
} cov_camera;

int cov_version(void);
const char* cov_last_error(void);
/* Number of SMs of the current device and bytes of opt-in shared memory per block (0 on failure). */
int cov_device_sm_count(void);

/* ------------------------------------------------------------------------------------------
 * ModelPose: obs_j = dist_mask * fov_mask [* weight_j];  sum = sum_j obs_j; d(sum)/d(pose).
 * ref: src/model.py:98-127 (ModelPose.forward/criterion), :50-57 (to_camera_frame).
 * One pass over the cloud: 12 B/point read (+4 B weight) + 4 B/point written.
 *   xyz_dev      (n,3) fp32              weight_dev  (n) fp32 or NULL (hpr mask / upstream grad)
 *   trans_dev    3 fp32                  quat_dev    4 fp32 (w,x,y,z)       K_dev 9 fp32 row-major
 *   obs_dev      (n) fp32 out or NULL    acc_dev     COV_POSE_ACC doubles out (this shard's sums)
 * ------------------------------------------------------------------------------------------ */
size_t cov_pose_workspace_bytes(int64_t n);
int cov_pose_fused(const float* xyz_dev, int64_t n, const float* weight_dev, const float* trans_dev,
                   const float* quat_dev, const float* K_dev, const cov_camera* cam, float* obs_dev,
                   double* acc_dev, void* workspace_dev, size_t workspace_bytes, void* stream);
/* O(1) epilogue on the (all-reduced) accumulators:
 * out_dev[0] = sum, out_dev[1..3] = d sum/d trans, out_dev[4..7] = d sum/d quat (raw, unnormalised). */
int cov_pose_epilogue(const double* acc_dev, const float* trans_dev, const float* quat_dev, float* out_dev,
                      void* stream);

/* ------------------------------------------------------------------------------------------
 * ModelTraj visibility term over W evaluated poses (the caller applies the wps_step selection).
 * ref: src/model.py:200-242 (ModelTraj.forward), :244-246 (criterion 'vis').
 * Pass A  cov_traj_minmax : per-pose min_j m_jw / max_j m_jw              (12 B/point)
 *         -> all-reduce MIN / MAX across ranks when the cloud is sharded
 * Pass B  cov_traj_fused  : rewards_j = sigmoid(sum_w logit(clip(p_jw))) and the shard-additive
 *         gradient accumulators (COV_ACC_STRIDE doubles per pose + 1 trailing sum of rewards)
 *         (12 B/point read + 4 B/point written)
 *         -> all-reduce SUM across ranks
 * Epilogue cov_traj_epilogue: mean reward and d(mean)/d(poses, quats).
 *   poses_dev (W,3) fp32, quats_dev (W,4) fp32, minmax_dev 2*W fp32: [0,W) minima, [W,2W) maxima
 *   upstream_dev: NULL (gradient of mean(rewards)) or (n) fp32 d(loss)/d(rewards_j)
 *   reward_index_dev: NULL, or (n) int32: point j of xyz_dev is point reward_index_dev[j] of the caller's cloud
 *   (the permutation cov_spatial_sort returns); rewards_dev and upstream_dev are then indexed in the caller's order.
 * ------------------------------------------------------------------------------------------ */
int cov_traj_max_poses(void);        /* poses one call takes on ANY path (the dense kernels' shared-memory pose table) */
int cov_traj_max_poses_pruned(void); /* ... when the call takes the pruned path (cov_traj_prefill_applies): the tile masks' width */
size_t cov_traj_workspace_bytes(int64_t n, int n_poses);

/* Per-call options of cov_traj_minmax / cov_traj_fused / cov_sweep_rewards; NULL = all zero = the defaults.
 * Exact pruning (default): a (point, pose) pair whose distance Gaussian alone bounds m below what could matter (a
 * sampled lower bound of the maximum in pass A once a zero minimum is known; the gate threshold in pass B) is never
 * evaluated.  Per call: pose table -> cull (boxes of 128 consecutive points against every pose) + ascending work list of
 * the tiles with a non-empty pose mask -> persistent evaluation kernel over the list (tile, boxes and mask arrive by
 * TMA; each warp re-tests against the box of its own points, then per point).  Normalisers and rewards are
 * bit-identical to the dense evaluation on ANY point order; the saving grows with the spatial coherence of
 * consecutive points (cov_spatial_sort).  Clouds below 65536 points always take the dense kernels. */
typedef struct cov_traj_opts {
    int dense;                     /* != 0: evaluate every (point, pose) pair (what an unordered cloud should ask for) */
    int rewards_prefilled;         /* cov_traj_fused: != 0: rewards_dev already holds 1/2 everywhere (skip the pre-fill);
                                      ignored by the dense path, which writes every reward itself */
    float* prefill_dev;            /* cov_traj_minmax: NULL, or the (n) rewards buffer of the cov_traj_fused call that
                                      follows: the pruned pass A fills it with 1/2 under its idle memory bandwidth
                                      (then pass rewards_prefilled = 1 to cov_traj_fused).  Honoured only when the call
                                      takes the pruned path (dense == 0 and n >= 65536): cov_traj_prefill_applies() */
    unsigned long long* stats_dev; /* NULL, or 8 device counters the evaluation kernels ADD to, in (warp, pose) pairs:
                                      [0] pass B all pairs, [1] evaluated (forward), [2],[3] same for pass A, [4] pass B
                                      pairs differentiated (evaluated again + gradient), [5] pass A pairs that ran the
                                      per-point pre-filter, [6]/[7] pass B/A pairs the cull listed
                                      (benchmark reporting; NULL in production) */
} cov_traj_opts;

/* != 0 when cov_traj_minmax with these options and this n honours prefill_dev (i.e. takes the pruned path). */
int cov_traj_prefill_applies(int64_t n, const cov_traj_opts* opts);

/* boxes_dev: NULL, or the bounding boxes cov_tile_boxes made for this cloud (built once per cloud; with NULL the
 * pruned kernels rebuild them into the workspace on every call).  workspace_dev: cov_traj_workspace_bytes(n, n_poses)
 * bytes, 256-byte aligned, shared by both calls (callers keep one per cloud: nothing in it outlives a call). */
int cov_traj_minmax(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_poses,
                    const float* K_dev, const cov_camera* cam, const float* boxes_dev, float* minmax_dev,
                    const cov_traj_opts* opts, void* workspace_dev, size_t workspace_bytes, void* stream);
int cov_traj_fused(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_poses,
                   const float* K_dev, const cov_camera* cam, const float* boxes_dev, const float* minmax_dev,
                   const float* upstream_dev, const int32_t* reward_index_dev, float* rewards_dev, double* acc_dev,
                   const cov_traj_opts* opts, void* workspace_dev, size_t workspace_bytes, void* stream);
/* out_dev: [0] mean reward, then (W,3) d/d poses, then (W,4) d/d quats  (1 + 7*W floats).
 * With upstream_mode != 0 the gradients are those of sum_j upstream_j * rewards_j (no 1/N). */
int cov_traj_epilogue(const double* acc_dev, const float* minmax_dev, const float* quats_dev, int n_poses,
                      int64_t n_total, int upstream_mode, float* out_dev, void* stream);

/* The O(W) regularisers of ModelTraj.criterion and their gradients in one launch (SURVEY.md 8f1).
 * ref: src/model.py:244-260 (criterion: l2, smooth, length), :135-139 (length_calc), :142-155 (mean_angle_calc).
 *   poses_dev, poses0_dev (W,3) fp32, W >= 3.  out_dev: 3 + 9*W floats: [0] l2 = |poses[0]-poses0[0]|,
 *   [1] smooth = w_s/(mean interior angle + eps), [2] length = w_l*|len(poses) - len(poses0)|, then d l2/d poses,
 *   d smooth/d poses, d length/d poses, (W,3) each.  fp64 inside; torch's conventions at the kinks (gradient 0). */
int cov_traj_regularizers(const float* poses_dev, const float* poses0_dev, int n_poses, float smoothness_weight,
                          float traj_length_weight, float eps, float* out_dev, void* stream);

/* Forward-only candidate sweep: n_traj trajectories x poses_per_traj poses each, sharing one cloud.
 * ref: no reference implementation (BASELINE config 5); semantics = ModelTraj.forward per trajectory
 * with every pose evaluated.  sum_rewards_dev[t] += sum_j rewards_j(t) over this shard (doubles,
 * zero it first); minmax_dev is (2, n_traj*poses_per_traj) produced by cov_traj_minmax.
 * boxes_dev as for cov_traj_fused; workspace_dev: cov_sweep_workspace_bytes(n, n_traj, poses_per_traj) bytes,
 * 256-byte aligned (the pruned pipeline runs the trajectories in chunks of pose-table size). */
size_t cov_sweep_workspace_bytes(int64_t n, int n_traj, int poses_per_traj);
int cov_sweep_rewards(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_traj,
                      int poses_per_traj, const float* K_dev, const cov_camera* cam, const float* boxes_dev,
                      const float* minmax_dev, double* sum_rewards_dev, const cov_traj_opts* opts, void* workspace_dev,
                      size_t workspace_bytes, void* stream);

/* Differentiable candidate sweep: for each of n_traj trajectories x poses_per_traj (= P) poses sharing one cloud, the
 * accumulators cov_traj_fused computes for that trajectory alone (W = P, no upstream), in one pass over the cloud per
 * chunk of cov_traj_max_poses_pruned() poses.
 * ref: no reference implementation; semantics = ModelTraj.forward + backward of mean(rewards) per trajectory with every
 * pose evaluated.  No per-point rewards are written.
 *   acc_dev: n_traj blocks of COV_SWEEP_ACC_BLOCK(P) doubles; block t = P rows of COV_ACC_STRIDE doubles then sum_j r_j(t),
 *   exactly what cov_traj_fused writes for trajectory t.  The call initialises every block itself.  Shard-additive: with
 *   a sharded cloud, SUM the blocks over the ranks, then run cov_sweep_epilogue.
 *   minmax_dev (2, n_traj*P): the global normalisers (cov_traj_minmax per chunk of poses, MIN/MAX over the ranks).
 *   opts: dense (or n < 65536) runs the dense cov_traj_fused once per trajectory (P <= cov_traj_max_poses()); the pruned
 *   path takes P <= cov_traj_max_poses_pruned().  stats_dev: on the pruned path the evaluation kernel adds the pass B
 *   counters [0], [1], [4], [6]; the dense path adds nothing (its kernels count no work).
 *   workspace_dev: cov_sweep_fused_workspace_bytes(n, n_traj, P, opts) bytes for the same n, P and opts, 256-byte aligned
 *   (the dense path's size includes n floats of reward scratch; the pruned path's does not). */
#define COV_SWEEP_ACC_BLOCK(P) ((size_t)(P) * COV_ACC_STRIDE + 1)
size_t cov_sweep_fused_workspace_bytes(int64_t n, int n_traj, int poses_per_traj, const cov_traj_opts* opts);
int cov_sweep_fused(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_traj,
                    int poses_per_traj, const float* K_dev, const cov_camera* cam, const float* boxes_dev,
                    const float* minmax_dev, double* acc_dev, const cov_traj_opts* opts, void* workspace_dev,
                    size_t workspace_bytes, void* stream);
/* out_dev (fp32): [n_traj means | n_traj*P*3 d mean_t/d poses | n_traj*P*4 d mean_t/d quats]; trajectory t's part is
 * what cov_traj_epilogue (upstream_mode 0) gives for block t with minmax [min_t | max_t] and quats_t, bit for bit. */
int cov_sweep_epilogue(const double* acc_dev, const float* minmax_dev, const float* quats_dev, int n_traj,
                       int poses_per_traj, int64_t n_total, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Prior log-odds (map memory): score coverage on top of what earlier, executed paths observed.
 * ref: no reference implementation; the fusion is OctoMap's: a point's fused log-odds x_j = prior_j + L_j, with
 * L_j = sum_w lo_jw formed in fp32 in pose order exactly as without a prior (one fp32 add), and r_j = 1/(1 + expf(-x_j)).
 * The min/max normalisers, the gate, the pruning and the per-pose terms do not change; a point no gated pair reaches
 * gets sigmoid(prior_j), and G_j = r_j (1 - r_j) uses the shifted r_j.  A prior of all zeros gives the rewards of the
 * entry points without a prior bit for bit (sigmoid(0) = 1/2 exactly).  Non-finite priors propagate; nothing checks them.
 *   prior_dev      (n) fp32, 16-byte aligned, one per point, shared by every pose and trajectory of the call.
 *                  cov_traj_*: indexed like rewards_dev and upstream_dev, i.e. in the CALLER'S order when
 *                  reward_index_dev is given.  cov_sweep_*: indexed like xyz_dev (the cloud's order).
 *   prior_sum_dev  1 double: sum_j sigmoid(prior_j) over this shard (cov_prior_reward_sum, once per prior state); it is
 *                  the reward sum of the points no listed pose reaches, read on the device (no host synchronisation).
 * With a sharded cloud each rank passes its slice of the prior and its own sum; the SUM all-reduce of the accumulators
 * makes the sums global as before.
 * cov_traj_minmax_prior: cov_traj_minmax whose pre-fill (opts->prefill_dev) writes sigmoid(prior_i), the value the
 *   pruned pass B leaves in place for the points it does not store (pass rewards_prefilled = 1 to cov_traj_fused_prior).
 * cov_traj_logodds: pass B's forward without the backward.  logodds_dev (n) fp32, indexed like rewards_dev, must hold
 *   the prior (or zeros) on entry; the call adds L_j where L_j != 0, so that it holds x_j: sigmoid of it is the reward
 *   cov_traj_fused_prior computes, bit for bit.  Folding an executed path into the map is prior := logodds.
 *   Takes cov_traj_workspace_bytes(n, n_poses) of workspace and the same options and paths as cov_traj_fused.
 * ------------------------------------------------------------------------------------------ */
int cov_prior_reward_sum(const float* prior_dev, int64_t n, double* prior_sum_dev, void* stream);
int cov_traj_minmax_prior(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_poses,
                          const float* K_dev, const cov_camera* cam, const float* boxes_dev, float* minmax_dev,
                          const float* prior_dev, const cov_traj_opts* opts, void* workspace_dev, size_t workspace_bytes,
                          void* stream);
int cov_traj_fused_prior(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_poses,
                         const float* K_dev, const cov_camera* cam, const float* boxes_dev, const float* minmax_dev,
                         const float* upstream_dev, const int32_t* reward_index_dev, float* rewards_dev, double* acc_dev,
                         const float* prior_dev, const double* prior_sum_dev, const cov_traj_opts* opts,
                         void* workspace_dev, size_t workspace_bytes, void* stream);
int cov_traj_logodds(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_poses,
                     const float* K_dev, const cov_camera* cam, const float* boxes_dev, const float* minmax_dev,
                     const int32_t* reward_index_dev, float* logodds_dev, const cov_traj_opts* opts, void* workspace_dev,
                     size_t workspace_bytes, void* stream);
int cov_sweep_rewards_prior(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_traj,
                            int poses_per_traj, const float* K_dev, const cov_camera* cam, const float* boxes_dev,
                            const float* minmax_dev, double* sum_rewards_dev, const float* prior_dev,
                            const double* prior_sum_dev, const cov_traj_opts* opts, void* workspace_dev,
                            size_t workspace_bytes, void* stream);
int cov_sweep_fused_prior(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_traj,
                          int poses_per_traj, const float* K_dev, const cov_camera* cam, const float* boxes_dev,
                          const float* minmax_dev, double* acc_dev, const float* prior_dev, const double* prior_sum_dev,
                          const cov_traj_opts* opts, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Point weights: what is worth seeing.  Weighted mean of the trajectory objective, mean_w = sum_j w_j r_j / sum_j w_j,
 * and its pose gradients (pass B's backward with G_j = w_j r_j (1 - r_j)), in the same pass as the unweighted call.
 * ref: no reference implementation.  The weight changes neither r_j nor the normalisers, the gate or the pruning: the
 * rewards of cov_traj_fused_weighted are bit-identical to those of the call without a weight.  It composes with the prior
 * (r_j = sigmoid(prior_j + L_j) as above).  A weight of all ones gives the unweighted sums up to the order of the fp64
 * additions.  Nothing checks the values: they must be finite and >= 0 with sum_j w_j > 0 (NaN/inf propagate).
 *   weight_dev       (n) fp32, 16-byte aligned, one per point, shared by every pose and trajectory of the call; indexed
 *                    like prior_dev (cov_traj_*: like rewards_dev; cov_sweep_*: like xyz_dev).
 *   prior_dev        NULL or the prior log-odds, as for the _prior entry points.  The weighted base below takes the
 *                    place of prior_sum_dev.
 *   weight_sums_dev  2 doubles from cov_weight_sums (once per weight and prior state), read on the device:
 *                    [0] sum_j w_j r0_j with r0_j = sigmoid(prior_j), or 1/2 without a prior: the weighted reward sum of
 *                        the points no listed pose reaches, where the accumulated sum starts;
 *                    [1] sum_j w_j: the denominator of the weighted means (cov_*_epilogue_dev).
 * Accumulators: the layouts of the unweighted calls, with sum_j w_j r_j in place of sum_j r_j.  Shard-additive: with a
 * sharded cloud each rank passes its slices and its own sums; SUM the accumulators as before, and SUM [1] over the ranks
 * (only [1]) before the epilogue.
 * cov_traj_fused_weighted: cov_traj_fused without upstream (the gradient of the weighted mean).  Pre-fill, options,
 *   workspace and paths as for cov_traj_fused (cov_traj_fused_prior with a prior).  The gradient through rewards_dev is
 *   the unweighted call's with upstream_dev: the rewards do not depend on the weight.
 * cov_sweep_rewards_weighted, cov_sweep_fused_weighted: the sweeps with sum_j w_j r_j(t) per trajectory; every path
 *   (pruned, dense, the small-cloud path of cov_sweep_fused) weighs.  Workspace as for the unweighted calls.
 * cov_traj_epilogue_dev, cov_sweep_epilogue_dev: cov_traj_epilogue (upstream_mode 0) and cov_sweep_epilogue with the
 *   denominator *den_dev (fp64, on the device; weight_sums_dev + 1) in place of n_total; with *den_dev == n_total the
 *   outputs are bit-identical to theirs.
 * ------------------------------------------------------------------------------------------ */
int cov_weight_sums(const float* weight_dev, const float* prior_dev, int64_t n, double* weight_sums_dev, void* stream);
int cov_traj_fused_weighted(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_poses,
                            const float* K_dev, const cov_camera* cam, const float* boxes_dev, const float* minmax_dev,
                            const int32_t* reward_index_dev, float* rewards_dev, double* acc_dev, const float* prior_dev,
                            const float* weight_dev, const double* weight_sums_dev, const cov_traj_opts* opts,
                            void* workspace_dev, size_t workspace_bytes, void* stream);
int cov_sweep_rewards_weighted(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev,
                               int n_traj, int poses_per_traj, const float* K_dev, const cov_camera* cam,
                               const float* boxes_dev, const float* minmax_dev, double* sum_rewards_dev,
                               const float* prior_dev, const float* weight_dev, const double* weight_sums_dev,
                               const cov_traj_opts* opts, void* workspace_dev, size_t workspace_bytes, void* stream);
int cov_sweep_fused_weighted(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_traj,
                             int poses_per_traj, const float* K_dev, const cov_camera* cam, const float* boxes_dev,
                             const float* minmax_dev, double* acc_dev, const float* prior_dev, const float* weight_dev,
                             const double* weight_sums_dev, const cov_traj_opts* opts, void* workspace_dev,
                             size_t workspace_bytes, void* stream);
int cov_traj_epilogue_dev(const double* acc_dev, const float* minmax_dev, const float* quats_dev, int n_poses,
                          const double* den_dev, float* out_dev, void* stream);
int cov_sweep_epilogue_dev(const double* acc_dev, const float* minmax_dev, const float* quats_dev, int n_traj,
                           int poses_per_traj, const double* den_dev, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Long trajectories: the trajectory objective, its gradients and the log-odds fold for any number of poses W (one
 * cov_traj_fused call takes at most cov_traj_max_poses_pruned()).  The poses run in chunks of pose_chunk; the fused
 * log-odds L_j = sum_w lo_jw (fp32, ascending pose order) is carried between chunks in fp32, so the outputs are those
 * of one cov_traj_fused / cov_traj_logodds call over all W poses, had it existed: normalisers, every reward and
 * sigmoid(logodds) bit for bit, the accumulators up to the order of the fp64 additions; the variants, index conventions
 * and tie accumulators are pass B's.  The pruned kernels run on every cloud size (they are exact on any point order).
 * ref: src/model.py:217-237 over all waypoints, with no pose limit.
 *   pose_chunk   0 = cov_traj_max_poses_pruned(); else 1 .. that (COV_ERR_ARG otherwise).  Results do not depend on it;
 *                smaller chunks need more workspace (one box mask row per chunk) and more launches.
 *   acc_dev      22 * W + 1 doubles, the layout of cov_traj_fused: the SUM all-reduce and the epilogues are unchanged.
 *   prior_dev, weight_dev, base_dev  NULL pointers select the variant: no prior and weight (base_dev NULL), a prior alone
 *                (base_dev = cov_prior_reward_sum), a weight with or without a prior (base_dev = cov_weight_sums; then
 *                upstream_dev must be NULL).  Indexed like rewards_dev, as for the _prior / _weighted entry points.
 *   opts         rewards_prefilled and stats_dev as for cov_traj_fused (stats: counters [0], [1], [4], [6], summed over
 *                the chunks to what one call would count).  dense != 0: one dense cov_traj_fused (cov_traj_logodds)
 *                call when W <= cov_traj_max_poses(), COV_ERR_UNSUPPORTED above that (there is no dense long path).
 *   workspace    cov_traj_long_workspace_bytes(n, W, pose_chunk) bytes, 256-byte aligned; it never grows with pose_chunk
 *                and also serves the per-chunk pass A below.  It grows with W: one mask row per listed 128-point box per
 *                chunk (up to 2 n bytes per chunk of 2048 poses) next to 4 n bytes of carried log-odds.
 * Pass A runs per chunk through cov_traj_minmax (the normalisers are per pose) into the W-wide layout.  For C callers:
 *   for each chunk [w0, w1) of at most cov_traj_max_poses_pruned() poses (cov_traj_max_poses() when n < 65536 or dense):
 *     cov_traj_minmax(.., poses + 3 w0, quats + 4 w0, w1 - w0, .., mm, opts, ws, ..)   (opts.prefill_dev = rewards on
 *     the first chunk only; cov_traj_minmax_prior with a prior), then copy mm[0, w1-w0) to minmax[w0, w1) and
 *     mm[w1-w0, 2(w1-w0)) to minmax[W + w0, W + w1);
 *   MIN/MAX all-reduce of minmax over the ranks (sharded clouds);
 *   cov_traj_fused_long(.., minmax, .., acc, .., opts.rewards_prefilled = cov_traj_prefill_applies(n, opts), ..);
 *   SUM all-reduce of acc; cov_traj_epilogue (cov_traj_epilogue_dev with a weight).
 * cov_traj_logodds_long: cov_traj_logodds over all W poses (logodds_dev holds the prior or zeros on entry).
 * ------------------------------------------------------------------------------------------ */
size_t cov_traj_long_workspace_bytes(int64_t n, int n_poses, int pose_chunk);
int cov_traj_fused_long(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_poses,
                        const float* K_dev, const cov_camera* cam, const float* boxes_dev, const float* minmax_dev,
                        const float* upstream_dev, const int32_t* reward_index_dev, float* rewards_dev, double* acc_dev,
                        const float* prior_dev, const double* base_dev, const float* weight_dev, int pose_chunk,
                        const cov_traj_opts* opts, void* workspace_dev, size_t workspace_bytes, void* stream);
int cov_traj_logodds_long(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev, int n_poses,
                          const float* K_dev, const cov_camera* cam, const float* boxes_dev, const float* minmax_dev,
                          const int32_t* reward_index_dev, float* logodds_dev, int pose_chunk, const cov_traj_opts* opts,
                          void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Prefix sweep: the reward sum of every prefix of every candidate trajectory in one pass over the cloud per chunk of
 * cov_traj_max_poses_pruned() poses (the chunking of cov_sweep_rewards).
 * ref: no reference implementation; entry [t*P + i] is what cov_sweep_rewards (or its _prior / _weighted form, with the
 * same prior and weight) returns for trajectory t cut after its pose i, i.e. poses_dev[t*P .. t*P + i], up to the order of
 * the fp64 additions: sum_j w_j r_j(t, first i + 1 poses) over this shard, w_j = 1 without a weight.  Each row is
 * non-decreasing in i up to the fp32 rounding of single terms.  A pose with 0/0 normalisers (it sees nothing) makes its
 * prefix and every later one NaN, as it makes the truncated sweeps'.  With a multi-camera rig (pose index
 * body*n_cams + cam) the prefix after body k is entry (k+1)*n_cams - 1.
 *   prefix_sums_dev  n_traj * P doubles, OVERWRITTEN (the call zeroes them first).  Shard-additive: SUM over the ranks.
 *   minmax_dev       (2, n_traj*P): the normalisers, as for cov_sweep_rewards.
 *   prior_dev, weight_dev  NULL, or as for the _prior / _weighted sweeps; NULL pointers select the plain variant.
 *   base_dev         NULL without prior and weight (the base is n/2); cov_prior_reward_sum's double with a prior alone;
 *                    cov_weight_sums' two doubles with a weight (with or without a prior).  Anything else: COV_ERR_ARG.
 *   opts             dense as for cov_sweep_rewards (no small-cloud threshold: the pruned path for any n unless dense);
 *                    stats_dev is not used (cov_sweep_rewards counts nothing either).  The pruned path takes
 *                    P <= cov_traj_max_poses_pruned() (else COV_ERR_UNSUPPORTED).
 *   workspace_dev    cov_sweep_workspace_bytes(n, n_traj, P) bytes, 256-byte aligned.
 * ------------------------------------------------------------------------------------------ */
int cov_sweep_prefix_rewards(const float* xyz_dev, int64_t n, const float* poses_dev, const float* quats_dev,
                             int n_traj, int poses_per_traj, const float* K_dev, const cov_camera* cam,
                             const float* boxes_dev, const float* minmax_dev, const float* prior_dev,
                             const float* weight_dev, const double* base_dev, double* prefix_sums_dev,
                             const cov_traj_opts* opts, void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Batched ModelPose: K candidate poses (t_k, q~_k) on one cloud, for every k the COV_POSE_ACC sums cov_pose_fused
 * computes for pose k alone ([0] sum m, [1..3] F, [4..6] T, [7] 0), in one pass over the cloud per chunk of poses.
 * ref: src/model.py:98-127 per pose (multi-start pose optimisation, scoring of candidate views); no per-point output.
 *   weight_dev (n) or NULL: one weight per point shared by all poses.  trans_dev (K,3), quats_dev (K,4) fp32.
 *   boxes_dev: NULL, or cov_tile_boxes of this cloud: a warp then skips a (128-point box, pose) pair whose distance
 *   Gaussian bound is below 2^-128, where every pair is exactly 0 (exact; pays on clouds much larger than the
 *   ~27 m reach of the default clip limits).  No boxes are built inside the call: with NULL every pair is evaluated.
 *   acc_dev: K blocks of COV_POSE_ACC doubles, initialised by the call.  Shard-additive: with a sharded cloud, SUM the
 *   blocks over the ranks, then run cov_pose_batch_epilogue.  Sums are fp32 within one (box, pose), fp64 above.
 *   opts: honours `dense` (ignore boxes_dev) and `stats_dev` ([0] (warp box, pose) pairs, [1] pairs evaluated).
 *   workspace_dev: cov_pose_batch_workspace_bytes(n, K, opts) bytes, 16-byte aligned (xyz and weight likewise).
 * ------------------------------------------------------------------------------------------ */
size_t cov_pose_batch_workspace_bytes(int64_t n, int n_poses, const cov_traj_opts* opts);
int cov_pose_batch_fused(const float* xyz_dev, int64_t n, const float* weight_dev, const float* trans_dev,
                         const float* quats_dev, int n_poses, const float* K_dev, const cov_camera* cam,
                         const float* boxes_dev, double* acc_dev, const cov_traj_opts* opts, void* workspace_dev,
                         size_t workspace_bytes, void* stream);
/* out_dev (K, 8) fp32: row k is what cov_pose_epilogue gives for acc block k and quat k, bit for bit. */
int cov_pose_batch_epilogue(const double* acc_dev, const float* quats_dev, int n_poses, float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * The two exchange steps of the point-sharded objective (MAX of the 2 W normalisers, SUM of the 22 W + 1 accumulator
 * doubles) as ONE small kernel each over NVLink peer memory, in place of a collective-library launch.
 * ref: no reference code (the reference is single-process); replaces the dist.all_reduce calls of SURVEY.md 8e.
 * Every rank (one process per GPU of one NVLink domain) owns an exchange buffer that all peers can address — the host
 * allocates it as symmetric memory and passes the world's pointers; it must be ZERO-INITIALISED once and then belongs
 * to the library.  Every rank issues the same sequence of calls.  The kernel pushes its vector into every peer's buffer,
 * raises per-slice flags, waits for the world's flags in its own buffer and reduces in rank order (bit-identical
 * results on all ranks); capturable in CUDA graphs (the call epoch is a device-side counter).
 *   kind: COV_PEER_MAX_F32 / COV_PEER_MINMAX_F32 (data_dev = n floats) or COV_PEER_SUM_F64 (n doubles), reduced IN PLACE.
 *   region_offset: where this call site's region starts inside the exchange buffers (256-byte aligned; one region of
 *   cov_peer_region_bytes(kind, n, world) bytes per call site and vector length).
 * ------------------------------------------------------------------------------------------ */
#define COV_MAX_PEERS 16
#define COV_PEER_MAX_F32 0
#define COV_PEER_SUM_F64 1
#define COV_PEER_MINMAX_F32 2 /* n floats: MIN over the first n/2, MAX over the rest (the 2 W normalisers) */
typedef struct cov_peers {
    void* ptr[COV_MAX_PEERS]; /* rank r's exchange buffer as addressable from THIS device */
    int world;
    int rank;
} cov_peers;
size_t cov_peer_region_bytes(int kind, int64_t n, int world);
int cov_peer_allreduce(int kind, void* data_dev, int64_t n, const cov_peers* peers, size_t region_offset, void* stream);

/* ------------------------------------------------------------------------------------------
 * Multi-camera front end: n_body waypoints (x, y, z, yaw) x n_cams fixed extrinsics -> camera poses in the layout
 * cov_traj_* / cov_sweep_rewards take (pose index = body*n_cams + cam), and the chain rule back.
 * ref: no reference implementation (BASELINE north_star item 3); the camera rig is the tf extrinsics of
 * src/pc_processor.py:33-39,161-165; the reference's optimisable parameters are the outputs (src/model.py:170-171).
 *   body_dev (n_body,4) fp32;  rig_dev (n_cams,7) fp32: unit quaternion q_body_cam (w,x,y,z), lever arm t_body_cam
 *   q_world_cam = q_z(yaw) (x) q_body_cam,  t_world_cam = xyz + R_z(yaw) t_body_cam
 *   backward: g_poses_dev (n_body*n_cams,3) and/or g_quats_dev (n_body*n_cams,4) (either may be NULL) ->
 *   g_body_dev (n_body,4) = scale * d/d(x,y,z,yaw).
 * ------------------------------------------------------------------------------------------ */
int cov_rig_poses(const float* body_dev, int n_body, const float* rig_dev, int n_cams, float* poses_dev,
                  float* quats_dev, void* stream);
int cov_rig_poses_backward(const float* body_dev, int n_body, const float* rig_dev, int n_cams,
                           const float* g_poses_dev, const float* g_quats_dev, float scale, float* g_body_dev,
                           void* stream);

/* ------------------------------------------------------------------------------------------
 * Binary frustum cull.  ref: src/tools.py:176-187 (get_cam_frustum_pts), src/model.py:34-39.
 *   xyz_dev (n,3) camera-frame points (row-major; the Python wrapper accepts the reference's 3xN).
 *   dist_mask_dev, fov_mask_dev: (n) uint8 out;  idx_dev: (n) int32 out, first *count entries valid,
 *   ascending;  count_dev: int64 out.
 * ------------------------------------------------------------------------------------------ */
size_t cov_cull_workspace_bytes(int64_t n);
int cov_frustum_cull(const float* xyz_dev, int64_t n, const float* K_dev, float img_width, float img_height,
                     float min_dist, float max_dist, uint8_t* dist_mask_dev, uint8_t* fov_mask_dev,
                     int32_t* idx_dev, int64_t* count_dev, void* workspace_dev, size_t workspace_bytes,
                     void* stream);

/* ------------------------------------------------------------------------------------------
 * Katz hidden-point removal.  ref: src/tools.py:38-53 (sphericalFlip), :56-64 (convexHull),
 * :67-85 (hidden_pts_removal).
 *   cov_hpr_flip: fp32, every operation rounded in the reference's order; radius_dev is 2 fp32:
 *   [0] = R = max|p| * scale (out), [1] = max|p| (scratch/out).
 *   cov_hpr_hull: vertex set of conv(flipped U {0}); writes vertex_mask (n) uint8 (1 = hull vertex) and
 *   info_dev (4 int32): [0] origin is a hull vertex, [1] number of decisions whose fp64 certificate could
 *   not be validated (0 on non-degenerate input), [2] number of vertices among the n points, [3] GJK iterations.
 * ------------------------------------------------------------------------------------------ */
int cov_hpr_flip(const float* xyz_dev, int64_t n, float scale /* 10**param */, float* flipped_dev,
                 float* radius_dev, void* stream);
size_t cov_hpr_hull_workspace_bytes(int64_t n);
int cov_hpr_hull(const float* flipped_dev, int64_t n, uint8_t* vertex_mask_dev, int32_t* info_dev,
                 void* workspace_dev, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * PointCloud2 payload <-> xyz on the device (SURVEY.md 8f3: keeps the host out of the per-message path).
 * ref: src/pointcloud_utils.py:58-80 (pointcloud2_to_array), :180-198 (get_xyz_points, pointcloud2_to_xyz_array),
 *      :290-338 (xyz_array_to_pointcloud2, xyzi_array_to_pointcloud2).
 *   data_dev: the message's `data` bytes on the device, n = width*height records of point_step bytes (little
 *   endian, as the reference assumes); off_x/y/z: byte offsets of the x, y, z fields; datatype: their PointField
 *   datatype, 7 = FLOAT32 or 8 = FLOAT64 (converted to fp32); fields need not be aligned.
 *   remove_nans != 0: keep only points whose x, y, z are all finite, order preserved (np.isfinite mask).
 *   xyz_dev (n,3) fp32 out, first *count_dev rows valid; count_dev int64 out.
 *   cov_xyz_to_pc2: (n,3) fp32 [+ (n) fp32 fourth field, or NULL] -> n records of 12 [16] bytes;
 *   is_dense_dev (int) != 0 iff every value written is finite (the message's is_dense).
 * ------------------------------------------------------------------------------------------ */
size_t cov_pc2_workspace_bytes(int64_t n);
int cov_pc2_to_xyz(const uint8_t* data_dev, int64_t n, int point_step, int off_x, int off_y, int off_z, int datatype,
                   int remove_nans, float* xyz_dev, int64_t* count_dev, void* workspace_dev, size_t workspace_bytes,
                   void* stream);
int cov_xyz_to_pc2(const float* xyz_dev, const float* extra_dev, int64_t n, uint8_t* data_dev, int* is_dense_dev,
                   void* stream);

/* ------------------------------------------------------------------------------------------
 * Voxel-grid downsample with an optional pass-through on one axis (SURVEY.md 8f4).
 * ref: launch/voxels_filtering.launch:8-21 (pcl/VoxelGrid nodelet in front of the optimiser: leaf_size 0.1,
 * filter_field_name z, filter_limit_min/max, filter_limit_negative False).  Algorithm restated from
 * pcl::VoxelGrid<PointXYZ>::applyFilter (PCL 1.8-1.10, third party, not in the reference tree): finite points with
 * limit_min <= p[filter_axis] <= limit_max (filter_axis -1: no pass-through) are binned into voxels of edge `leaf`
 * anchored at floor(min/leaf); output = one fp32 centroid per occupied voxel, ascending voxel index (x fastest).
 *   xyz_out_dev (n,3) fp32, first *count_dev rows valid;  info_dev 8 int32: [0..2] min_b, [3..5] div_b,
 *   [6] != 0: the grid would have more than 2^31-1 cells (PCL: "Leaf size is too small"), nothing is written,
 *   [7] number of voxels.
 * ------------------------------------------------------------------------------------------ */
size_t cov_voxel_grid_workspace_bytes(int64_t n);
int cov_voxel_grid(const float* xyz_dev, int64_t n, float leaf, int filter_axis, float limit_min, float limit_max,
                   float* xyz_out_dev, int64_t* count_dev, int32_t* info_dev, void* workspace_dev,
                   size_t workspace_bytes, void* stream);

/* Spatial (Morton) ordering of a cloud, done once per cloud (the reference hands the optimiser one fixed cloud:
 * src/trajectory_optimization.py:83-96, src/model.py:164), so that consecutive points are close in space and the
 * tile-level pruning above applies.  Keys are 30-bit Morton codes of the points quantised to a cubic grid of
 * 1024 cells along the longest extent of the bounding box; the sort is stable, hence deterministic.
 *   xyz_sorted_dev (n,3) fp32 out;  perm_dev (n) int32 out: xyz_sorted[j] = xyz[perm[j]]  (n < 2^31). */
size_t cov_spatial_sort_workspace_bytes(int64_t n);
/* Bounding boxes of runs of COV_BOX_POINTS consecutive points of a cloud (any order; tight after cov_spatial_sort):
 * boxes_dev receives cov_tile_boxes_count(n) boxes of 8 fp32 each, (lo.xyz, 0, hi.xyz, 0); boxes past the end of the
 * cloud are empty (+inf, -inf).  16-byte aligned. */
#define COV_BOX_POINTS 128
int64_t cov_tile_boxes_count(int64_t n);
int cov_tile_boxes(const float* xyz_dev, int64_t n, float* boxes_dev, void* stream);
int cov_spatial_sort(const float* xyz_dev, int64_t n, float* xyz_sorted_dev, int32_t* perm_dev, void* workspace_dev,
                     size_t workspace_bytes, void* stream);

/* The stable radix sort of (uint32 key, int32 value) pairs that cov_spatial_sort and cov_voxel_grid are built on (own
 * kernels, csrc/cov_radix.cuh), on its own: sorts in place by key bits [begin_bit, end_bit), equal keys keep their order.
 * No reference counterpart (torch.sort / pcl's std::sort would be the nearest); exported for tests and tools. */
size_t cov_sort_pairs_workspace_bytes(int64_t n);
int cov_sort_pairs(uint32_t* keys_dev, int32_t* vals_dev, int64_t n, int begin_bit, int end_bit, void* workspace_dev,
                   size_t workspace_bytes, void* stream);

/* FP32 FMA / MUFU.EX2 throughput probes used by bench.py for the roofline denominators.
 * Each runs `iters` dependent-chain iterations on a full grid and writes a checksum; the caller
 * times them with CUDA events.  Returns the number of FMA (or ex2) operations issued. */
int64_t cov_probe_fma(int iters, float* sink_dev, void* stream);
int64_t cov_probe_fma2(int iters, float* sink_dev, void* stream); /* packed pairs: fma.rn.f32x2 (FFMA2) */
int64_t cov_probe_ex2(int iters, float* sink_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* COVERAGE_B200_H */
