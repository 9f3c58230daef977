// cov_common.cuh — device math shared by every coverage kernel (sm_100a).
//
// One (point, pose) visibility evaluation, written with explicit round-to-nearest
// intrinsics so that every kernel that instantiates it (min/max pass, fused pass, the
// gradient walk, the sweep) produces BIT-IDENTICAL m for the same inputs: the tie tests
// of the min/max-normalisation backward (m - a == b, m == a) rely on that.
//
// Math (SURVEY.md App. A.1; reference src/model.py:13-57), restated in the world frame with the
// pose translation folded into per-pose constants (P = K R^T, c = R^T (x - t)):
//   e   = x - td,            td = t + R mu1            (|e|^2 = |c - mu1|^2)
//   den = P2.x + (eps - P2.t)                          (= h2 + eps)
//   g0  = cw (P0.x - P0.t),  g1 = ch (P1.x - P1.t)     (cw = sqrt(kf)/W, ch = sqrt(kf)/H, kf = log2e/2)
//   r   = 1/((1 + 2^(-log2e (den - eps))) den);  zi = r (1 + ..) = 1/(h2+eps);  s = r den = sigmoid(h2)
//   du  = g0 zi - sqrt(kf)/2 (= sqrt(kf) (u/W - 1/2)),  dv likewise
//   m   = s * 2^-(kd |e|^2 + du^2 + dv^2),  kd = log2e/(2 sigma^2)
// 26 FP32-pipe instructions + 1 FMNMX + 3 MUFU (2 ex2, 1 rcp) per evaluation: the three Gaussians
// share one ex2, the sigmoid and the projection share one rcp.
// Gradient w.r.t. the point in the world frame (verified against fp64 autograd through the oracle):
//   dm/dx = m [ -e/sigma^2 + A P0' + B P1' + (1-s - A (du-c0) - B (dv-c0)) P2 ],
//   A = -2 ln2 du zi, B = -2 ln2 dv zi, P0' = cw P0, P1' = ch P1, c0 = -sqrt(kf)/2
//   dm/dtheta (world-frame rotation of the camera about its centre) = dm/dx x (x - t).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define COV_LOG2E_F 1.4426950408889634f
#define COV_LN2_F 0.6931471805599453f
#define COV_THREADS 256
#define COV_MAX_GRID 1024

// Per-launch constants, computed on the host from cov_camera.
struct CovConst {
    float eps;      // added to the depth in the two projections
    float kd;       // 0.5*log2(e)/sigma^2
    float zk;       // -log2(e)
    float zc;       // log2(e)*eps        (2^(zk*den + zc) = exp(-h2))
    float c0;       // -0.5*sqrt(0.5*log2(e))
    float cw, ch;   // sqrt(0.5*log2(e))/img_width, /img_height
    float inv_s2;   // 1/sigma^2
    float mu;       // (min_dist+max_dist)/2
    float hi;       // fp32(1 - eps): upper clip of the normalised observation
};

// One pose row = 6 float4 in shared memory (broadcast LDS.128):
//   v0 = (cw P0, -cw P0.t)   v1 = (ch P1, -ch P1.t)   v2 = (P2, eps - P2.t)   v3 = (td, a)
//   v4 = (hb, b, 1/b, 0)     v5 = (t, 0)              a = min_j m, b = max_j m - a, hb = b/2
// The forward needs v0..v3 (+v4 in the fused pass); v5 only feeds the rare gradient path.
#define COV_ROW_F4 6

__device__ __forceinline__ float cov_ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float cov_rcp(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float cov_lg2(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Build one pose row from (t, q~, K): R(q) camera->world with q = q~/max(|q~|,1e-12)
// (F.normalize, src/model.py:53), P = K R^T.  Computed in fp64, stored fp32.
__device__ inline void cov_pose_row(const float* __restrict__ t3, const float* __restrict__ q4,
                                    const float* __restrict__ K9, const CovConst& C, float4* __restrict__ row) {
    double w = q4[0], x = q4[1], y = q4[2], z = q4[3];
    double n = sqrt(w * w + x * x + y * y + z * z);
    n = n > 1e-12 ? n : 1e-12;
    w /= n; x /= n; y /= n; z /= n;
    const double R[3][3] = {{1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)},
                            {2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)},
                            {2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)}};
    const double t[3] = {t3[0], t3[1], t3[2]};
    double P[3][3], pt[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j)
            P[i][j] = (double)K9[i * 3 + 0] * R[j][0] + (double)K9[i * 3 + 1] * R[j][1] + (double)K9[i * 3 + 2] * R[j][2];
        pt[i] = P[i][0] * t[0] + P[i][1] * t[1] + P[i][2] * t[2];
    }
    const double cw = C.cw, ch = C.ch, mu = C.mu;
    row[0] = make_float4((float)(cw * P[0][0]), (float)(cw * P[0][1]), (float)(cw * P[0][2]), (float)(-cw * pt[0]));
    row[1] = make_float4((float)(ch * P[1][0]), (float)(ch * P[1][1]), (float)(ch * P[1][2]), (float)(-ch * pt[1]));
    row[2] = make_float4((float)P[2][0], (float)P[2][1], (float)P[2][2], (float)((double)C.eps - pt[2]));
    row[3] = make_float4((float)(t[0] + mu * (R[0][0] + R[0][1] + R[0][2])), (float)(t[1] + mu * (R[1][0] + R[1][1] + R[1][2])),
                         (float)(t[2] + mu * (R[2][0] + R[2][1] + R[2][2])), 0.f);
    row[4] = make_float4(0.f, 0.f, 0.f, 0.f);
    row[5] = make_float4(t3[0], t3[1], t3[2], 0.f);
}

// Normalisation constants of a pose row from its extrema a = min_j m and mx = max_j m: row[4] = (b/2, b, 1/b, a),
// b = mx - a, and the conservative gate threshold thr = (a + b/2)(1 - 2^-20) (no pair below it is gated), which goes
// where the caller's table layout keeps it.  thr is written before row[4] (not returned): for a row in shared memory
// the other store order costs the dense sweep kernel 4 more registers.
__device__ __forceinline__ void cov_norm_row(float4* row, float a, float mx, float& thr) {
    const float b = __fsub_rn(mx, a);
    const float hb = 0.5f * b;
    thr = (a + hb) * (1.f - 9.5367431640625e-07f);
    row[4] = make_float4(hb, b, __frcp_rn(b), a);
}

// |x - td|^2 exactly as cov_vis computes it (same three instructions per component), for the pruning
// pre-filter:  m = s * 2^-(kd q2 + ...) <= 2^-(kd q2) * (1 + 1.3e-5)   (s <= 1 up to the rcp rounding).
__device__ __forceinline__ float cov_q2(float x, float y, float z, const float4& v3) {
    const float ex = __fsub_rn(x, v3.x), ey = __fsub_rn(y, v3.y), ez = __fsub_rn(z, v3.z);
    return __fmaf_rn(ez, ez, __fmaf_rn(ey, ey, __fmul_rn(ex, ex)));
}

// Lower bound of cov_q2(x, y, z, v3) over every point of the box [lo, hi].  Rounding is monotone, so with the same
// operation sequence as cov_q2 (fsub, then fmul/fma/fma) the bound holds for the COMPUTED q2 of each point, exactly:
// |fl(x - td)| >= max(fl(lo - td), fl(td - hi), 0) for lo <= x <= hi.  An empty box (lo = +inf) gives +inf.
__device__ __forceinline__ float box_q2lb(const float4& lo, const float4& hi, const float4& v3) {
    const float dx = fmaxf(fmaxf(__fsub_rn(lo.x, v3.x), __fsub_rn(v3.x, hi.x)), 0.f);
    const float dy = fmaxf(fmaxf(__fsub_rn(lo.y, v3.y), __fsub_rn(v3.y, hi.y)), 0.f);
    const float dz = fmaxf(fmaxf(__fsub_rn(lo.z, v3.z), __fsub_rn(v3.z, hi.z)), 0.f);
    return __fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx)));
}

struct CovEval {  // intermediates the gradient needs
    float ex, ey, ez, zi, s, e2z, du, dv;
};

// m for one (point, pose).  WANT = true also fills the intermediates.
template <bool WANT>
__device__ __forceinline__ float cov_vis(float x, float y, float z, const float4& v0, const float4& v1,
                                         const float4& v2, const float4& v3, const CovConst& C, CovEval* ev) {
    const float ex = __fsub_rn(x, v3.x), ey = __fsub_rn(y, v3.y), ez = __fsub_rn(z, v3.z);
    const float q2 = __fmaf_rn(ez, ez, __fmaf_rn(ey, ey, __fmul_rn(ex, ex)));
    const float g0 = __fmaf_rn(v0.z, z, __fmaf_rn(v0.y, y, __fmaf_rn(v0.x, x, v0.w)));
    const float g1 = __fmaf_rn(v1.z, z, __fmaf_rn(v1.y, y, __fmaf_rn(v1.x, x, v1.w)));
    const float den = __fmaf_rn(v2.z, z, __fmaf_rn(v2.y, y, __fmaf_rn(v2.x, x, v2.w)));
    const float e2z = cov_ex2(fminf(__fmaf_rn(den, C.zk, C.zc), 80.f));  // exp(-h2), capped
    const float opz = __fadd_rn(1.f, e2z);
    const float r = cov_rcp(__fmul_rn(opz, den));
    const float zi = __fmul_rn(r, opz);   // 1/(h2+eps)
    const float s = __fmul_rn(r, den);    // sigmoid(h2)
    const float du = __fmaf_rn(g0, zi, C.c0), dv = __fmaf_rn(g1, zi, C.c0);
    const float Q = __fmaf_rn(q2, C.kd, __fmaf_rn(dv, dv, __fmul_rn(du, du)));
    const float E = cov_ex2(-Q);
    if (WANT) {
        ev->ex = ex; ev->ey = ey; ev->ez = ez;
        ev->zi = zi; ev->s = s; ev->e2z = e2z; ev->du = du; ev->dv = dv;
    }
    return __fmul_rn(E, s);
}

// Log-odds term of a gated (point, pose) with v4 = (b/2, b, 1/b, a) (cov_norm_row): the pair is gated exactly when
// p = d/b >= 1/2 for d = m - a, i.e. when d >= b/2, and then adds logit(min(p, hi)) to the point's log-odds sum.  The
// gate test stays with the callers: the dense pass B takes a warp ballot of it before it branches to the log-odds and
// the tie test, and folding the test in here would split that branch in two (more instructions in its hot loop).
__device__ __forceinline__ float cov_logodds(float d, const float4& v4, const CovConst& C) {
    const float p = __fmul_rn(d, v4.z);
    const float qc = (p > C.hi) ? C.hi : p;  // upper clip; a NaN p (pose that sees nothing: 0/0) stays NaN, as torch.clip
    return COV_LN2_F * cov_lg2(qc * cov_rcp(1.f - qc));
}

// A point's reward from its fused log-odds x (prior + L): the expression every pass B and sweep kernel uses, so that a
// reward computed anywhere (pre-fill, pass B, sweeps, sigma of the fused log-odds output) is the same float.
__device__ __forceinline__ float cov_sigmoid(float x) { return 1.f / (1.f + expf(-x)); }
__device__ __forceinline__ float4 cov_sigmoid4(float4 x) {
    return make_float4(cov_sigmoid(x.x), cov_sigmoid(x.y), cov_sigmoid(x.z), cov_sigmoid(x.w));
}
// x = prior + L, one IEEE add (the fused log-odds output writes the same float)
__device__ __forceinline__ float cov_fuse_prior(float prior, float L) { return __fadd_rn(prior, L); }

// ---- packed fp32 pairs (sm_100: fma/mul/add/sub.rn.f32x2 -> FFMA2 / FMUL2 / FADD2) --------------------------------
// One instruction does the IEEE round-to-nearest operation on both halves of a 64-bit register pair, at half the issue
// rate of the scalar instruction: the same flop/s, HALF THE ISSUE SLOTS.  The evaluation is issue-bound (26 FP32-pipe
// instructions next to 3 MUFU and the loop skeleton), so packing two evaluations into one instruction stream frees the
// issue slots the FP32 pipe was waiting for.  Per half the results are bit-identical to the scalar __f*_rn intrinsics.
typedef unsigned long long f2_t;
__device__ __forceinline__ f2_t f2_pack(float lo, float hi) {
    f2_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void f2_unpack(f2_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f2_t f2_fma(f2_t a, f2_t b, f2_t c) {
    f2_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ f2_t f2_mul(f2_t a, f2_t b) {
    f2_t r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f2_t f2_add(f2_t a, f2_t b) {
    f2_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f2_t f2_sub(f2_t a, f2_t b) {
    f2_t r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f2_t f2_lo(const float4& v) { return f2_pack(v.x, v.y); }
__device__ __forceinline__ f2_t f2_hi(const float4& v) { return f2_pack(v.z, v.w); }

// Per-launch constants as broadcast pairs (built once per kernel).
struct CovConst2 {
    f2_t kd, zk, zc, c0, one;
};
__device__ __forceinline__ CovConst2 cov_make_const2(const CovConst& C) {
    CovConst2 c;
    c.kd = f2_pack(C.kd, C.kd);
    c.zk = f2_pack(C.zk, C.zk);
    c.zc = f2_pack(C.zc, C.zc);
    c.c0 = f2_pack(C.c0, C.c0);
    c.one = f2_pack(1.f, 1.f);
    return c;
}

// Rows v0..v3 of TWO poses (A, B) interleaved component-wise, the layout the dense kernels keep in shared memory so
// that one LDS.128 delivers two packed constants:  q[2i] = (v_i.x A, v_i.x B, v_i.y A, v_i.y B),
// q[2i+1] = (v_i.z A, v_i.z B, v_i.w A, v_i.w B), i = 0..3.  A pose PAIR occupies COV_PAIR_F4 float4:
// q[0..7], then v4 A, v4 B, v5 A, v5 B.
#define COV_PAIR_F4 12
__device__ __forceinline__ void cov_pair_store(float4* __restrict__ pair, int slot, const float4* __restrict__ row) {
    float* f = reinterpret_cast<float*>(pair);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        f[(2 * i) * 4 + slot] = row[i].x;
        f[(2 * i) * 4 + 2 + slot] = row[i].y;
        f[(2 * i + 1) * 4 + slot] = row[i].z;
        f[(2 * i + 1) * 4 + 2 + slot] = row[i].w;
    }
    pair[8 + slot] = row[4];
    pair[10 + slot] = row[5];
}
// scalar row i (0..3) of the pose in `slot` out of the pair layout (rare paths: gradient walk, tie sets)
__device__ __forceinline__ float4 cov_pair_row(const float4* __restrict__ pair, int slot, int i) {
    const float* f = reinterpret_cast<const float*>(pair);
    return make_float4(f[(2 * i) * 4 + slot], f[(2 * i) * 4 + 2 + slot], f[(2 * i + 1) * 4 + slot], f[(2 * i + 1) * 4 + 2 + slot]);
}

// m of ONE point against a pose PAIR: (m_A, m_B), each half bit-identical to cov_vis with that pose's rows.
// X, Y, Z are the point's coordinates as broadcast pairs (built once per tile); q[0..7] as laid out above.
__device__ __forceinline__ f2_t cov_vis2p(f2_t X, f2_t Y, f2_t Z, const float4& q0, const float4& q1, const float4& q2_,
                                          const float4& q3, const float4& q4, const float4& q5, const float4& q6,
                                          const float4& q7, const CovConst2& C) {
    const f2_t ex = f2_sub(X, f2_lo(q6)), ey = f2_sub(Y, f2_hi(q6)), ez = f2_sub(Z, f2_lo(q7));
    const f2_t q2 = f2_fma(ez, ez, f2_fma(ey, ey, f2_mul(ex, ex)));
    const f2_t g0 = f2_fma(f2_lo(q1), Z, f2_fma(f2_hi(q0), Y, f2_fma(f2_lo(q0), X, f2_hi(q1))));
    const f2_t g1 = f2_fma(f2_lo(q3), Z, f2_fma(f2_hi(q2_), Y, f2_fma(f2_lo(q2_), X, f2_hi(q3))));
    const f2_t den = f2_fma(f2_lo(q5), Z, f2_fma(f2_hi(q4), Y, f2_fma(f2_lo(q4), X, f2_hi(q5))));
    float ta, tb;
    f2_unpack(f2_fma(den, C.zk, C.zc), ta, tb);
    const f2_t e2z = f2_pack(cov_ex2(fminf(ta, 80.f)), cov_ex2(fminf(tb, 80.f)));  // exp(-h2), capped
    const f2_t opz = f2_add(C.one, e2z);
    float pa, pb;
    f2_unpack(f2_mul(opz, den), pa, pb);
    const f2_t r = f2_pack(cov_rcp(pa), cov_rcp(pb));
    const f2_t zi = f2_mul(r, opz);   // 1/(h2+eps)
    const f2_t s = f2_mul(r, den);    // sigmoid(h2)
    const f2_t du = f2_fma(g0, zi, C.c0), dv = f2_fma(g1, zi, C.c0);
    float Qa, Qb;
    f2_unpack(f2_fma(q2, C.kd, f2_fma(dv, dv, f2_mul(du, du))), Qa, Qb);
    return f2_mul(f2_pack(cov_ex2(-Qa), cov_ex2(-Qb)), s);
}

// dm/dx (world frame) from the intermediates; g = 0 when m is not a positive finite number.
__device__ __forceinline__ void cov_vis_grad(float m, const CovEval& ev, const float4& v0, const float4& v1,
                                             const float4& v2, const CovConst& C, float& gx, float& gy, float& gz) {
    const float oms = ev.e2z * ev.s;                          // 1 - sigmoid(h2)
    const float A = (-2.f * COV_LN2_F) * ev.du * ev.zi;       // coefficient of row 0 (cw P0)
    const float B = (-2.f * COV_LN2_F) * ev.dv * ev.zi;       // coefficient of row 1 (ch P1)
    const float Cz = oms - A * (ev.du - C.c0) - B * (ev.dv - C.c0);  // coefficient of P2
    const float ax = -ev.ex * C.inv_s2 + A * v0.x + B * v1.x + Cz * v2.x;
    const float ay = -ev.ey * C.inv_s2 + A * v0.y + B * v1.y + Cz * v2.y;
    const float az = -ev.ez * C.inv_s2 + A * v0.z + B * v1.z + Cz * v2.z;
    const bool ok = m > 0.f;
    gx = ok ? m * ax : 0.f;
    gy = ok ? m * ay : 0.f;
    gz = ok ? m * az : 0.f;
}

__device__ __forceinline__ float cov_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double cov_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// 8 sums over 32 lanes in 9 shuffles, in a fixed order: halve the number of values a lane carries at offsets 16, 8, 4 (a
// lane keeps the half its lane bit selects and hands the other half over), then two plain steps.  Afterwards the lanes
// with (lane & 3) == 0 hold in v[0] the warp sum of component (lane bits 4,3,2); v[1..7] are left as scratch.
__device__ __forceinline__ void cov_warp_sum8(float (&v)[8], int lane) {
    {
        const bool up = (lane & 16) != 0;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float keep = up ? v[q + 4] : v[q], send = up ? v[q] : v[q + 4];
            v[q] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
    }
    {
        const bool up = (lane & 8) != 0;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const float keep = up ? v[q + 2] : v[q], send = up ? v[q] : v[q + 2];
            v[q] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
    }
    {
        const bool up = (lane & 4) != 0;
        const float keep = up ? v[1] : v[0], send = up ? v[0] : v[1];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    }
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 2);
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
}

// ---- TMA bulk copies (global -> shared) completing on an mbarrier ------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_copy(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// the labels live inside the { } scope, so every inlined copy of the loop has its own
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// ---- host-side helpers (cov_api.cu) ----
void cov_set_error(const char* fmt, ...);
int cov_check_launch(const char* what);
CovConst cov_make_const(const struct cov_camera* cam);
int cov_sm_count_cached();
int cov_sweep_rewards_dense(const float* xyz, int64_t n, const float* poses, const float* quats, int n_traj, int per_traj,
                            const float* K, const struct cov_camera* cam, const float* minmax, double* sum_rewards,
                            const float* prior, const double* prior_sum, const float* weight, void* stream,
                            bool prefix = false);
