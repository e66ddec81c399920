// fmb_common.cuh -- shared device helpers for the FM hot path (sm_100a).
//
// Parity-critical fp32 arithmetic is written with explicit round-to-nearest intrinsics
// (__fmul_rn/__fadd_rn/__fsub_rn/__fmaf_rn/__fdiv_rn/__fsqrt_rn) so nvcc can never contract a
// multiply-add that ATen executes as two roundings (SURVEY.md section 7 "hard parts"); the
// library is additionally built with -fmad=false.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "fmb_aten_math.cuh"

#define FMB_API extern "C" __attribute__((visibility("default")))

// ---- error plumbing (thread-local message, int status; no exceptions cross the C ABI) ----
void fmb_set_error(const char* fmt, ...);
#define FMB_OK 0
#define FMB_ERR_ARG (-1)
#define FMB_ERR_CUDA (-2)
#define FMB_ERR_WS (-3)
#define FMB_CHECK_ARG(cond, ...)                         \
    do {                                                 \
        if (!(cond)) { fmb_set_error(__VA_ARGS__); return FMB_ERR_ARG; } \
    } while (0)
#define FMB_CHECK_LAUNCH(name)                                                           \
    do {                                                                                 \
        cudaError_t e__ = cudaGetLastError();                                            \
        if (e__ != cudaSuccess) { fmb_set_error("%s: %s", name, cudaGetErrorString(e__)); return FMB_ERR_CUDA; } \
    } while (0)

static inline int fmb_round_up(int x, int m) { return (x + m - 1) / m * m; }

// x / d by multiplication, for d >= 1 and x * d < 2^31: __umulhi(2x, floor(2^31 / d) + 1).  The error term of the
// multiplier, x * (d - 2^31 mod d) / (d * 2^31), stays below 1/d.  (The 2^32 form, multiplier ceil(2^32 / d), has no
// 32-bit multiplier for d = 1.)
static inline uint32_t fmb_div_magic(unsigned d) { return 0x80000000u / d + 1u; }
__device__ __forceinline__ int fmb_div_by_magic(unsigned x, uint32_t m) { return (int)__umulhi(x << 1, m); }

namespace fmb {

// ---------------------------------------------------------------------------------------------
// portable fp32 expf/logf (Cephes-style, oracle/oracle_math.h group 2): used only for nn.BCELoss values and
// torch.pow in the hedge step (continuous updates, never sign-amplified).  sigmoid / log_sigmoid / sqrt are
// the ATen mirrors of fmb_aten_math.cuh.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float pow2i(int n) { return __int_as_float((n + 127) << 23); }

__device__ __forceinline__ float expf_p(float x) {
    if (x != x) return x;
    if (x > 88.7228317f) return __int_as_float(0x7f800000);
    if (x < -103.972084f) return 0.0f;
    float fn = rintf(__fmul_rn(x, 1.44269504f));
    float r = __fmaf_rn(fn, -0.693359375f, x);
    r = __fmaf_rn(fn, 2.12194440e-4f, r);
    float p = 1.9875691500e-4f;
    p = __fmaf_rn(p, r, 1.3981999507e-3f);
    p = __fmaf_rn(p, r, 8.3334519073e-3f);
    p = __fmaf_rn(p, r, 4.1665795894e-2f);
    p = __fmaf_rn(p, r, 1.6666665459e-1f);
    p = __fmaf_rn(p, r, 5.0000001201e-1f);
    float r2 = __fmul_rn(r, r);
    float y = __fmaf_rn(p, r2, r);
    y = __fadd_rn(y, 1.0f);
    int n = (int)fn;
    int n1 = n / 2;
    int n2 = n - n1;
    y = __fmul_rn(y, pow2i(n1));
    y = __fmul_rn(y, pow2i(n2));
    return y;
}

__device__ __forceinline__ float logf_p(float x) {
    if (x != x) return x;
    if (x < 0.0f) return __int_as_float(0x7fc00000);
    if (x == 0.0f) return __int_as_float(0xff800000);
    if (x == __int_as_float(0x7f800000)) return x;
    int e = 0;
    if (x < 1.17549435e-38f) { x = __fmul_rn(x, 8388608.0f); e = -23; }
    uint32_t b = (uint32_t)__float_as_int(x);
    e += (int)((b >> 23) & 0xffu) - 126;
    float m = __int_as_float((int)((b & 0x807fffffu) | 0x3f000000u));
    if (m < 0.707106781f) { e -= 1; m = __fsub_rn(__fadd_rn(m, m), 1.0f); } else { m = __fsub_rn(m, 1.0f); }
    float z = __fmul_rn(m, m);
    float y = 7.0376836292e-2f;
    y = __fmaf_rn(y, m, -1.1514610310e-1f);
    y = __fmaf_rn(y, m, 1.1676998740e-1f);
    y = __fmaf_rn(y, m, -1.2420140846e-1f);
    y = __fmaf_rn(y, m, 1.4249322787e-1f);
    y = __fmaf_rn(y, m, -1.6668057665e-1f);
    y = __fmaf_rn(y, m, 2.0000714765e-1f);
    y = __fmaf_rn(y, m, -2.4999993993e-1f);
    y = __fmaf_rn(y, m, 3.3333331174e-1f);
    y = __fmul_rn(__fmul_rn(y, m), z);
    float fe = (float)e;
    y = __fmaf_rn(-2.12194440e-4f, fe, y);
    y = __fmaf_rn(-0.5f, z, y);
    float r = __fadd_rn(m, y);
    r = __fmaf_rn(0.693359375f, fe, r);
    return r;
}

// log(1 + u) for any u > -1 (u == -1 -> -inf)
__device__ __forceinline__ float log1pf_p(float u) {
    float w = __fadd_rn(1.0f, u);
    if (w == 1.0f) return u;
    if (w == 0.0f) return __int_as_float(0xff800000);
    float l = logf_p(w);
    float c = __fdiv_rn(__fsub_rn(__fsub_rn(w, 1.0f), u), w);
    return __fsub_rn(l, c);
}

__device__ __forceinline__ float powf_p(float b, float e) { return expf_p(__fmul_rn(e, logf_p(b))); }

// ---------------------------------------------------------------------------------------------
// update rules (SURVEY.md section 8 A6/A12).  mode 0: torch.optim.Adam, first step with fresh
// state, lr an fp32 scalar; mode 1: plain SGD p -= lr*g.
// ---------------------------------------------------------------------------------------------
// astep = -(lr / 0.1f), the (negated) bias-corrected step size: loop-invariant, so callers that update many
// parameters compute it once (adam_astep) and call adam1_a.
__device__ __forceinline__ float adam_astep(float lr) { return -__fdiv_rn(lr, 0.1f); }
// adam1_a in two parts, so that a caller with several coordinates per thread can run the cheap part on all of them
// without branches and the rest only where it is needed (fm_step.cu):
//   adam1_window: true + the result when the window test settles the coordinate; `in_domain` tells adam1_rest which way
//   the test was skipped or failed.
__device__ __forceinline__ bool adam1_in_domain(float g, float a) {
    const float ag = fabsf(g);
    return ag >= 1e-25f && ag < 1e15f && fabsf(a) >= 1e-9f;
}
__device__ __forceinline__ bool adam1_window(float p, float g, float a, float& out) {
    // Exact window test (the common case: ~12 instructions, no sqrt, no division).  In real numbers the step is
    // Q = a*0.1f*g / (sqrt(0.001f)*|g|/c + 1e-8f) = A*g / (|g| + c0), A = a*0.1f/kappa, c0 = 1e-8f/kappa,
    // kappa = sqrt(0.001f)/c = 1.0000000775921325.  The roundings of the float pipeline below (m, v twice -- halved by
    // the root --, MKL's square root at most 1.5 ulp off, the quotient by c, the sum, a*m, the final quotient) keep its
    // result q within 9*2^-24 of Q; the estimate U = fl(fl(A*g) * rcp(fl(|g| + c0))) with MUFU.RCP (1 ulp) is within
    // 8*2^-24 of Q.  So q lies strictly between U*(1 - 2^-19) and U*(1 + 2^-19), and because fl(p + x) is monotone in
    // x, whenever both ends round to the same float that float IS fl(p + q).  Valid wherever every intermediate of
    // both forms is a normal float (or an underflow of v whose effect on the denominator is below 2^-40):
    // 1e-25 <= |g| < 1e15, |a| >= 1e-9.  Measured: worst |q - U| = 7.83 * 2^-24 * |U| over every binade of that range
    // (oracle/verify_math.c qbound: 6.3e8 cases, reciprocal perturbed by +-1 ulp), and 0 disagreements of the window
    // result with the full pipeline on 4e8 random (p, g, lr) triples (verify_math.c window).  The window is ambiguous
    // with probability ~ 2^-18 * lr / ulp(p); those fall through to the full pipeline.
    const float ag = fabsf(g);
    float rc;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(__fadd_rn(ag, 9.99999905e-09f)));   // |g| + fl(1e-8f / kappa)
    const float U = __fmul_rn(__fmul_rn(__fmul_rn(a, 0.099999994f), g), rc);              // a * fl(0.1f / kappa) * g
    const float xa = __fmaf_rn(U, 1.9073486328125e-06f, U), xb = __fmaf_rn(-U, 1.9073486328125e-06f, U);
    const float ra = __fadd_rn(p, xa), rb = __fadd_rn(p, xb);
    out = ra;
    return adam1_in_domain(g, a) && ra == rb;
}
// everything the window test did not settle: the quarter-ulp shortcut (only outside the window's domain, as in adam1_a's
// original control flow), then the full pipeline
__device__ __forceinline__ float adam1_rest(float p, float g, float a, bool in_domain) {
    const float bc2s = 0.03162277660168381f;
    if (!in_domain) {
        // Exact shortcut for the gradients of saturated logits (~1e-30).  The step is q = fl(fl(a*m)/d) with
        // d >= 1e-8f, so |q| <= |a|*0.1*|g|*1e8*(1+2^-22).  When that bound is below a quarter ulp of p the sum
        // fl(p+q) is p itself (and denormal operands would send div.rn/sqrt.rn down their ~100-instruction slow paths).
        const float ap = fabsf(p);
        if (ap > 1e-20f) {
            const float bound = __fmul_rn(__fmul_rn(__fmul_rn(fabsf(a), 0.1f), fabsf(g)), 1.0001e8f);
            if (bound < __fmul_rn(ap, 1.4901161e-8f)) return p;   // 2^-26 * |p|
        }
    }
    float m = __fmul_rn(0.1f, g);
    float v = __fmul_rn(__fmul_rn(0.001f, g), g);
    // denom = exp_avg_sq.sqrt() / bias_correction2_sqrt + eps.  Tensor.sqrt() is MKL's vsSqrt (sqrt_mkl).  For a normal
    // v the quotient s / bc2s is formed without the division: q = RN(s * RN(1/c)), r = s - q*c exactly (one fma),
    // RN(q + r * RN(1/c)) is the correctly rounded quotient -- checked against s / c for ALL 2^23 mantissas of every
    // binade of s from 2^-104 to 2^122 (sqrt of a normal float lies in [2^-63, 2^64)).
    float d1;
    const uint32_t vb = (uint32_t)__float_as_int(v);
    if (vb - 0x00800000u < 0x7f000000u) {
        const float s = sqrt_mkl_normal(v);
        const float rc = 0x1.f9f6e6p+4f;        // RN(1 / bc2s) = 31.6227779...
        const float q = __fmul_rn(s, rc);
        d1 = __fmaf_rn(__fmaf_rn(-q, bc2s, s), rc, q);
    } else {
        d1 = __fdiv_rn(sqrt_mkl(v), bc2s);
    }
    const float d = __fadd_rn(d1, 1e-8f);
    return __fadd_rn(p, __fdiv_rn(__fmul_rn(a, m), d));
}
__device__ __forceinline__ float adam1_a(float p, float g, float a) {
    float out;
    if (adam1_window(p, g, a, out)) return out;
    return adam1_rest(p, g, a, adam1_in_domain(g, a));
}
__device__ __forceinline__ float adam1(float p, float g, float lr) { return adam1_a(p, g, adam_astep(lr)); }
__device__ __forceinline__ float apply_update(float p, float g, float lr, int mode) {
    return mode == 0 ? adam1(p, g, lr) : __fmaf_rn(g, -lr, p);   // SGD: ATen's add_(grad, alpha=-lr) is one fma
}
// mode 2: per-coordinate FTRL-Proximal (McMahan et al. 2013; SURVEY.md 8f.4 -- the reference's FM_FTRL is the
// unregularised linearised form, models/models_online/FM_FTRL.py:76-80, and never keeps n): state z, n per coordinate,
//   n' = n + g^2;  sigma = (sqrt(n') - sqrt(n)) / alpha;  z' = z + (g - sigma*w);
//   w' = |z'| <= l1 ? 0 : -(z' - sign(z')*l1) / ((beta + sqrt(n')) / alpha + l2)
// every operation rounded once, in this order (oracle/fm_oracle.c orc_ftrl_update is the same sequence).
struct FtrlState {
    float* zn;        // [R][2][rowp]: z sub-row, n sub-row of every packed table row (NULL = mode 2 unavailable)
    float* bias_zn;   // [2]: z, n of the bias
    float beta, l1, l2;
};
__device__ __forceinline__ float ftrl_update(float w, float g, float& z, float& n, float alpha, float beta, float l1,
                                             float l2) {
    const float nn = __fadd_rn(n, __fmul_rn(g, g));
    const float sn = __fsqrt_rn(n), snn = __fsqrt_rn(nn);
    const float sigma = __fdiv_rn(__fsub_rn(snn, sn), alpha);
    const float zz = __fadd_rn(z, __fsub_rn(g, __fmul_rn(sigma, w)));
    z = zz; n = nn;
    if (fabsf(zz) <= l1) return 0.f;
    const float num = __fsub_rn(zz, copysignf(l1, zz));
    const float den = __fadd_rn(__fdiv_rn(__fadd_rn(beta, snn), alpha), l2);
    return -__fdiv_rn(num, den);
}
// mode 3: torch.optim.Adagrad (lr_decay = 0, weight_decay = 0) with a persistent per-coordinate sum s, in the order
// torch 2.11's CPU _single_tensor_adagrad rounds it (tests/adagrad_oracle.c orc_adagrad_update is the same sequence, pinned on torch):
//   s' = fma(g, g, s)   (state_sum.addcmul_(grad, grad, value=1))
//   std = sqrt(s') + eps   (state_sum.sqrt(): MKL vsSqrt = sqrt_mkl, then add_(eps))
//   p' = p + (-lr * g) / std   (param.addcdiv_(grad, std, value=-lr): the product first, then the quotient)
// A zero gradient leaves p and s exactly as they are, so updating only the rows a batch hits is the dense optimizer.
struct AdagradState {
    float* sums;      // [R][rowp]: row r's sums at row r's offsets of the packed table (NULL = mode 3 unavailable)
    float* bias_sum;  // [1]
    float eps;
};
// the per-coordinate state of modes 2 and 3 in one kernel argument
union UpdateState {
    FtrlState ftrl;
    AdagradState ada;
};
__device__ __forceinline__ float adagrad_update(float p, float g, float& s, float lr, float eps) {
    const float ss = __fmaf_rn(g, g, s);
    s = ss;
    const float sd = __fadd_rn(sqrt_mkl(ss), eps);
    return __fadd_rn(p, __fdiv_rn(__fmul_rn(-lr, g), sd));
}
// same with the Adam step size precomputed
__device__ __forceinline__ float apply_update_a(float p, float g, float lr, float astep, int mode) {
    return mode == 0 ? adam1_a(p, g, astep) : __fmaf_rn(g, -lr, p);
}

// ---------------------------------------------------------------------------------------------
// F.binary_cross_entropy_with_logits value + gradient for sample b of a batch of B (SURVEY.md 8a A6).
//   kind 0: loss(z)           delta = (sigmoid(z) - y) / B
//   kind 1: loss(sigmoid(z))  delta = (((sigmoid(p) - y) / B) * (1 - p)) * p,  p = sigmoid(z)
// Both sigmoids are torch.sigmoid calls on the [B] tensor, so their bits depend on the position b.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void bce_logits_value_grad(int kind, float z, float y, int b, int B, float& lossv,
                                                      float& delta) {
    float in = z, pr = 0.f;
    if (kind == 1) { pr = sigmoid_at(z, b, B); in = pr; }
    lossv = __fsub_rn(__fmul_rn(__fsub_rn(1.0f, y), in), log_sigmoid(in));
    float d = __fdiv_rn(__fsub_rn(sigmoid_at(in, b, B), y), (float)B);
    if (kind == 1) d = __fmul_rn(__fmul_rn(d, __fsub_rn(1.0f, pr)), pr);
    delta = d;
}

// ---------------------------------------------------------------------------------------------
// ATen's x86 (AVX2 build, 8 lanes x 4 ilp) sum order of a contiguous fp32 row, evaluated by ONE
// thread.  Valid for n < 512 (the 16-step cascade never triggers); restates oracle orc_sum_aten.
// ---------------------------------------------------------------------------------------------
template <typename Load>
__device__ __forceinline__ float aten_row_sum_small(Load ld, int n) {
    if (n < 8) {
        float p0 = 0.f, p1 = 0.f, p2 = 0.f, p3 = 0.f;
        int i = 0;
        if (n >= 4) { p0 = __fadd_rn(p0, ld(0)); p1 = __fadd_rn(p1, ld(1)); p2 = __fadd_rn(p2, ld(2)); p3 = __fadd_rn(p3, ld(3)); i = 4; }
        for (; i < n; ++i) p0 = __fadd_rn(p0, ld(i));
        p0 = __fadd_rn(p0, p1); p0 = __fadd_rn(p0, p2); p0 = __fadd_rn(p0, p3);
        return p0;
    }
    const int vec_size = n >> 3, size_ilp = vec_size >> 2;
    float fin = 0.f;
    for (int i = vec_size << 3; i < n; ++i) fin = __fadd_rn(fin, ld(i));
#pragma unroll 1
    for (int l = 0; l < 8; ++l) {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        for (int i = 0; i < size_ilp; ++i) {
            a0 = __fadd_rn(a0, ld(i * 32 + l));
            a1 = __fadd_rn(a1, ld(i * 32 + 8 + l));
            a2 = __fadd_rn(a2, ld(i * 32 + 16 + l));
            a3 = __fadd_rn(a3, ld(i * 32 + 24 + l));
        }
        for (int v = size_ilp << 2; v < vec_size; ++v) a0 = __fadd_rn(a0, ld(v * 8 + l));
        a0 = __fadd_rn(a0, a1); a0 = __fadd_rn(a0, a2); a0 = __fadd_rn(a0, a3);
        fin = __fadd_rn(fin, a0);
    }
    return fin;
}

// The same order (n < 512) evaluated by a group of 8 consecutive lanes of a warp: lane l8 owns vector lane l8 of ATen's
// accumulators, so the eight per-lane chains run side by side and only the final fold (scalar tail, then lanes 0..7
// in order) is serial: ~20 dependent adds for n = 39 instead of 71.  All 8 lanes of the group must call; every lane
// returns the result.  `mask` names the calling lanes of the warp (whole groups).
template <typename Load>
__device__ __forceinline__ float aten_row_sum_lanes8(Load ld, int n, int l8, unsigned mask) {
    if (n < 8) return aten_row_sum_small(ld, n);
    const int vec_size = n >> 3, size_ilp = vec_size >> 2;
    float fin = 0.f;
    for (int i = vec_size << 3; i < n; ++i) fin = __fadd_rn(fin, ld(i));
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    for (int i = 0; i < size_ilp; ++i) {
        a0 = __fadd_rn(a0, ld(i * 32 + l8));
        a1 = __fadd_rn(a1, ld(i * 32 + 8 + l8));
        a2 = __fadd_rn(a2, ld(i * 32 + 16 + l8));
        a3 = __fadd_rn(a3, ld(i * 32 + 24 + l8));
    }
    for (int v = size_ilp << 2; v < vec_size; ++v) a0 = __fadd_rn(a0, ld(v * 8 + l8));
    a0 = __fadd_rn(a0, a1); a0 = __fadd_rn(a0, a2); a0 = __fadd_rn(a0, a3);
#pragma unroll
    for (int l = 0; l < 8; ++l) fin = __fadd_rn(fin, __shfl_sync(mask, a0, l, 8));
    return fin;
}

// The same order evaluated by ONE WARP for any n (cascade included): lane a = t*8+l owns
// accumulator (ilp t, vector lane l) and walks elements a, a+32, a+64, ...  Result in every lane.
__device__ __forceinline__ float aten_row_sum_warp(const float* __restrict__ x, int64_t n) {
    const int lane = threadIdx.x & 31;
    if (n < 8) {
        float r = 0.f;
        if (lane == 0) r = aten_row_sum_small([&](int i) { return x[i]; }, (int)n);
        return __shfl_sync(0xffffffffu, r, 0);
    }
    const int64_t vec_size = n >> 3, size_ilp = vec_size >> 2;
    int lp = 0;
    while (((int64_t)1 << lp) < size_ilp) ++lp;
    lp >>= 2;
    const int level_power = lp > 4 ? lp : 4;
    const int64_t level_step = (int64_t)1 << level_power, level_mask = level_step - 1;
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
    int64_t i = 0;
    while (i + level_step <= size_ilp) {
        for (int64_t j = 0; j < level_step; ++j, ++i) acc0 = __fadd_rn(acc0, x[i * 32 + lane]);
        // cascade (uniform control flow: i is warp-uniform)
        acc1 = __fadd_rn(acc1, acc0); acc0 = 0.f;
        if ((i & (level_mask << level_power)) == 0) {
            acc2 = __fadd_rn(acc2, acc1); acc1 = 0.f;
            if ((i & (level_mask << (2 * level_power))) == 0) { acc3 = __fadd_rn(acc3, acc2); acc2 = 0.f; }
        }
    }
    for (; i < size_ilp; ++i) acc0 = __fadd_rn(acc0, x[i * 32 + lane]);
    acc0 = __fadd_rn(acc0, acc1); acc0 = __fadd_rn(acc0, acc2); acc0 = __fadd_rn(acc0, acc3);
    // left-over vectors go to ilp accumulator 0 (lanes 0..7)
    if (lane < 8)
        for (int64_t v = size_ilp << 2; v < vec_size; ++v) acc0 = __fadd_rn(acc0, x[v * 8 + lane]);
    // fold ilp accumulators: ((a0 + a1) + a2) + a3 per vector lane
    float t1 = __shfl_down_sync(0xffffffffu, acc0, 8);
    float t2 = __shfl_down_sync(0xffffffffu, acc0, 16);
    float t3 = __shfl_down_sync(0xffffffffu, acc0, 24);
    float folded = __fadd_rn(__fadd_rn(__fadd_rn(acc0, t1), t2), t3);  // valid in lanes 0..7
    float fin = 0.f;
    for (int64_t k = vec_size << 3; k < n; ++k) fin = __fadd_rn(fin, x[k]);  // scalar tail (uniform)
#pragma unroll
    for (int l = 0; l < 8; ++l) fin = __fadd_rn(fin, __shfl_sync(0xffffffffu, folded, l));
    return fin;
}

}  // namespace fmb
