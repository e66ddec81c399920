// afm.cu -- Attentional Factorization Machine (SURVEY.md 8f.3; BASELINE.json north_star lists AFM among the offline models).
//
// The reference's models/models_online_deep/afm_adam.py cannot run (a float is passed to .view at :67,69; undefined
// attributes at :121-123,167), so this implements the model of the AFM paper (Xiao et al., IJCAI 2017, eq. 8) with the
// reference's parameter set (afm_adam.py:34-41) and the family's update rule; the definition it is checked against is
// oracle/afm.py (plain PyTorch autograd).
//     e_i = x_i V_i;  z_ij = e_i (.) e_j (i < j);  a'_ij = H . relu(W z_ij + c);  a = softmax_pairs(a');
//     logit = bias + sum_i x_i w_i + sum_ij a_ij (P . z_ij);  loss = mean BCE-with-logits
// One CTA per sample: pass 1 scores every pair, a block-wide softmax, pass 2 back-propagates through attention and
// projection, pass 3 folds the pair gradients back onto the fields in a fixed order (no float atomics anywhere).  The
// per-entry embedding gradients are staged at their sorted positions and summed / applied by the run kernel of
// fm_backward.cu (min_run = 1), exactly like the FM step; the dense parameters' per-sample gradients are summed over the
// batch in a fixed order by afm_dense_update_kernel.
#include "fmb_common.cuh"

extern "C" size_t fmb_bwd_workspace_bytes(int64_t, int);

namespace {

constexpr int AT = 128;       // threads per sample
constexpr int MAXK = 16, MAXA = 8;

struct AfmParams {
    const int32_t* ids; const float* xv; const float* y; const uint32_t* posflag;
    const float* table; const float* bias;
    const float* W; const float* c; const float* H; const float* P;   // attention_linear.weight [A,k], .bias [A], H [A], P [k]
    const unsigned char* pair_i; const unsigned char* pair_j;          // [NP]
    int B, F, k, A, NP, rowp, loss_kind;
    float* z_out;        // [B] logits (nullable)
    float* delta;        // [B]   (nullable: forward only)
    float* lossv;        // [B]
    float* dense_g;      // [B][PD] per-sample gradients of W | c | H | P
    float* G; int64_t Npad;   // staged per-entry gradients (component-major, sorted positions)
};

__device__ __forceinline__ float block_reduce_sum(float v, float* red) {
    // fixed-order tree over the AT threads: deterministic
    const int tid = threadIdx.x;
    red[tid] = v;
    __syncthreads();
    for (int o = AT / 2; o > 0; o >>= 1) { if (tid < o) red[tid] = __fadd_rn(red[tid], red[tid + o]); __syncthreads(); }
    const float r = red[0];
    __syncthreads();
    return r;
}
__device__ __forceinline__ float block_reduce_max(float v, float* red) {
    const int tid = threadIdx.x;
    red[tid] = v;
    __syncthreads();
    for (int o = AT / 2; o > 0; o >>= 1) { if (tid < o) red[tid] = fmaxf(red[tid], red[tid + o]); __syncthreads(); }
    const float r = red[0];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(AT) afm_kernel(AfmParams p) {
    extern __shared__ __align__(16) float sm[];
    const int F = p.F, k = p.k, A = p.A, NP = p.NP, tid = threadIdx.x, b = blockIdx.x;
    float* e_s = sm;                 // [F][k]
    float* x_s = e_s + F * k;        // [F]
    float* att = x_s + F;            // [NP] a' then a
    float* sc = att + NP;            // [NP] P . z
    float* dz = sc + NP;             // [NP][k]
    float* red = dz + (size_t)NP * k;   // [AT]
    float* par = red + AT;           // W [A*k] | c [A] | H [A] | P [k]
    float* de = par + A * k + 2 * A + k;   // [F][k]
    __shared__ float first_s, delta_s;
    for (int i = tid; i < A * k; i += AT) par[i] = p.W[i];
    if (tid < A) { par[A * k + tid] = p.c[tid]; par[A * k + A + tid] = p.H[tid]; }
    if (tid < k) par[A * k + 2 * A + tid] = p.P[tid];
    const float* Ws = par; const float* cs = par + A * k; const float* Hs = cs + A; const float* Ps = Hs + A;
    for (int f = tid; f < F; f += AT) x_s[f] = p.xv ? p.xv[(size_t)b * F + f] : 1.0f;
    __syncthreads();
    for (int i = tid; i < F * k; i += AT) {
        const int f = i / k, j = i - f * k;
        e_s[i] = __fmul_rn(p.table[(size_t)p.ids[(size_t)b * F + f] * p.rowp + j], x_s[f]);
    }
    if (tid == 0) {
        float s = 0.f;
        for (int f = 0; f < F; ++f) s = __fadd_rn(s, __fmul_rn(p.table[(size_t)p.ids[(size_t)b * F + f] * p.rowp + k], x_s[f]));
        first_s = s;
    }
    __syncthreads();
    // pass 1: pair scores
    float lmax = -3.4e38f;
    for (int q = tid; q < NP; q += AT) {
        const float* ei = e_s + p.pair_i[q] * k; const float* ej = e_s + p.pair_j[q] * k;
        float z[MAXK], a = 0.f, s = 0.f;
#pragma unroll
        for (int j = 0; j < MAXK; ++j) if (j < k) { z[j] = __fmul_rn(ei[j], ej[j]); s = __fmaf_rn(Ps[j], z[j], s); }
        for (int t = 0; t < A; ++t) {
            float u = cs[t];
#pragma unroll
            for (int j = 0; j < MAXK; ++j) if (j < k) u = __fmaf_rn(Ws[t * k + j], z[j], u);
            a = __fmaf_rn(Hs[t], fmaxf(u, 0.f), a);
        }
        att[q] = a; sc[q] = s;
        lmax = fmaxf(lmax, a);
    }
    const float mx = block_reduce_max(lmax, red);
    float lsum = 0.f;
    for (int q = tid; q < NP; q += AT) { const float ex = __expf(__fsub_rn(att[q], mx)); att[q] = ex; lsum = __fadd_rn(lsum, ex); }
    const float tot = block_reduce_sum(lsum, red);
    float lz = 0.f;
    for (int q = tid; q < NP; q += AT) { const float a = __fdiv_rn(att[q], tot); att[q] = a; lz = __fmaf_rn(a, sc[q], lz); }
    const float z2 = block_reduce_sum(lz, red);
    if (tid == 0) {
        const float zl = __fadd_rn(__fadd_rn(p.bias[0], first_s), z2);
        if (p.z_out) p.z_out[b] = zl;
        if (p.delta) {
            float lv, d;
            fmb::bce_logits_value_grad(p.loss_kind, zl, p.y[b], b, p.B, lv, d);
            p.delta[b] = d; p.lossv[b] = lv; delta_s = d;
        }
    }
    __syncthreads();
    if (!p.delta) return;
    // pass 2: back through softmax, attention net and projection; per-thread sums of the dense gradients
    const float d = delta_s;
    const float dsoft = __fmul_rn(d, z2);        // sum_q a_q * (d * s_q)
    float gW[MAXA * MAXK], gc[MAXA], gH[MAXA], gP[MAXK];
#pragma unroll
    for (int i = 0; i < MAXA * MAXK; ++i) gW[i] = 0.f;
#pragma unroll
    for (int i = 0; i < MAXA; ++i) { gc[i] = 0.f; gH[i] = 0.f; }
#pragma unroll
    for (int i = 0; i < MAXK; ++i) gP[i] = 0.f;
    for (int q = tid; q < NP; q += AT) {
        const float* ei = e_s + p.pair_i[q] * k; const float* ej = e_s + p.pair_j[q] * k;
        const float a = att[q];
        const float da = __fmul_rn(a, __fsub_rn(__fmul_rn(d, sc[q]), dsoft));   // d loss / d a'_q
        const float ds = __fmul_rn(d, a);                                        // d loss / d (P . z_q)
        float z[MAXK], g[MAXK];
#pragma unroll
        for (int j = 0; j < MAXK; ++j) if (j < k) { z[j] = __fmul_rn(ei[j], ej[j]); g[j] = __fmul_rn(ds, Ps[j]); gP[j] = __fmaf_rn(ds, z[j], gP[j]); }
#pragma unroll
        for (int t = 0; t < MAXA; ++t) if (t < A) {
            float u = cs[t];
#pragma unroll
            for (int j = 0; j < MAXK; ++j) if (j < k) u = __fmaf_rn(Ws[t * k + j], z[j], u);
            gH[t] = __fmaf_rn(da, fmaxf(u, 0.f), gH[t]);
            if (u > 0.f) {
                const float du = __fmul_rn(da, Hs[t]);
                gc[t] = __fadd_rn(gc[t], du);
#pragma unroll
                for (int j = 0; j < MAXK; ++j) if (j < k) { gW[t * MAXK + j] = __fmaf_rn(du, z[j], gW[t * MAXK + j]); g[j] = __fmaf_rn(du, Ws[t * k + j], g[j]); }
            }
        }
#pragma unroll
        for (int j = 0; j < MAXK; ++j) if (j < k) dz[(size_t)q * k + j] = g[j];
    }
    // dense gradients of this sample: block sums in a fixed order
    float* dg = p.dense_g + (size_t)b * (A * k + 2 * A + k);
    for (int t = 0; t < A; ++t)
        for (int j = 0; j < k; ++j) { const float v = block_reduce_sum(gW[t * MAXK + j], red); if (tid == 0) dg[t * k + j] = v; }
    for (int t = 0; t < A; ++t) { const float v = block_reduce_sum(gc[t], red); if (tid == 0) dg[A * k + t] = v; }
    for (int t = 0; t < A; ++t) { const float v = block_reduce_sum(gH[t], red); if (tid == 0) dg[A * k + A + t] = v; }
    for (int j = 0; j < k; ++j) { const float v = block_reduce_sum(gP[j], red); if (tid == 0) dg[A * k + 2 * A + j] = v; }
    __syncthreads();
    // pass 3: pair gradients back onto the fields, partner fields in ascending order (fixed order: no atomics)
    for (int i = tid; i < F * k; i += AT) {
        const int f = i / k, j = i - f * k;
        float acc = 0.f;
        for (int g = 0; g < F; ++g) {
            if (g == f) continue;
            const int lo = g < f ? g : f, hi = g < f ? f : g;
            const int q = lo * F - lo * (lo + 1) / 2 + (hi - lo - 1);     // index of pair (lo, hi) in row-major upper triangle
            acc = __fmaf_rn(dz[(size_t)q * k + j], e_s[g * k + j], acc);
        }
        de[i] = acc;
    }
    __syncthreads();
    // stage d loss / d V_row = de * x and d loss / d w_row = delta * x at the entry's sorted position
    for (int i = tid; i < F * (k + 1); i += AT) {
        const int f = i / (k + 1), j = i - f * (k + 1);
        const size_t pos = p.posflag[(size_t)b * F + f] & 0x7fffffffu;
        p.G[(size_t)j * p.Npad + pos] = j < k ? __fmul_rn(de[f * k + j], x_s[f]) : __fmul_rn(d, x_s[f]);
    }
}

// sum the per-sample dense gradients over the batch (lane l adds samples l, l+32, ... in order, then the 32 lane sums are
// added in lane order) and apply the update: one warp per parameter
__global__ void afm_dense_update_kernel(const float* __restrict__ dense_g, int B, int PD, float* W, float* c, float* H,
                                        float* P, int A, int k, float lr, int mode, float* grads_out) {
    const int col = blockIdx.x, lane = threadIdx.x;
    float a = 0.f;
    for (int b = lane; b < B; b += 32) a = __fadd_rn(a, dense_g[(size_t)b * PD + col]);
    float tot = 0.f;
    for (int l = 0; l < 32; ++l) tot = __fadd_rn(tot, __shfl_sync(0xffffffffu, a, l));
    if (lane == 0) {
        if (grads_out) grads_out[col] = tot;
        float* dst = col < A * k ? W + col : col < A * k + A ? c + (col - A * k) : col < A * k + 2 * A ? H + (col - A * k - A)
                                                                                                      : P + (col - A * k - 2 * A);
        *dst = fmb::apply_update(*dst, tot, lr, mode);
    }
}

}  // namespace

FMB_API size_t fmb_afm_dense_floats(int k, int A) { return (size_t)A * k + 2 * A + k; }

// AFM forward (+ backward when delta != NULL): logits z [B] (nullable), delta / lossv [B], per-sample dense gradients
// dense_g [B][A*k + 2A + k], per-entry embedding gradients staged into ws (fmb_bwd_workspace_bytes(B*F, k)) at the sorted
// positions given by posflag (fmb_pos_flags).  pair_i / pair_j [F(F-1)/2]: the field pairs in row-major upper-triangle
// order.  F <= 64, k <= 16, A <= 8.
FMB_API int fmb_afm_step(const int32_t* ids, const float* xv, const float* y, const uint32_t* posflag, const float* table,
                         const float* bias, const float* W, const float* c, const float* H, const float* P,
                         const unsigned char* pair_i, const unsigned char* pair_j, int B, int F, int k, int A,
                         int loss_kind, float* z_out, float* delta, float* lossv, float* dense_g, void* ws,
                         size_t ws_bytes, cudaStream_t stream) {
    FMB_CHECK_ARG(ids && table && bias && W && c && H && P && pair_i && pair_j, "fmb_afm_step: null pointer");
    FMB_CHECK_ARG(B > 0 && F >= 2 && F <= 64 && k > 0 && k <= MAXK && A > 0 && A <= MAXA, "fmb_afm_step: need 2 <= F <= 64, k <= 16, A <= 8");
    FMB_CHECK_ARG(!delta || (y && posflag && lossv && dense_g && ws), "fmb_afm_step: backward needs y, posflag, lossv, dense_g, ws");
    const int64_t N = (int64_t)B * F;
    if (delta && ws_bytes < fmb_bwd_workspace_bytes(N, k)) { fmb_set_error("fmb_afm_step: workspace too small"); return FMB_ERR_WS; }
    AfmParams p;
    p.ids = ids; p.xv = xv; p.y = y; p.posflag = posflag; p.table = table; p.bias = bias;
    p.W = W; p.c = c; p.H = H; p.P = P; p.pair_i = pair_i; p.pair_j = pair_j;
    p.B = B; p.F = F; p.k = k; p.A = A; p.NP = F * (F - 1) / 2; p.rowp = fmb_round_up(k + 1, 16); p.loss_kind = loss_kind;
    p.z_out = z_out; p.delta = delta; p.lossv = lossv; p.dense_g = dense_g;
    p.G = (float*)ws; p.Npad = (N + 3) / 4 * 4 + 64;
    const size_t smem = sizeof(float) * ((size_t)2 * F * k + F + 2 * p.NP + (size_t)p.NP * k + AT + A * k + 2 * A + k);
    FMB_CHECK_ARG(smem <= 200 * 1024, "fmb_afm_step: F*F*k too large for one CTA");
    static bool attr = false;
    if (!attr) { cudaFuncSetAttribute(afm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); attr = true; }
    afm_kernel<<<B, AT, smem, stream>>>(p);
    FMB_CHECK_LAUNCH("afm_kernel");
    return FMB_OK;
}

// batch sum of the dense gradients + update of attention_linear / H / P; grads_out [A*k + 2A + k] nullable (tests)
FMB_API int fmb_afm_dense_update(const float* dense_g, int B, int k, int A, float* W, float* c, float* H, float* P, float lr,
                                 int mode, float* grads_out, cudaStream_t stream) {
    FMB_CHECK_ARG(dense_g && W && c && H && P && B > 0, "fmb_afm_dense_update: bad arguments");
    FMB_CHECK_ARG(mode != 3, "fmb_afm_dense_update: update mode 3 (Adagrad) is not supported by AFM");
    const int PD = A * k + 2 * A + k;
    afm_dense_update_kernel<<<PD, 32, 0, stream>>>(dense_g, B, PD, W, c, H, P, A, k, lr, mode, grads_out);
    FMB_CHECK_LAUNCH("afm_dense_update_kernel");
    return FMB_OK;
}
