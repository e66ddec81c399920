// mlp.cu -- the DeepFM / NFM tower on the Bi-Interaction vector, forward and backward, fp32 SIMT.
//
// Replaces `hidden_layers[i]` + relu + autograd (models/models_online_deep/deepfm_adam.py:79-89,
// nfm_adam.py:78-88, deepfm_onn.py:88-102; SURVEY.md 8a A4/A5/A7).  Every contraction accumulates
// its index LEFT TO RIGHT with one fused multiply-add per term, exactly like oracle/fm_oracle.c, so
// this path is bit-comparable with the oracle.  It is the path used where the tower is not a real
// dense contraction (H=10, B=1..2500: the reference's own configuration, main_experiment.py:50-54)
// and the fp32-exact fallback of the tensor-core path for large B*H.
//
// One generic tiled kernel: C[m][n] = epilogue( sum_k A(m,k) * B(k,n) ), 64x64x16 tiles, 4x4
// outputs per thread, operands addressed through (row, col) strides so NT / TN / NN all map onto it.
#include "fmb_common.cuh"
#include <cstdlib>

namespace {

enum { EPI_NONE = 0, EPI_BIAS_RELU = 1, EPI_MASK = 2 };

struct GemmParams {
    const float* A; int64_t sam, sak;   // A(m,k) = A[m*sam + k*sak]
    const float* B; int64_t sbk, sbn;   // B(k,n) = B[k*sbk + n*sbn]
    float* C; int64_t scm;              // C[m*scm + n]
    int M, N, K;
    int epi;
    const float* bias;                  // EPI_BIAS_RELU: [N]
    const float* mask; int64_t smm;     // EPI_MASK: keep where mask[m*smm + n] > 0
    float* colsum;                      // optional: colsum[m] = sum_k A(m,k) (plain adds, k ascending)
    float* rowsum;                      // optional (EPI_BIAS_RELU, N <= 64.. any): not used
};

constexpr int TM = 64, TN = 64, TK = 16;

__global__ void __launch_bounds__(256) gemm_kernel(GemmParams p) {
    __shared__ float As[TK][TM + 4];
    __shared__ float Bs[TK][TN + 4];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float csum[4] = {0.f, 0.f, 0.f, 0.f};
    const bool do_colsum = p.colsum && blockIdx.x == 0 && tx == 0;
    const bool a_kcontig = (p.sak == 1), b_kcontig = (p.sbk == 1);
    for (int k0 = 0; k0 < p.K; k0 += TK) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const int e = t + 256 * r;
            int kk, mm;
            if (a_kcontig) { kk = e & 15; mm = e >> 4; } else { mm = e & 63; kk = e >> 6; }
            const int gm = m0 + mm, gk = k0 + kk;
            As[kk][mm] = (gm < p.M && gk < p.K) ? p.A[gm * p.sam + gk * p.sak] : 0.f;
            int kb, nn;
            if (b_kcontig) { kb = e & 15; nn = e >> 4; } else { nn = e & 63; kb = e >> 6; }
            const int gn = n0 + nn, gkb = k0 + kb;
            Bs[kb][nn] = (gn < p.N && gkb < p.K) ? p.B[gkb * p.sbk + gn * p.sbn] : 0.f;
        }
        __syncthreads();
        const int klim = min(TK, p.K - k0);
        for (int kk = 0; kk < klim; ++kk) {
            const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = __fmaf_rn(a[i], b[j], acc[i][j]);
            if (do_colsum) {
#pragma unroll
                for (int i = 0; i < 4; ++i) csum[i] = __fadd_rn(csum[i], a[i]);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= p.M) continue;
        if (do_colsum) p.colsum[gm] = csum[i];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= p.N) continue;
            float v = acc[i][j];
            if (p.epi == EPI_BIAS_RELU) { v = __fadd_rn(v, p.bias[gn]); v = v > 0.f ? v : 0.f; }
            else if (p.epi == EPI_MASK) { v = p.mask[gm * p.smm + gn] > 0.f ? v : 0.f; }
            p.C[gm * p.scm + gn] = v;
        }
    }
}

}  // namespace

int fmb_gemm_tc_launch(const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbk, int64_t sbn, float* C,
                       int64_t scm, int M, int N, int K, int epi, const float* bias, const float* mask, int64_t smm,
                       float* colsum, cudaStream_t stream);
static int g_use_tc = 1;
// Products of at least 2^24 multiply-adds (every product of the cfg4 tower, including the K = batch weight
// gradient of the k-wide first layer) go to the tcgen05 3xTF32 kernel (gemm_tc.cu); smaller ones -- every
// shape of the reference's own scripts (H = 10, B <= 2500, main_experiment.py:50-54) -- stay on the exact SIMT kernel.
constexpr int TC_THRESHOLD_LOG2 = 24;
FMB_API void fmb_set_tensor_cores(int on) { g_use_tc = on ? 1 : 0; }
FMB_API int fmb_tensor_cores_enabled(void) { return g_use_tc; }
FMB_API int fmb_tensor_core_threshold_log2(void) { return TC_THRESHOLD_LOG2; }

namespace {

static int launch_gemm(const GemmParams& p, cudaStream_t stream) {
    if (g_use_tc && (int64_t)p.M * p.N * p.K >= ((int64_t)1 << TC_THRESHOLD_LOG2))
        return fmb_gemm_tc_launch(p.A, p.sam, p.sak, p.B, p.sbk, p.sbn, p.C, p.scm, p.M, p.N, p.K, p.epi, p.bias, p.mask,
                                  p.smm, p.colsum, stream);
    dim3 grid((p.N + TN - 1) / TN, (p.M + TM - 1) / TM);
    gemm_kernel<<<grid, 256, 0, stream>>>(p);
    return 0;
}

// head[b] = sum_j act[b][j] in ATen's row order, one warp per sample
__global__ void head_sum_kernel(const float* __restrict__ act, int B, int H, float* __restrict__ head) {
    const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= B) return;
    const float s = fmb::aten_row_sum_warp(act + (size_t)b * H, H);
    if ((threadIdx.x & 31) == 0) head[b] = s;
}

// gp[b][o] = act[b][o] > 0 ? gtop[b] : 0   (threshold_backward of the broadcast head gradient)
__global__ void top_grad_kernel(const float* __restrict__ act, const float* __restrict__ gtop, int B, int H,
                                float* __restrict__ gp) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)B * H) return;
    gp[i] = act[i] > 0.f ? gtop[i / H] : 0.f;
}

// hedge single pass: gp[b][o] = act[b][o] > 0 ? alpha[i] * gtop[b] : 0  (init != 0: overwrite; else add to gp)
__global__ void hedge_inject_kernel(const float* __restrict__ act, const float* __restrict__ gtop,
                                    const float* __restrict__ alpha, int i, int B, int H, int init, float* __restrict__ gp) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)B * H) return;
    const float t = act[e] > 0.f ? __fmul_rn(alpha[i], gtop[e / H]) : 0.f;
    gp[e] = init ? t : __fadd_rn(gp[e], t);
}

}  // namespace

static size_t mlp_w_off(int k, int H, int l) {
    return l == 0 ? 0 : (size_t)H * k + H + (size_t)(l - 1) * ((size_t)H * H + H);
}

FMB_API int64_t fmb_mlp_numel(int k, int L, int H) { return L > 0 ? (int64_t)mlp_w_off(k, H, L) : 0; }

// A4: x_0 = relu(bi W_0^T + c_0), x_l = relu(x_{l-1} W_l^T + c_l)   (deepfm_adam.py:82-86)
//   bi [B,ldbi] (row pitch ldbi >= k), mlp = W0[H,k] c0[H] W1[H,H] c1[H] ..., act [L,B,H],
//   head [L,B] = sum_j act[l][b][j] (nullable).
FMB_API int fmb_mlp_forward(const float* bi, int ldbi, const float* mlp, int B, int k, int L, int H, float* act,
                            float* head, cudaStream_t stream) {
    FMB_CHECK_ARG(bi && mlp && act && B > 0 && k > 0 && L > 0 && H > 0, "fmb_mlp_forward: bad arguments");
    for (int l = 0; l < L; ++l) {
        const int nin = l == 0 ? k : H;
        GemmParams p = {};
        p.A = l == 0 ? bi : act + (size_t)(l - 1) * B * H; p.sam = l == 0 ? ldbi : H; p.sak = 1;
        p.B = mlp + mlp_w_off(k, H, l); p.sbk = 1; p.sbn = nin;  // B(k,n) = W[n][k]
        p.C = act + (size_t)l * B * H; p.scm = H;
        p.M = B; p.N = H; p.K = nin; p.epi = EPI_BIAS_RELU; p.bias = mlp + mlp_w_off(k, H, l) + (size_t)H * nin;
        { const int rcg = launch_gemm(p, stream); if (rcg) return rcg; }
        if (head) head_sum_kernel<<<(B + 7) / 8, 256, 0, stream>>>(p.C, B, H, head + (size_t)l * B);
    }
    FMB_CHECK_LAUNCH("fmb_mlp_forward");
    return FMB_OK;
}

FMB_API size_t fmb_mlp_bwd_workspace_bytes(int B, int H) { return (size_t)2 * B * H * sizeof(float) + 256; }

// backward of head `top` (gradient gtop[b] on sum_j act[top][b][j]) through layers top..0.
//   gmlp: same layout as mlp, layers 0..top are overwritten (layers above `top` are left untouched)
//   gbi [B,ldgbi] (nullable): gradient on the Bi-Interaction vector.
FMB_API int fmb_mlp_backward(const float* bi, int ldbi, const float* mlp, const float* act, const float* gtop,
                             int top, int B, int k, int L, int H, float* gmlp, float* gbi, int ldgbi, void* ws,
                             size_t ws_bytes, cudaStream_t stream) {
    FMB_CHECK_ARG(bi && mlp && act && gtop && gmlp && ws, "fmb_mlp_backward: null pointer");
    FMB_CHECK_ARG(top >= 0 && top < L, "fmb_mlp_backward: top=%d out of range", top);
    if (ws_bytes < fmb_mlp_bwd_workspace_bytes(B, H)) { fmb_set_error("fmb_mlp_backward: workspace too small"); return FMB_ERR_WS; }
    float* gpA = (float*)ws;
    float* gpB = gpA + (size_t)B * H;
    const int64_t n = (int64_t)B * H;
    top_grad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(act + (size_t)top * B * H, gtop, B, H, gpA);
    float* gp = gpA;
    float* gnext = gpB;
    for (int l = top; l >= 0; --l) {
        const int nin = l == 0 ? k : H;
        const float* xin = l == 0 ? bi : act + (size_t)(l - 1) * B * H;
        const int64_t ldx = l == 0 ? ldbi : H;
        const float* W = mlp + mlp_w_off(k, H, l);
        // gW[o][i] = sum_b gp[b][o] * xin[b][i]  and  gc[o] = sum_b gp[b][o]
        GemmParams q = {};
        q.A = gp; q.sam = 1; q.sak = H;          // A(m=o, k=b)
        q.B = xin; q.sbk = ldx; q.sbn = 1;       // B(k=b, n=i)
        q.C = gmlp + mlp_w_off(k, H, l); q.scm = nin;
        q.M = H; q.N = nin; q.K = B; q.epi = EPI_NONE;
        q.colsum = gmlp + mlp_w_off(k, H, l) + (size_t)H * nin;
        { const int rcg = launch_gemm(q, stream); if (rcg) return rcg; }
        // gx[b][i] = sum_o gp[b][o] * W[o][i]  (masked by relu of the layer below)
        if (l > 0 || gbi) {
            GemmParams r = {};
            r.A = gp; r.sam = H; r.sak = 1;      // A(m=b, k=o)
            r.B = W; r.sbk = nin; r.sbn = 1;     // B(k=o, n=i)
            r.M = B; r.N = nin; r.K = H;
            if (l > 0) { r.C = gnext; r.scm = H; r.epi = EPI_MASK; r.mask = act + (size_t)(l - 1) * B * H; r.smm = H; }
            else { r.C = gbi; r.scm = ldgbi; r.epi = EPI_NONE; }
            { const int rcg = launch_gemm(r, stream); if (rcg) return rcg; }
        }
        float* tmp = gp; gp = gnext; gnext = tmp;
    }
    FMB_CHECK_LAUNCH("fmb_mlp_backward");
    return FMB_OK;
}

// A7 in ONE backward pass (SURVEY.md A7 "equivalent single pass"): acc = sum_{i >= l} alpha_i dL_i/dW_l for every layer l,
// obtained by injecting alpha_i * dL_i/d(head_i) at every head on the way down instead of running one backward pass per head
// (deepfm_onn.py:127-141 runs L passes; hedge_accumulate adds them).  Same mathematics, different rounding (the L-pass form
// rounds each alpha_i * grad_i separately): used for towers whose products run on the tensor cores, where the per-pass
// results are themselves within tolerance, not bit-exact; the reference's own shapes (H = 10) keep the L-pass form.
//   gtop_all [L,B]: d(BCELoss_i)/d(pre-sigmoid logit of head i) (fmb_hedge_head_grad), alpha [L] (device), acc: mlp layout.
FMB_API int fmb_mlp_backward_hedge(const float* bi, int ldbi, const float* mlp, const float* act, const float* gtop_all,
                                   const float* alpha, int B, int k, int L, int H, float* acc, void* ws, size_t ws_bytes,
                                   cudaStream_t stream) {
    FMB_CHECK_ARG(bi && mlp && act && gtop_all && alpha && acc && ws && L > 0, "fmb_mlp_backward_hedge: bad arguments");
    if (ws_bytes < fmb_mlp_bwd_workspace_bytes(B, H)) { fmb_set_error("fmb_mlp_backward_hedge: workspace too small"); return FMB_ERR_WS; }
    float* gp = (float*)ws;
    float* gnext = gp + (size_t)B * H;
    const int64_t n = (int64_t)B * H;
    const unsigned grid = (unsigned)((n + 255) / 256);
    hedge_inject_kernel<<<grid, 256, 0, stream>>>(act + (size_t)(L - 1) * B * H, gtop_all + (size_t)(L - 1) * B, alpha, L - 1, B, H, 1, gp);
    for (int l = L - 1; l >= 0; --l) {
        const int nin = l == 0 ? k : H;
        const float* xin = l == 0 ? bi : act + (size_t)(l - 1) * B * H;
        const int64_t ldx = l == 0 ? ldbi : H;
        GemmParams q = {};
        q.A = gp; q.sam = 1; q.sak = H;
        q.B = xin; q.sbk = ldx; q.sbn = 1;
        q.C = acc + mlp_w_off(k, H, l); q.scm = nin;
        q.M = H; q.N = nin; q.K = B; q.epi = EPI_NONE;
        q.colsum = acc + mlp_w_off(k, H, l) + (size_t)H * nin;
        { const int rcg = launch_gemm(q, stream); if (rcg) return rcg; }
        if (l > 0) {
            GemmParams r = {};
            r.A = gp; r.sam = H; r.sak = 1;
            r.B = mlp + mlp_w_off(k, H, l); r.sbk = nin; r.sbn = 1;
            r.M = B; r.N = nin; r.K = H;
            r.C = gnext; r.scm = H; r.epi = EPI_MASK; r.mask = act + (size_t)(l - 1) * B * H; r.smm = H;
            { const int rcg = launch_gemm(r, stream); if (rcg) return rcg; }
            hedge_inject_kernel<<<grid, 256, 0, stream>>>(act + (size_t)(l - 1) * B * H, gtop_all + (size_t)(l - 1) * B, alpha, l - 1, B, H, 0, gnext);
            float* tmp = gp; gp = gnext; gnext = tmp;
        }
    }
    FMB_CHECK_LAUNCH("fmb_mlp_backward_hedge");
    return FMB_OK;
}
