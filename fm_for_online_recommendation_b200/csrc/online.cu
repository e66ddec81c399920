// online.cu -- per-example online mode as ONE persistent kernel.
//
// Replaces the reference's `run_experiment` loop (models/models_online_deep/fm_adam.py:90-119, identical
// in the five classes; SURVEY.md 8a A8): for every example, strictly in order, `predict` and then `fit`
// with batch size 1 -- a fresh-Adam sign step on everything for the Adam family
// (fm_adam.py:71-82, deepfm_adam.py:106-117, nfm_adam.py:105-116) or a hedge-backprop step on the tower
// (deepfm_onn.py:109-154, nfm_onn.py:111-156).  The reference pays two host round trips and a dense
// Adam step over all 11 M parameters per example; here one CTA walks the stream without leaving the
// device, so example i+1 sees exactly the state example i wrote (no silent mini-batching).
// Arithmetic is the batch path's, specialised to B = 1 (same op order as oracle/fm_oracle.c).
// Latency-bound by construction: reported as examples/s, no roofline fraction claimed.
#include "fmb_common.cuh"

namespace {

constexpr int OT = 256;

struct OnlineParams {
    int kind;  // 0 FMAdam, 1 DeepFMAdam, 2 NFMAdam, 3 DeepFMOnn, 4 NFMOnn
    int N, F, k, L, H, rowp, kp4, cu, ql_log;
    const int32_t* ids;  // [N,F] global row ids
    const float* xv;     // [N,F] or NULL
    const float* y;      // [N]
    float* table;
    float* bias;
    float* mlp;
    float* alpha;
    float* acc;          // [n_mlp] hedge accumulator (ONN)
    float lr, hb, hs;
    int mode;
    float* ada_sums;     // mode 3 (Adagrad): sums of the table [R][rowp], the bias [1] and the tower [n_mlp];
    float* ada_bias;     // mode 4 (SparseAdam): m and v of the table [R][2][rowp], the bias [2] and the tower [2][n_mlp]
    float* ada_mlp;
    union {
        float eps;                // mode 3
        const float* sa_steps;    // mode 4: [4 + 5N] = (1-b1, b2, 1-b2, eps), then the five scalars of every example
    };
    uint8_t* preds;      // [N]
    int64_t* conf;       // [4] tp, fp, tn, fn
};

__device__ __forceinline__ size_t w_off(int k, int H, int l) {
    return l == 0 ? 0 : (size_t)H * k + H + (size_t)(l - 1) * ((size_t)H * H + H);
}

// The Adam family's update of one parameter of group grp (0 table, 1 bias, 2 tower) at example n.  The kernel is
// instantiated once per kind of state SK, so that the other modes' kernel stays as it is: 0 none, 1 Adagrad (mode 3:
// the sum *s), 2 SparseAdam on the table and Adam on the bias and the tower (mode 4: m at s[0], v one sub-row / one
// group further; the step's scalars from the host-filled table p.sa_steps).
template <int SK>
__device__ __forceinline__ float online_update(const OnlineParams& p, float w, float g, float* s, int grp, int n) {
    if (SK == 1) {
        float sv = *s;
        const float o = fmb::adagrad_update(w, g, sv, p.lr, p.eps);
        *s = sv;
        return o;
    }
    if (SK == 2) {
        const float* c = p.sa_steps;
        const float* st = c + 4 + (size_t)5 * n;
        const size_t vo = grp == 0 ? (size_t)p.rowp : grp == 1 ? 1 : w_off(p.k, p.H, p.L);
        float m = s[0], v = s[vo], o;
        if (grp == 0) {
            const fmb::SparseAdamState a = {nullptr, c[0], c[2], c[3], st[0]};
            o = fmb::sparse_adam_update(w, g, m, v, a);
        } else {
            const fmb::AdamState a = {nullptr, c[0], c[1], c[2], c[3], st[grp == 1 ? 1 : 3], st[grp == 1 ? 2 : 4]};
            o = fmb::adam_update(w, g, m, v, a);
        }
        s[0] = m; s[vo] = v;
        return o;
    }
    return fmb::apply_update(w, g, p.lr, p.mode);
}

template <int SK>
__global__ void __launch_bounds__(OT) online_deep_kernel(OnlineParams p) {
    extern __shared__ __align__(16) float sm[];
    const int F = p.F, k = p.k, L = p.L, H = p.H, rp = p.cu * 4;
    float* rows = sm;                    // [F][rp]
    float* xs = rows + F * rp;           // [F]
    float* first = xs + F;               // [F]
    float* Sv = first + F;               // [k]
    float* bi = Sv + k;                  // [k]
    float* act = bi + k;                 // [L][H]
    float* gp = act + L * H;             // [max(H,k)]
    float* gx = gp + max(H, k);          // [max(H,k)]
    float* gbi = gx + max(H, k);         // [k]
    float* head = gbi + k;               // [L]
    float* pl = head + L;                // [L]
    float* sc = pl + L;                  // scalars: 0 sf, 1 sb, 2 zfm, 3 base, 4 z, 5 delta, 6 du
    const bool is_onn = p.kind >= 3, is_nfm = (p.kind == 2 || p.kind == 4), has_mlp = p.kind != 0;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int64_t tp = 0, fp = 0, tn = 0, fn = 0;

    for (int n = 0; n < p.N; ++n) {
        const int32_t* id = p.ids + (size_t)n * F;
        // ---- gather the F rows of this example (old values: used by forward AND backward)
        {
            const int q = tid & ((1 << p.ql_log) - 1);
            if (q < p.cu)
                for (int f = tid >> p.ql_log; f < F; f += OT >> p.ql_log)
                    *reinterpret_cast<float4*>(rows + f * rp + q * 4) =
                        *reinterpret_cast<const float4*>(p.table + (size_t)id[f] * p.rowp + q * 4);
            for (int f = tid; f < F; f += OT) xs[f] = p.xv ? p.xv[(size_t)n * F + f] : 1.0f;
        }
        __syncthreads();
        // ---- A1-A3
        for (int j = tid; j < k + F; j += OT) {
            if (j < k) {
                float S = 0.f, Q = 0.f;
                for (int f = 0; f < F; ++f) {
                    const float e = __fmul_rn(rows[f * rp + j], xs[f]);
                    S = __fadd_rn(S, e);
                    Q = __fadd_rn(Q, __fmul_rn(e, e));
                }
                Sv[j] = S;
                bi[j] = __fmul_rn(__fsub_rn(__fmul_rn(S, S), Q), 0.5f);
            } else {
                const int f = j - k;
                first[f] = __fmul_rn(rows[f * rp + k], xs[f]);
            }
        }
        __syncthreads();
        if (tid == 0) {
            const float sf = fmb::aten_row_sum_small([&](int f) { return first[f]; }, F);
            const float sb = fmb::aten_row_sum_small([&](int j) { return bi[j]; }, k);
            const float b0 = p.bias[0];
            sc[0] = sf; sc[1] = sb;
            sc[2] = __fadd_rn(__fadd_rn(sf, sb), b0);
            sc[3] = is_nfm ? __fadd_rn(sf, b0) : sc[2];
            sc[4] = sc[2];
        }
        __syncthreads();
        // ---- A4/A5 tower forward
        if (has_mlp) {
            for (int l = 0; l < L; ++l) {
                const int nin = l == 0 ? k : H;
                const float* xin = l == 0 ? bi : act + (l - 1) * H;
                const float* W = p.mlp + w_off(k, H, l);
                const float* c = W + (size_t)H * nin;
                for (int o = tid; o < H; o += OT) {
                    float a = 0.f;
                    for (int i = 0; i < nin; ++i) a = __fmaf_rn(xin[i], W[(size_t)o * nin + i], a);
                    a = __fadd_rn(a, c[o]);
                    act[l * H + o] = a > 0.f ? a : 0.f;
                }
                __syncthreads();
                if (warp == 0) {
                    const float hsum = fmb::aten_row_sum_warp(act + l * H, H);
                    if (lane == 0) {
                        head[l] = hsum;
                        if (is_onn) pl[l] = fmb::sigmoid_at(__fadd_rn(sc[3], hsum), 0, 1);   // B = 1: ATen's scalar path
                        else if (l == L - 1) sc[4] = __fadd_rn(sc[3], hsum);
                    }
                }
                __syncthreads();
            }
        }
        // ---- predict (fm_adam.py:84-88 / deepfm_onn.py:171-175)
        const float yy = p.y[n];
        const float zout = is_onn ? pl[L - 1] : sc[4];
        const bool pred = fmb::sigmoid_at(zout, 0, 1) > 0.5f;
        if (tid == 0) {
            p.preds[n] = pred;
            const bool pos = yy == 1.0f;
            if ((pred ? 1.0f : 0.0f) == yy) { if (pos) ++tp; else ++tn; } else { if (pos) ++fn; else ++fp; }
        }
        // ---- fit
        if (!is_onn) {
            // Adam family: FM / DeepFM use BCEWithLogits(sigmoid(z)), NFM uses BCEWithLogits(z); B = 1
            if (tid == 0) {
                const float z = sc[4];
                float in = z, pr = 0.f;
                const int kindl = (p.kind == 2) ? 0 : 1;
                if (kindl == 1) { pr = fmb::sigmoid_at(z, 0, 1); in = pr; }
                float d = __fdiv_rn(__fsub_rn(fmb::sigmoid_at(in, 0, 1), yy), 1.0f);
                if (kindl == 1) d = __fmul_rn(__fmul_rn(d, __fsub_rn(1.0f, pr)), pr);
                sc[5] = d;
            }
            __syncthreads();
            const float d = sc[5];
            if (has_mlp) {
                for (int o = tid; o < H; o += OT) gp[o] = act[(L - 1) * H + o] > 0.f ? d : 0.f;
                __syncthreads();
                for (int l = L - 1; l >= 0; --l) {
                    const int nin = l == 0 ? k : H;
                    const float* xin = l == 0 ? bi : act + (l - 1) * H;
                    float* W = p.mlp + w_off(k, H, l);
                    float* c = W + (size_t)H * nin;
                    for (int i = tid; i < nin; i += OT) {  // gradient on the layer input, old weights
                        float a = 0.f;
                        for (int o = 0; o < H; ++o) a = __fmaf_rn(gp[o], W[(size_t)o * nin + i], a);
                        gx[i] = a;
                    }
                    __syncthreads();
                    for (int q = tid; q < H * nin; q += OT) {  // fresh-Adam step on W_l (gradient = gp[o]*x[i], B = 1)
                        const int o = q / nin, i = q - o * nin;
                        W[q] = online_update<SK>(p, W[q], __fmaf_rn(gp[o], xin[i], 0.f), p.ada_mlp + w_off(k, H, l) + q, 2, n);
                    }
                    for (int o = tid; o < H; o += OT)
                        c[o] = online_update<SK>(p, c[o], __fadd_rn(0.f, gp[o]), p.ada_mlp + w_off(k, H, l) + (size_t)H * nin + o, 2, n);
                    __syncthreads();
                    if (l > 0) { for (int i = tid; i < H; i += OT) gp[i] = act[(l - 1) * H + i] > 0.f ? gx[i] : 0.f; }
                    else { for (int i = tid; i < k; i += OT) gbi[i] = gx[i]; }
                    __syncthreads();
                }
            }
            // rows: every field hits a different row, so each row has exactly one entry
            const bool use_fm2 = !is_nfm, gv = has_mlp;
            for (int it = tid; it < F * (k + 1); it += OT) {
                const int f = it / (k + 1), j = it - f * (k + 1);
                const float x = xs[f], v = rows[f * rp + j];
                float g;
                if (j < k) {
                    const float ej = __fmul_rn(v, x);
                    float a = 0.f, c = 0.f;
                    if (use_fm2) a = __fmul_rn(__fsub_rn(__fmul_rn(d, Sv[j]), __fmul_rn(d, ej)), x);
                    if (gv) c = __fmul_rn(__fsub_rn(__fmul_rn(gbi[j], Sv[j]), __fmul_rn(gbi[j], ej)), x);
                    g = (use_fm2 && gv) ? __fadd_rn(__fadd_rn(0.f, a), __fadd_rn(0.f, c)) : __fadd_rn(0.f, gv ? c : a);
                } else {
                    g = __fadd_rn(0.f, __fmul_rn(d, x));
                }
                p.table[(size_t)id[f] * p.rowp + j] = online_update<SK>(p, v, g, p.ada_sums + (size_t)id[f] * (SK == 2 ? 2 : 1) * p.rowp + j, 0, n);
            }
            if (tid == 0) p.bias[0] = online_update<SK>(p, p.bias[0], __fadd_rn(0.f, d), p.ada_bias, 1, n);
        } else {
            // hedge backpropagation, batch_size = 1: L backward passes, only the tower and alpha change
            const size_t nm = w_off(k, H, L);
            for (int i = 0; i < L; ++i) {
                if (tid == 0) {
                    const float pr = pl[i];
                    const float l1 = fmaxf(fmb::log1pf_p(-pr), -100.f), l0 = fmaxf(fmb::logf_p(pr), -100.f);
                    const float lossv = __fsub_rn(__fmul_rn(__fsub_rn(yy, 1.0f), l1), __fmul_rn(yy, l0));
                    head[i] = __fdiv_rn(__fadd_rn(0.f, lossv), 1.0f);  // mean over one element (head[] is free now)
                    const float den = fmaxf(__fmul_rn(__fsub_rn(1.0f, pr), pr), 1e-12f);
                    const float dp = __fdiv_rn(__fmul_rn(__fdiv_rn(1.0f, 1.0f), __fsub_rn(pr, yy)), den);
                    sc[6] = __fmul_rn(__fmul_rn(dp, __fsub_rn(1.0f, pr)), pr);
                }
                __syncthreads();
                const float du = sc[6], ai = p.alpha[i];
                for (int o = tid; o < H; o += OT) gp[o] = act[i * H + o] > 0.f ? du : 0.f;
                __syncthreads();
                for (int l = i; l >= 0; --l) {
                    const int nin = l == 0 ? k : H;
                    const float* xin = l == 0 ? bi : act + (l - 1) * H;
                    const float* W = p.mlp + w_off(k, H, l);
                    float* aW = p.acc + w_off(k, H, l);
                    float* ac = aW + (size_t)H * nin;
                    if (l > 0)
                        for (int j = tid; j < nin; j += OT) {
                            float a = 0.f;
                            for (int o = 0; o < H; ++o) a = __fmaf_rn(gp[o], W[(size_t)o * nin + j], a);
                            gx[j] = a;
                        }
                    for (int q = tid; q < H * nin; q += OT) {
                        const int o = q / nin, j = q - o * nin;
                        const float term = __fmul_rn(ai, __fmaf_rn(gp[o], xin[j], 0.f));
                        aW[q] = (l == i) ? term : __fadd_rn(aW[q], term);
                    }
                    for (int o = tid; o < H; o += OT) {
                        const float term = __fmul_rn(ai, __fadd_rn(0.f, gp[o]));
                        ac[o] = (l == i) ? term : __fadd_rn(ac[o], term);
                    }
                    __syncthreads();
                    if (l > 0) { for (int j = tid; j < H; j += OT) gp[j] = act[(l - 1) * H + j] > 0.f ? gx[j] : 0.f; }
                    __syncthreads();
                }
            }
            for (size_t t = tid; t < nm; t += OT) p.mlp[t] = __fsub_rn(p.mlp[t], __fmul_rn(p.lr, p.acc[t]));
            if (tid == 0) {
                const float floorv = __fdiv_rn(p.hs, (float)L);
                for (int i = 0; i < L; ++i) p.alpha[i] = fmaxf(__fmul_rn(p.alpha[i], fmb::powf_p(p.hb, head[i])), floorv);
                const float zt = fmb::aten_row_sum_small([&](int j) { return p.alpha[j]; }, L);
                for (int i = 0; i < L; ++i) p.alpha[i] = __fdiv_rn(p.alpha[i], zt);
            }
        }
        __syncthreads();
    }
    if (tid == 0) { p.conf[0] = tp; p.conf[1] = fp; p.conf[2] = tn; p.conf[3] = fn; }
}

static int ilog2_ceil(int x) { int l = 0; while ((1 << l) < x) ++l; return l; }

}  // namespace

// A8: run_experiment over N examples in one launch.  kind 0..4 = FMAdam, DeepFMAdam, NFMAdam, DeepFMOnn,
// NFMOnn; ids [N,F] global row ids, xv [N,F] or NULL, y [N]; mlp/alpha/acc may be NULL for kind 0 (acc:
// [fmb_mlp_numel] scratch, ONN only).  Outputs: preds [N] (the prediction made BEFORE fitting example i),
// conf [4] = tp, fp, tn, fn (int64).
// _ex: update mode 3 (Adagrad) of the Adam family (kinds 0-2) reads and writes the sums in `ada` (the table's, the
// bias's and, with a tower, the tower's); mode 4 (SparseAdam) takes an fmb_sparse_adam_t in the same slot whose steps_dev
// holds the scalars of the N examples' steps (fmb_sparse_adam_online_steps).  The ONN kinds' hedge step uses no optimizer
// and ignores the mode.
struct fmb_adagrad_t { float* sums; float* bias_sum; float* mlp_sums; float eps; };   // include/fmb200.h
FMB_API int fmb_online_deep_run_ex(int kind, const int32_t* ids, const float* xv, const float* y, int N, int F, int k,
                                   int L, int H, float* table, float* bias, float* mlp, float* alpha, float* acc,
                                   float lr, float hb, float hs, int mode, const fmb_adagrad_t* ada, uint8_t* preds,
                                   int64_t* conf, cudaStream_t stream) {
    FMB_CHECK_ARG(kind >= 0 && kind <= 4, "fmb_online_deep_run: unknown model kind %d", kind);
    FMB_CHECK_ARG(ids && y && table && bias && preds && conf, "fmb_online_deep_run: null pointer");
    FMB_CHECK_ARG(N > 0 && F > 0 && F < 512 && k > 0 && k <= 124, "fmb_online_deep_run: bad shape N=%d F=%d k=%d (need F < 512, k <= 124)",
                  N, F, k);
    FMB_CHECK_ARG(kind == 0 || (mlp && L > 0 && H > 0 && H < 512), "fmb_online_deep_run: tower needs mlp, 0 < H < 512");
    FMB_CHECK_ARG(kind < 3 || (alpha && acc), "fmb_online_deep_run: ONN needs alpha and acc");
    FMB_CHECK_ARG(mode != 3 || kind >= 3 || (ada && ada->sums && ada->bias_sum && (kind == 0 || ada->mlp_sums)),
                  "fmb_online_deep_run: update mode 3 needs the Adagrad state (sums of the table, the bias and the tower)");
    const fmb_sparse_adam_t* sa = mode == 4 && kind < 3 ? reinterpret_cast<const fmb_sparse_adam_t*>(ada) : nullptr;
    FMB_CHECK_ARG(mode != 4 || kind >= 3 || (sa && sa->mv && sa->bias_mv && sa->steps_dev && (kind == 0 || sa->mlp_mv)),
                  "fmb_online_deep_run: update mode 4 needs the SparseAdam state (moments of the table, the bias and the "
                  "tower, and the examples' step scalars)");
    OnlineParams p;
    p.kind = kind; p.N = N; p.F = F; p.k = k; p.L = kind == 0 ? 0 : L; p.H = kind == 0 ? 0 : H;
    p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4); p.cu = (k + 1 + 3) / 4; p.ql_log = ilog2_ceil(p.cu);
    p.ids = ids; p.xv = xv; p.y = y; p.table = table; p.bias = bias; p.mlp = mlp; p.alpha = alpha; p.acc = acc;
    p.lr = lr; p.hb = hb; p.hs = hs; p.mode = mode; p.preds = preds; p.conf = conf;
    p.ada_sums = p.ada_bias = p.ada_mlp = nullptr; p.eps = 0.f;
    if (mode == 3 && ada) { p.ada_sums = ada->sums; p.ada_bias = ada->bias_sum; p.ada_mlp = ada->mlp_sums; p.eps = ada->eps; }
    if (sa) { p.ada_sums = sa->mv; p.ada_bias = sa->bias_mv; p.ada_mlp = sa->mlp_mv; p.sa_steps = sa->steps_dev; }
    const int mx = p.H > k ? p.H : k;
    const size_t fl = (size_t)F * p.cu * 4 + 2 * F + 2 * k + (size_t)p.L * p.H + 2 * mx + k + 2 * (p.L > 0 ? p.L : 1) + 16;
    const size_t smb = fl * sizeof(float);
    FMB_CHECK_ARG(smb <= 200 * 1024, "fmb_online_deep_run: model too large for one CTA's shared memory (F=%d k=%d L=%d H=%d: %zu bytes > 200 KB)",
                  F, k, p.L, p.H, smb);
    if (mode == 3 && kind < 3) {
        cudaFuncSetAttribute(online_deep_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        online_deep_kernel<1><<<1, OT, smb, stream>>>(p);
    } else if (sa) {
        cudaFuncSetAttribute(online_deep_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        online_deep_kernel<2><<<1, OT, smb, stream>>>(p);
    } else {
        cudaFuncSetAttribute(online_deep_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        online_deep_kernel<0><<<1, OT, smb, stream>>>(p);
    }
    FMB_CHECK_LAUNCH("online_deep_kernel");
    return FMB_OK;
}

FMB_API int fmb_online_deep_run(int kind, const int32_t* ids, const float* xv, const float* y, int N, int F, int k,
                                int L, int H, float* table, float* bias, float* mlp, float* alpha, float* acc,
                                float lr, float hb, float hs, int mode, uint8_t* preds, int64_t* conf,
                                cudaStream_t stream) {
    return fmb_online_deep_run_ex(kind, ids, xv, y, N, F, k, L, H, table, bias, mlp, alpha, acc, lr, hb, hs, mode, nullptr,
                                  preds, conf, stream);
}
