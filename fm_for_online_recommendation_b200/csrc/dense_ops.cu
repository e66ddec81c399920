// dense_ops.cu -- small dense pieces of the training step: loss/delta, ATen-order reductions,
// dense parameter updates (bias, MLP), and the fused end-of-step kernel.
// Reference: F.binary_cross_entropy_with_logits + loss.backward() + torch.optim.Adam.step in
// models/models_online_deep/fm_adam.py:60-68 (SURVEY.md 8a A6, A12).
#include "fmb_common.cuh"

namespace {

__global__ void loss_delta_kernel(int kind, const float* __restrict__ z, const float* __restrict__ y, int B,
                                  float* __restrict__ delta, float* __restrict__ lossv) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float yy = y[b];
    float lv, d;
    fmb::bce_logits_value_grad(kind, z[b], yy, b, B, lv, d);
    if (lossv) lossv[b] = lv;
    delta[b] = d;
}

// element-wise evaluation of the ATen mirrors (fmb_aten_math.cuh), so tests can compare them with the oracle's
__global__ void math_eval_kernel(int op, const float* __restrict__ x, float* __restrict__ y, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float v = x[i];
    float r;
    switch (op) {
        case 0: r = fmb::sigmoid_at(v, (int)i, (int)n); break;   // torch.sigmoid of a contiguous [n] tensor
        case 1: r = fmb::log_sigmoid(v); break;
        case 2: r = fmb::sqrt_mkl(v); break;
        default: r = fmb::expf_glibc(v); break;
    }
    y[i] = r;
}

__global__ void sum_aten_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ out) {
    const float s = fmb::aten_row_sum_warp(x, n);
    if (threadIdx.x == 0) out[0] = s;
}

__global__ void update_dense_kernel(float* __restrict__ p, const float* __restrict__ g, int64_t n, float lr,
                                    int mode) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = fmb::apply_update(p[i], g[i], lr, mode);
}

// update mode 3 (Adagrad) of dense parameters: sums [n] next to the parameters
__global__ void update_dense_adagrad_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ sums,
                                            int64_t n, float lr, float eps) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        float s = sums[i];
        p[i] = fmb::adagrad_update(p[i], g[i], s, lr, eps);
        sums[i] = s;
    }
}

// update mode 4's dense Adam of the tower: m [n] at mv, v [n] at mv + n
__global__ void update_dense_adam_kernel(float* __restrict__ p, const float* __restrict__ g, int64_t n, fmb::AdamState st) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        float m = st.mv[i], v = st.mv[n + i];
        p[i] = fmb::adam_update(p[i], g[i], m, v, st);
        st.mv[i] = m; st.mv[n + i] = v;
    }
}

// ATen-order sum of x[0:n], parallel where the order allows it.  ATen's cascade (SumKernel.cpp multi_row_sum)
// adds rows of 32 floats (4 ilp x 8 lanes) in blocks of `level_step` rows: a block's sum is
// ((0 + r0) + r1) + ... and depends on nothing else, only the way block sums are folded upwards is serial.
// So: phase A, every warp computes block sums (one lane per accumulator, 16 loads in flight); phase B, one warp
// folds the block sums through levels 1..3 exactly like the serial loop, adds the left-over rows, the left-over
// vectors and the scalar tail.  Bit-identical to fmb::aten_row_sum_warp / orc_sum_aten.
constexpr int FIN_THREADS = 1024;
constexpr int FIN_MAX_BLOCKS = 2048;   // block sums kept in shared memory per array (n <= 2048*16*32 = 1 M)

__device__ float aten_sum_cta(const float* __restrict__ x, int64_t n, float* bs /*[FIN_MAX_BLOCKS][32]*/, int w0,
                              int nw) {
    // called by warps [w0, w0+nw) of the CTA with the same arguments; result valid in warp w0
    const int warp = (threadIdx.x >> 5) - w0, lane = threadIdx.x & 31;
    const int64_t vec_size = n >> 3, size_ilp = vec_size >> 2;
    int lp = 0;
    while (((int64_t)1 << lp) < size_ilp) ++lp;
    lp >>= 2;
    const int level_power = lp > 4 ? lp : 4;
    const int64_t level_step = (int64_t)1 << level_power, level_mask = level_step - 1;
    const int64_t nblocks = size_ilp / level_step;
    // phase A: block sums
    for (int64_t bi = warp; bi < nblocks; bi += nw) {
        const float* r = x + bi * level_step * 32 + lane;
        float a = 0.f;
        for (int64_t j = 0; j < level_step; j += 16) {
            float v[16];
#pragma unroll
            for (int u = 0; u < 16; ++u) v[u] = r[(j + u) * 32];
#pragma unroll
            for (int u = 0; u < 16; ++u) a = __fadd_rn(a, v[u]);
        }
        bs[bi * 32 + lane] = a;
    }
    // all participating warps must have written their block sums
    asm volatile("bar.sync %0, %1;" ::"r"(1 + (w0 ? 1 : 0)), "r"(nw * 32));
    float total = 0.f;
    if (warp == 0) {
        float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
        for (int64_t bi = 0; bi < nblocks; ++bi) {
            const int64_t i = (bi + 1) * level_step;   // rows consumed so far
            acc1 = __fadd_rn(acc1, bs[bi * 32 + lane]);
            if ((i & (level_mask << level_power)) == 0) {
                acc2 = __fadd_rn(acc2, acc1); acc1 = 0.f;
                if ((i & (level_mask << (2 * level_power))) == 0) { acc3 = __fadd_rn(acc3, acc2); acc2 = 0.f; }
            }
        }
        for (int64_t i = nblocks * level_step; i < size_ilp; ++i) acc0 = __fadd_rn(acc0, x[i * 32 + lane]);
        float a = __fadd_rn(__fadd_rn(__fadd_rn(acc0, acc1), acc2), acc3);
        if (lane < 8)
            for (int64_t v = size_ilp << 2; v < vec_size; ++v) a = __fadd_rn(a, x[v * 8 + lane]);
        const float t1 = __shfl_down_sync(0xffffffffu, a, 8);
        const float t2 = __shfl_down_sync(0xffffffffu, a, 16);
        const float t3 = __shfl_down_sync(0xffffffffu, a, 24);
        const float folded = __fadd_rn(__fadd_rn(__fadd_rn(a, t1), t2), t3);
        float fin = 0.f;
        for (int64_t q = vec_size << 3; q < n; ++q) fin = __fadd_rn(fin, x[q]);
#pragma unroll
        for (int l = 0; l < 8; ++l) fin = __fadd_rn(fin, __shfl_sync(0xffffffffu, folded, l));
        total = fin;
    }
    return total;
}

// warps 0..15: bias -= step(sum(delta));  warps 16..31: loss_out = sum(lossv) / B.  SA: update mode 4 (Adam on st.adam, an
// instantiation of its own so that the other modes' kernel stays as it is)
template <bool SA>
__global__ void __launch_bounds__(FIN_THREADS) finish_step_kernel(const float* __restrict__ delta,
                                                                  const float* __restrict__ lossv, int B, float* bias,
                                                                  float lr, int mode, float* loss_out,
                                                                  float* scratch /*[2][nblocks*32] or NULL*/,
                                                                  fmb::UpdateState st) {
    extern __shared__ __align__(16) float fin_sm[];
    const int half = (threadIdx.x >> 5) >= 16 ? 1 : 0;
    const float* src = half == 0 ? (bias ? delta : nullptr) : ((loss_out && lossv) ? lossv : nullptr);
    if (!src) return;
    const int64_t n = B;
    const int lane = threadIdx.x & 31;
    float total;
    if (n < 8) {
        if ((threadIdx.x >> 5) != half * 16) return;
        total = fmb::aten_row_sum_warp(src, n);
    } else {
        float* bs = scratch ? scratch + (size_t)half * FIN_MAX_BLOCKS * 32 : fin_sm + (size_t)half * 512 * 32;
        total = aten_sum_cta(src, n, bs, half * 16, 16);
        if ((threadIdx.x >> 5) != half * 16) return;
    }
    if (lane == 0) {
        if (half == 0) {
            if (SA) {
                float m = st.adam.mv[0], v = st.adam.mv[1];
                bias[0] = fmb::adam_update(bias[0], total, m, v, st.adam);
                st.adam.mv[0] = m; st.adam.mv[1] = v;
            } else if (mode == 2) {
                const fmb::FtrlState& ftrl = st.ftrl;
                float z = ftrl.bias_zn[0], n = ftrl.bias_zn[1];
                bias[0] = fmb::ftrl_update(bias[0], total, z, n, lr, ftrl.beta, ftrl.l1, ftrl.l2);
                ftrl.bias_zn[0] = z; ftrl.bias_zn[1] = n;
            } else if (mode == 3) {
                float s = st.ada.bias_sum[0];
                bias[0] = fmb::adagrad_update(bias[0], total, s, lr, st.ada.eps);
                st.ada.bias_sum[0] = s;
            } else {
                bias[0] = fmb::apply_update(bias[0], total, lr, mode);
            }
        }
        else loss_out[0] = __fdiv_rn(total, (float)B);
    }
}

}  // namespace

// BCEWithLogits value and gradient per sample.  kind 0: loss(z); kind 1: loss(sigmoid(z)).
// delta[B] = dLoss/dz (mean reduction folded in); lossv[B] (nullable) = per-sample loss.
FMB_API int fmb_loss_delta(int kind, const float* z, const float* y, int B, float* delta, float* lossv,
                           cudaStream_t stream) {
    FMB_CHECK_ARG(z && y && delta && B > 0, "fmb_loss_delta: bad arguments");
    FMB_CHECK_ARG(kind == 0 || kind == 1, "fmb_loss_delta: unknown loss kind %d", kind);
    loss_delta_kernel<<<(B + 255) / 256, 256, 0, stream>>>(kind, z, y, B, delta, lossv);
    FMB_CHECK_LAUNCH("loss_delta_kernel");
    return FMB_OK;
}

// y[i] = f(x[i]) for the ATen mirrors: op 0 torch.sigmoid (element i of a contiguous [n] tensor, n < 2^31),
// 1 at::log_sigmoid, 2 Tensor.sqrt (MKL vsSqrt), 3 glibc expf.  Exists so that parity tests can sweep them.
FMB_API int fmb_math_eval(int op, const float* x, float* y, int64_t n, cudaStream_t stream) {
    FMB_CHECK_ARG(x && y && n > 0 && n < ((int64_t)1 << 31) && op >= 0 && op <= 3, "fmb_math_eval: bad arguments");
    math_eval_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(op, x, y, n);
    FMB_CHECK_LAUNCH("math_eval_kernel");
    return FMB_OK;
}

// out[0] = sum(x[0:n]) in ATen's CPU order (what torch.sum / .mean() / the bias gradient use)
FMB_API int fmb_sum_aten(const float* x, int64_t n, float* out, cudaStream_t stream) {
    FMB_CHECK_ARG(x && out && n > 0, "fmb_sum_aten: bad arguments");
    sum_aten_kernel<<<1, 32, 0, stream>>>(x, n, out);
    FMB_CHECK_LAUNCH("sum_aten_kernel");
    return FMB_OK;
}

// p[i] <- update(p[i], g[i]) for dense parameters (bias, MLP weights); mode as in fmb_fm_backward_update
FMB_API int fmb_update_dense(float* p, const float* g, int64_t n, float lr, int mode, cudaStream_t stream) {
    FMB_CHECK_ARG(p && g && n > 0, "fmb_update_dense: bad arguments");
    FMB_CHECK_ARG(mode == 0 || mode == 1, "fmb_update_dense: unknown update mode %d", mode);
    update_dense_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(p, g, n, lr, mode);
    FMB_CHECK_LAUNCH("update_dense_kernel");
    return FMB_OK;
}

// _ex: update mode 3 (Adagrad) with the parameters' sums [n] (read and written; NULL in the other modes)
FMB_API int fmb_update_dense_ex(float* p, const float* g, int64_t n, float lr, int mode, float* sums, float eps,
                                cudaStream_t stream) {
    if (mode != 3) return fmb_update_dense(p, g, n, lr, mode, stream);
    FMB_CHECK_ARG(p && g && n > 0 && sums, "fmb_update_dense: bad arguments (mode 3 needs the Adagrad sums)");
    update_dense_adagrad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(p, g, sums, n, lr, eps);
    FMB_CHECK_LAUNCH("update_dense_adagrad_kernel");
    return FMB_OK;
}

// update mode 4: torch.optim.Adam on the tower's n parameters with the moments a->mlp_mv [2][n] and the scalars of
// a->cur (fmb_sparse_adam_advance with tower = 1)
FMB_API int fmb_update_dense_adam(float* p, const float* g, int64_t n, const fmb_sparse_adam_t* a, cudaStream_t stream) {
    FMB_CHECK_ARG(p && g && n > 0 && a && a->mlp_mv, "fmb_update_dense_adam: bad arguments (needs the tower's moments)");
    update_dense_adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(p, g, n, fmb_sa_dense(a, true));
    FMB_CHECK_LAUNCH("update_dense_adam_kernel");
    return FMB_OK;
}

// end of a training step: bias update from sum(delta) (bias nullable) and mean loss (loss_out nullable).
// B <= 1 M samples (block sums are staged in shared memory up to 256 K samples, in `fmb_finish_scratch` above).
static float* g_fin_scratch = nullptr;
struct fmb_ftrl_t { float* zn; float* bias_zn; float beta, l1, l2; };   // include/fmb200.h
struct fmb_adagrad_t { float* sums; float* bias_sum; float* mlp_sums; float eps; };   // include/fmb200.h (mode 3's state)

FMB_API int fmb_finish_step_ex(const float* delta, const float* lossv, int B, float* bias, float lr, int mode,
                               const fmb_ftrl_t* ftrl, float* loss_out, cudaStream_t stream) {
    FMB_CHECK_ARG(delta && B > 0, "fmb_finish_step: bad arguments");
    FMB_CHECK_ARG((int64_t)B <= (int64_t)FIN_MAX_BLOCKS * 16 * 32, "fmb_finish_step: B=%d too large", B);
    // block sums: 2 arrays x (B/512) blocks x 32 floats; shared memory up to 512 blocks per array (128 KB total)
    const int64_t nblocks = ((int64_t)B >> 5) / 16;
    float* scratch = nullptr;
    size_t smem = 0;
    if (nblocks <= 512) {
        smem = (size_t)2 * 512 * 32 * sizeof(float);
    } else {
        if (!g_fin_scratch && cudaMalloc(&g_fin_scratch, (size_t)2 * FIN_MAX_BLOCKS * 32 * sizeof(float)) != cudaSuccess) {
            fmb_set_error("fmb_finish_step: scratch allocation failed");
            return FMB_ERR_CUDA;
        }
        scratch = g_fin_scratch;
    }
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(finish_step_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 132 * 1024);
        cudaFuncSetAttribute(finish_step_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 132 * 1024);
        attr = true;
    }
    fmb::UpdateState fs;
    fs.ftrl = {nullptr, nullptr, 0.f, 0.f, 0.f};
    if (mode == 2) {
        FMB_CHECK_ARG(ftrl && ftrl->bias_zn, "fmb_finish_step: update mode 2 needs the FTRL state");
        fs.ftrl.zn = ftrl->zn; fs.ftrl.bias_zn = ftrl->bias_zn; fs.ftrl.beta = ftrl->beta; fs.ftrl.l1 = ftrl->l1; fs.ftrl.l2 = ftrl->l2;
    } else if (mode == 3) {   // the state slot carries an fmb_adagrad_t in mode 3 (include/fmb200.h)
        const fmb_adagrad_t* a = reinterpret_cast<const fmb_adagrad_t*>(ftrl);
        FMB_CHECK_ARG(bias == nullptr || (a && a->bias_sum), "fmb_finish_step: update mode 3 needs the Adagrad state");
        if (a) { fs.ada.sums = a->sums; fs.ada.bias_sum = a->bias_sum; fs.ada.eps = a->eps; }
    } else if (mode == 4) {   // the state slot carries an fmb_sparse_adam_t advanced to this step (include/fmb200.h)
        const fmb_sparse_adam_t* a = reinterpret_cast<const fmb_sparse_adam_t*>(ftrl);
        FMB_CHECK_ARG(bias == nullptr || (a && a->bias_mv), "fmb_finish_step: update mode 4 needs the SparseAdam state");
        if (a) fs.adam = fmb_sa_dense(a, false);
    }
    if (mode == 4) finish_step_kernel<true><<<1, FIN_THREADS, smem, stream>>>(delta, lossv, B, bias, lr, mode, loss_out, scratch, fs);
    else finish_step_kernel<false><<<1, FIN_THREADS, smem, stream>>>(delta, lossv, B, bias, lr, mode, loss_out, scratch, fs);
    FMB_CHECK_LAUNCH("finish_step_kernel");
    return FMB_OK;
}

// host-side handle of the kernel, for graph-node identification in session.cu (argument 6 of 9 = loss_out)
FMB_API const void* fmb_finish_kernel_fn(void) { return (const void*)finish_step_kernel<false>; }
// the mode-4 instantiation (argument 8 = the bias's Adam state, re-pointed at every step's scalars by session.cu)
const void* fmb_finish_sa_kernel_fn() { return (const void*)finish_step_kernel<true>; }

FMB_API int fmb_finish_step(const float* delta, const float* lossv, int B, float* bias, float lr, int mode,
                            float* loss_out, cudaStream_t stream) {
    return fmb_finish_step_ex(delta, lossv, B, bias, lr, mode, nullptr, loss_out, stream);
}
