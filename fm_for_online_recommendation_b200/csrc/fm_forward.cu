// fm_forward.cu -- field-embedding gather + FM second-order term / NFM Bi-Interaction pooling.
//
// Replaces the reference's 2F `nn.Embedding` gathers and ~6F elementwise kernels
// (models/models_online_deep/deepfm_adam.py:46-77, fm_adam.py:34-54; SURVEY.md 8a rows A1-A3).
//
// One CTA stages the packed rows [v(k) | w | pad] of SB samples x F fields in shared memory with
// 128-bit cp.async gathers (all of the tile's row reads are in flight at once: one DRAM latency per
// tile), then reduces over fields left to right (python sum() order, deepfm_adam.py:62,67) with one
// thread per (sample, component), and finishes each sample's logit in ATen's row-sum order.
// HBM-bound: algorithmic bytes/sample = 4F(k+1) row reads + 8F ids/values + outputs.
#include "fmb_common.cuh"

namespace {

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
}

struct FwdParams {
    const int32_t* ids;
    const float* xv;
    const float* table;
    const float* bias;
    int B, F, k, rowp, kp4, SB;
    int cu;      // 16-byte chunks of a row that hold data: ceil((k+1)/4)
    int ql_log;  // log2 of lanes per (sample, field) in the gather phase (pow2 >= cu)
    int jl_log;  // log2 of lanes per sample in the reduce phase (pow2 >= kp4)
    float* first;
    float* S;
    float* bi;
    float* sum_first;
    float* z;
    // fused loss (optional)
    const float* y;
    int loss_kind;
    float* delta;
    float* lossv;
};

__global__ void __launch_bounds__(256) fm_forward_kernel(FwdParams p) {
    extern __shared__ __align__(16) float smem[];
    const int F = p.F, k = p.k, SB = p.SB;
    const int rp = p.cu * 4;                       // shared-memory row pitch (floats)
    float* rows_s = smem;                          // [SB][F][rp]
    float* x_s = rows_s + (size_t)SB * F * rp;     // [SB][F]
    float* bi_s = x_s + SB * F;                    // [SB][k]
    int32_t* ids_s = reinterpret_cast<int32_t*>(bi_s + SB * k);  // [SB][F]
    const int b0 = blockIdx.x * SB;
    const int nv = min(SB, p.B - b0);

    // phase 0: the tile's row ids and values, coalesced (one memory latency for the whole tile)
    for (int e = threadIdx.x; e < nv * F; e += blockDim.x) {
        ids_s[e] = __ldg(p.ids + (size_t)b0 * F + e);
        x_s[e] = p.xv ? __ldg(p.xv + (size_t)b0 * F + e) : 1.0f;
    }
    __syncthreads();
    // phase 1: gather rows, 16 B per cp.async; every row read of the tile is in flight at once.
    // 2^ql_log lanes per (sample, field): no integer division on the address path.
    {
        const int q = threadIdx.x & ((1 << p.ql_log) - 1);
        const int estep = blockDim.x >> p.ql_log;
        if (q < p.cu)
            for (int ef = threadIdx.x >> p.ql_log; ef < nv * F; ef += estep)
                cp_async16(rows_s + (size_t)ef * rp + q * 4, p.table + (size_t)ids_s[ef] * p.rowp + q * 4);
    }
    cp_async_wait_all();
    __syncthreads();

    // phase 2: one thread per (sample, component): S = sum_f e_f, Q = sum_f e_f^2, left to right
    {
        const int j = threadIdx.x & ((1 << p.jl_log) - 1);
        const int sstep = blockDim.x >> p.jl_log;
        if (j < p.kp4)
            for (int s = threadIdx.x >> p.jl_log; s < nv; s += sstep) {
                float Sj = 0.f;
                if (j < k) {
                    float Qj = 0.f;
                    const float* r = rows_s + (size_t)s * F * rp + j;
                    const float* xs = x_s + s * F;
#pragma unroll 4
                    for (int f = 0; f < F; ++f) {
                        const float e = __fmul_rn(r[(size_t)f * rp], xs[f]);
                        Sj = __fadd_rn(Sj, e);
                        Qj = __fadd_rn(Qj, __fmul_rn(e, e));
                    }
                    bi_s[s * k + j] = __fmul_rn(__fsub_rn(__fmul_rn(Sj, Sj), Qj), 0.5f);
                }
                if (p.S) p.S[(size_t)(b0 + s) * p.kp4 + j] = Sj;
            }
    }
    __syncthreads();

    // optional dense outputs (API parity with first_order()/second_order())
    if (p.first)
        for (int e = threadIdx.x; e < nv * F; e += blockDim.x)
            p.first[(size_t)b0 * F + e] = __fmul_rn(rows_s[(size_t)e * rp + k], x_s[e]);
    if (p.bi)
        for (int e = threadIdx.x; e < nv * k; e += blockDim.x) p.bi[(size_t)b0 * k + e] = bi_s[e];

    // phase 3: one thread per sample finishes the logit in ATen's row order
    if (threadIdx.x < nv) {
        const int s = threadIdx.x, b = b0 + s;
        const float* r = rows_s + (size_t)s * F * rp + k;
        const float* xs = x_s + s * F;
        const float sf = fmb::aten_row_sum_small([&](int f) { return __fmul_rn(r[(size_t)f * rp], xs[f]); }, F);
        const float* bs = bi_s + s * k;
        const float sb = fmb::aten_row_sum_small([&](int j) { return bs[j]; }, k);
        const float z = __fadd_rn(__fadd_rn(sf, sb), __ldg(p.bias));
        if (p.sum_first) p.sum_first[b] = sf;
        if (p.z) p.z[b] = z;
        if (p.y) {
            const float y = p.y[b];
            float lv, d;
            fmb::bce_logits_value_grad(p.loss_kind, z, y, b, p.B, lv, d);
            p.lossv[b] = lv;
            p.delta[b] = d;
        }
    }
}

static int ilog2_ceil(int x) { int l = 0; while ((1 << l) < x) ++l; return l; }

}  // namespace

// A1-A3 (+ optional fused loss/delta of A6).  All pointers are device pointers; nullable ones noted.
//   ids   [B,F] int32 global row ids (field offset + local id)
//   xv    [B,F] fp32 feature values, NULL = all ones (Criteo, utils/data_preprocess.py:41)
//   table [R,rowp] packed rows, rowp = fmb_rowp(k) = round_up(k+1, 16): 64-byte aligned rows, so a
//         random row read costs exactly ceil(4(k+1)/64) DRAM bursts
//   bias  [1]
//   first [B,F], S [B,kp4], bi [B,k], sum_first [B], z [B]   (each nullable)
//   y [B] labels: when non-NULL also writes delta[B], lossv[B] for loss kind 0 (BCEWithLogits(z))
//   or 1 (BCEWithLogits(sigmoid(z))).
FMB_API int fmb_fm_forward(const int32_t* ids, const float* xv, const float* table, const float* bias, int B, int F,
                           int k, float* first, float* S, float* bi, float* sum_first, float* z, const float* y,
                           int loss_kind, float* delta, float* lossv, cudaStream_t stream) {
    FMB_CHECK_ARG(ids && table && bias, "fmb_fm_forward: null ids/table/bias");
    FMB_CHECK_ARG(B > 0 && F > 0 && k > 0, "fmb_fm_forward: bad shape B=%d F=%d k=%d", B, F, k);
    FMB_CHECK_ARG(F < 512 && k <= 252, "fmb_fm_forward: bad shape F=%d k=%d (need F < 512, k <= 252)", F, k);
    FMB_CHECK_ARG(!y || (delta && lossv), "fmb_fm_forward: y given without delta/lossv");
    FwdParams p;
    p.ids = ids; p.xv = xv; p.table = table; p.bias = bias;
    p.B = B; p.F = F; p.k = k; p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4);
    p.cu = (k + 1 + 3) / 4; p.ql_log = ilog2_ceil(p.cu); p.jl_log = ilog2_ceil(p.kp4);
    p.first = first; p.S = S; p.bi = bi; p.sum_first = sum_first; p.z = z;
    p.y = y; p.loss_kind = loss_kind; p.delta = delta; p.lossv = lossv;
    int SB = 256 >> p.jl_log;  // samples whose (sample, component) lanes fill one 256-thread pass
    if (SB < 4) SB = 4;
    if (SB > 32) SB = 32;
    auto bytes = [&](int sb) {
        return sizeof(float) * ((size_t)sb * F * p.cu * 4 + (size_t)2 * sb * F + (size_t)sb * k);
    };
    while (SB > 1 && bytes(SB) > 48 * 1024) SB >>= 1;
    FMB_CHECK_ARG(bytes(SB) <= 200 * 1024, "fmb_fm_forward: F*k too large for one sample tile (F=%d k=%d)", F, k);
    p.SB = SB;
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(fm_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr_set = true;
    }
    const int grid = (B + SB - 1) / SB;
    fm_forward_kernel<<<grid, 256, bytes(SB), stream>>>(p);
    FMB_CHECK_LAUNCH("fm_forward_kernel");
    return FMB_OK;
}
