// fm_step.cu -- the FM-only training step (forward_fm + BCE-with-logits + sparse backward + row update) with the
// rows read ONCE: one kernel gathers the rows of a tile of samples, computes the logits, the loss gradient and
// -- because the stable sort of the batch's row ids has already told it which entries are the only hit of their
// row -- applies the update of those rows from the copy it holds in shared memory.  Entries of rows hit several
// times write their contribution to the component-major staging buffer G at their SORTED position; the run
// kernel of fm_backward.cu then sums each run in sample order (the reference's embedding_dense_backward order)
// and updates those rows.
//
// Replaces, for FMAdam.update_embedding / fit and the update_embedding of the other four classes
// (models/models_online_deep/fm_adam.py:56-82, deepfm_adam.py:91-104, nfm_adam.py:90-103, deepfm_onn.py:156-169,
// nfm_onn.py:158-171), the round-1 sequence fm_forward_kernel -> fm_bwd_entry1_kernel (which read every row a
// second time: 31 MB of the step's 68 MB of DRAM traffic at cfg5) -> fm_bwd_runs_kernel.
//
// Safety of updating inside the forward kernel: a row that is hit by exactly one entry of the batch is read by
// exactly one CTA -- the one that updates it -- so no other sample's forward pass can observe the new value.
// Algorithmic bytes per sample (k = 10, F = 39): ids 4F + position/flag words 4F + rows read 4F(k+1) + rows
// written 4F(k+1) + delta/loss 8 = 3 752 B (SURVEY.md 8d's figure; the sorted-position words replace the
// sorted-key reads of the entry kernel).
#include "fmb_common.cuh"
#include <cstdlib>

extern "C" size_t fmb_bwd_workspace_bytes(int64_t, int);

namespace {

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
}

// The four per-batch pointers are separate kernel arguments (not members of StepParams) so that a captured CUDA
// graph of the step can be re-pointed at another batch with cudaGraphExecKernelNodeSetParams (session.cu).
struct StepParams {
    float* table;              // [R,rowp]
    const float* bias;         // [1]
    int B, F, k, rowp, kp4, SB;
    int cu;                    // 16-byte chunks of a row that hold data: ceil((k+1)/4)
    int ql_log;                // log2 of lanes per (sample, field) in the gather phase (pow2 >= cu)
    int jl_log;                // log2 of lanes per sample in the reduce phase (pow2 >= kp4)
    uint32_t mF, mcu;          // fmb_div_magic(F), fmb_div_magic(cu): x / F == fmb_div_by_magic(x, mF) (x < SB*F*cu)
    int loss_kind, mode;
    float lr, astep;
    float* delta;              // [B] out
    float* lossv;              // [B] out
    float* G;                  // [k+1][Npad] staged contributions of multi-hit entries
    int64_t Npad;
    union {                    // the update rule's per-coordinate state (same size as the FTRL state alone)
        fmb::FtrlState ftrl;       // mode 2 only
        fmb::AdagradState ada;     // mode 3 only
    };
    long long* tdbg;           // debug only: per-CTA phase timestamps [grid][8] (globaltimer ns), else NULL
    int dbg;                   // debug/attribution only (fmb_debug_set_step_flags): 1 = skip phase 4a, 2 = skip phase 4b
};

//   ids [B,F] global row ids;  xv [B,F] or NULL (all ones);  y [B];
//   posflag [B*F] entry-major: sorted position of the entry | 0x80000000 if its row is hit more than once
// Template parameters: CU = 16-byte chunks per row when known at compile time (3 for k = 8..11: the row pitch in shared
// memory is then a constant and the field loop addresses with immediates), 0 = read it from the parameters;
// XV = the batch carries real feature values (else all ones: no loads, no multiplications by x -- a product with 1.0f
// is exact, so skipping it changes no bit); MODE = update rule (0 fresh-Adam sign step, 1 SGD, 2 FTRL-Proximal,
// 3 Adagrad).
// 32 registers (8 CTAs per SM): the 1 024 tiles of an 8 192-sample batch are then resident at once.
template <int CU, bool XV, int MODE>
__global__ void __launch_bounds__(256, MODE == 2 ? 4 : 8) fm_step_fused_kernel(const int32_t* __restrict__ ids, const float* __restrict__ xv,
                                                            const float* __restrict__ y, const uint32_t* __restrict__ posflag,
                                                            StepParams p) {
    extern __shared__ __align__(16) float smem[];
    const int F = p.F, k = p.k, SB = p.SB;
    const int cu = CU ? CU : p.cu;
    const int rp = cu * 4;                         // shared-memory row pitch (floats)
    float* rows_s = smem;                          // [SB][F][rp]
    float* S_s = rows_s + (size_t)SB * F * rp;     // [SB][rp]  (16-byte aligned: read as float4)
    float* x_s = S_s + SB * rp;                    // [SB][F]   (XV only)
    float* bi_s = x_s + (XV ? SB * F : 0);         // [SB][k]
    float* d_s = bi_s + SB * k;                    // [SB]
    int32_t* ids_s = reinterpret_cast<int32_t*>(d_s + SB);            // [SB][F]
    uint32_t* pos_s = reinterpret_cast<uint32_t*>(ids_s + SB * F);    // [SB][F]
    uint16_t* single_s = reinterpret_cast<uint16_t*>(pos_s + SB * F); // [SB*F] entries whose row is hit once
    uint16_t* multi_s = single_s + SB * F;                            // [SB*F] the others
    __shared__ int n_single, n_multi;
    if (threadIdx.x == 0) { n_single = 0; n_multi = 0; }
    __syncthreads();
    const int b0 = blockIdx.x * SB;
    const int nv = min(SB, p.B - b0);
    // programmatic dependent launch: the run kernel behind this one may be launched (and run its prologue: segment
    // counts, list entry, mbarriers) as soon as every CTA of this grid has started; it waits for this grid's completion
    // (griddepcontrol.wait) before it reads the staged contributions.  No effect without the launch attribute.
    asm volatile("griddepcontrol.launch_dependents;\n" ::);
#define FMB_TS(i) do { if (p.tdbg && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_)); p.tdbg[(size_t)blockIdx.x * 8 + (i)] = (long long)t_; } } while (0)
    FMB_TS(0);

    // phase 0: the tile's row ids, values and sorted positions, coalesced; the entries are split into two compact
    // lists (row hit once / several times) so that the update phase runs full warps down one code path each
    for (int e0 = (threadIdx.x & ~31); e0 < nv * F; e0 += blockDim.x) {
        const int e = e0 + (threadIdx.x & 31);
        const bool valid = e < nv * F;
        uint32_t pf = 0;
        if (valid) {
            ids_s[e] = __ldg(ids + (size_t)b0 * F + e);
            if (XV) x_s[e] = __ldg(xv + (size_t)b0 * F + e);
            pf = __ldg(posflag + (size_t)b0 * F + e);
            pos_s[e] = pf;
        }
        const unsigned ms = __ballot_sync(0xffffffffu, valid && !(pf >> 31));
        const unsigned mm = __ballot_sync(0xffffffffu, valid && (pf >> 31));
        int bs = 0, bm = 0;
        if ((threadIdx.x & 31) == 0) { bs = atomicAdd(&n_single, __popc(ms)); bm = atomicAdd(&n_multi, __popc(mm)); }
        bs = __shfl_sync(0xffffffffu, bs, 0);
        bm = __shfl_sync(0xffffffffu, bm, 0);
        const unsigned lt = (1u << (threadIdx.x & 31)) - 1u;
        if (valid) {
            if (pf >> 31) multi_s[bm + __popc(mm & lt)] = (uint16_t)e;
            else single_s[bs + __popc(ms & lt)] = (uint16_t)e;
        }
    }
    __syncthreads();
    FMB_TS(1);
    // phase 1: gather rows, 16 B per cp.async; every row read of the tile is in flight at once
    {
        const int q = threadIdx.x & ((1 << p.ql_log) - 1);
        const int estep = blockDim.x >> p.ql_log;
        if (q < cu)
            for (int ef = threadIdx.x >> p.ql_log; ef < nv * F; ef += estep)
                cp_async16(rows_s + (size_t)ef * rp + q * 4, p.table + (size_t)ids_s[ef] * p.rowp + q * 4);
    }
    cp_async_wait_all();
    __syncthreads();
    FMB_TS(2);

    // phase 2: one thread per (sample, component): S = sum_f e_f, Q = sum_f e_f^2, left to right (python sum() order)
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
#pragma unroll 8
                    for (int f = 0; f < F; ++f) {
                        const float e = XV ? __fmul_rn(r[(size_t)f * rp], xs[f]) : r[(size_t)f * rp];
                        Sj = __fadd_rn(Sj, e);
                        Qj = __fadd_rn(Qj, __fmul_rn(e, e));
                    }
                    bi_s[s * k + j] = __fmul_rn(__fsub_rn(__fmul_rn(Sj, Sj), Qj), 0.5f);
                }
                S_s[s * rp + j] = Sj;
            }
    }
    __syncthreads();
    FMB_TS(3);

    // phase 3: eight lanes per sample: logit in ATen's row-sum order (the eight vector-lane chains side by side),
    // then lane 0 of the group: loss value and gradient on the logit
    {
        const int s = threadIdx.x >> 3, l8 = threadIdx.x & 7;
        const int nv8 = (nv + 3) & ~3;                        // whole warps take part in the shuffles
        if (s < nv8) {
            const unsigned mask = 0xffffffffu;
            const int sc = min(s, nv - 1);                    // padding groups recompute the last sample (discarded)
            const float* r = rows_s + (size_t)sc * F * rp + k;
            const float* xs = x_s + sc * F;
            const float sf = fmb::aten_row_sum_lanes8(
                [&](int f) { return XV ? __fmul_rn(r[(size_t)f * rp], xs[f]) : r[(size_t)f * rp]; }, F, l8, mask);
            const float* bs = bi_s + sc * k;
            const float sb = fmb::aten_row_sum_lanes8([&](int j) { return bs[j]; }, k, l8, mask);
            if (l8 == 0 && s < nv) {
                const int b = b0 + s;
                const float z = __fadd_rn(__fadd_rn(sf, sb), __ldg(p.bias));
                float lv, d;
                fmb::bce_logits_value_grad(p.loss_kind, z, y[b], b, p.B, lv, d);
                p.lossv[b] = lv;
                p.delta[b] = d;
                d_s[s] = d;
            }
        }
    }
    __syncthreads();
    FMB_TS(4);

    // phase 4a: rows hit once, one thread per (entry, 16-byte chunk): the gradient is the entry's contribution alone
    // (0 + contribution, like the reference's zero-initialised grad row); the row is updated from the shared-memory
    // copy.  Chunks no coordinate of which moved are not written back (on saturated samples the sign step is below a
    // quarter ulp of every weight).  Item -> (entry, chunk) and entry -> sample by multiplication with the
    // precomputed reciprocals (a runtime integer division is ~20 instructions, and there were two per item).
    const int ns = n_single, nm = n_multi;
    for (int it = threadIdx.x; it < ((p.dbg & 1) ? 0 : ns * cu); it += blockDim.x) {
        const int li = fmb_div_by_magic((unsigned)it, p.mcu), q = it - li * cu;
        const int ef = single_s[li];
        const int s = fmb_div_by_magic((unsigned)ef, p.mF);
        const float x = XV ? x_s[ef] : 1.0f, d = d_s[s];
        const float4 S4 = *reinterpret_cast<const float4*>(S_s + s * rp + q * 4);
        const float4 v4 = *reinterpret_cast<const float4*>(rows_s + (size_t)ef * rp + q * 4);
        const float Sq[4] = {S4.x, S4.y, S4.z, S4.w};
        const float v[4] = {v4.x, v4.y, v4.z, v4.w};
        if (MODE != 2) {
            // Saturated samples (the reference's N(0,1) initialisation puts |z| ~ 90 on Criteo-shaped rows) leave their
            // rows exactly where they are; two exact item-level tests spare them the per-coordinate work.
            // (i) delta == 0 (sigmoid rounded to y): every gradient is +0 after the `0 +`, and the Adam step of a zero
            //     gradient returns p for every p (shortcut, or p + (-0) in the full pipeline); SGD: fma(+0, -lr, p) = p;
            //     Adagrad: fma(+0, +0, s) = s and p + (-0) / std = p.
            if (d == 0.0f) continue;
            // (ii) |delta| < 1e-30 with |S_j| < 1e4 and 1e-9 < |p| < 1e4: |g| <= 2.0001e-26 is below the window test's
            //     range, and the quarter-ulp bound |a|*0.1*|g|*1.0001e8 <= 2.001e-18 (|a| <= 10) is below
            //     2^-26*|p| >= 1.49e-17: adam1_a returns p.
            if (MODE == 0 && !XV && fabsf(d) < 1e-30f && fabsf(p.astep) <= 10.0f) {
                bool same = true;
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    const int j = q * 4 + t;
                    const float av = fabsf(v[t]);
                    if (j <= k) same = same && av > 1e-9f && av < 1e4f;
                    if (j < k) same = same && fabsf(Sq[t]) < 1e4f;
                }
                if (same) continue;
            }
        }
        if (MODE == 3) {
            // Adagrad: the row's sums sit at the row's offsets of their own table (read + written: 8F(k+1) more bytes per
            // sample).  Gradient and update per coordinate, so that only one gradient is live at a time (32 registers).
            float* srow = p.ada.sums + (size_t)ids_s[ef] * p.rowp + q * 4;
            const float4 s4 = *reinterpret_cast<const float4*>(srow);
            float sv[4] = {s4.x, s4.y, s4.z, s4.w}, o[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                const int j = q * 4 + t;
                o[t] = v[t];
                if (j <= k) {
                    float a;
                    if (j < k) {
                        const float ej = XV ? __fmul_rn(v[t], x) : v[t];
                        a = __fsub_rn(__fmul_rn(d, Sq[t]), __fmul_rn(d, ej));
                        if (XV) a = __fmul_rn(a, x);
                    } else {
                        a = XV ? __fmul_rn(d, x) : d;
                    }
                    o[t] = fmb::adagrad_update(v[t], __fadd_rn(0.f, a), sv[t], p.lr, p.ada.eps);
                }
            }
            *reinterpret_cast<float4*>(p.table + (size_t)ids_s[ef] * p.rowp + q * 4) = make_float4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<float4*>(srow) = make_float4(sv[0], sv[1], sv[2], sv[3]);   // padding lanes: as read
            continue;
        }
        float o[4];
        bool moved = false;
        float zz[4] = {0.f, 0.f, 0.f, 0.f}, nn[4] = {0.f, 0.f, 0.f, 0.f};
        float* zrow = nullptr;
        if (MODE == 2) {   // FTRL-Proximal: the row's z and n sub-rows (read + written: 16F(k+1) more bytes per sample)
            zrow = p.ftrl.zn + (size_t)ids_s[ef] * 2 * p.rowp + q * 4;
            const float4 z4 = *reinterpret_cast<const float4*>(zrow), n4 = *reinterpret_cast<const float4*>(zrow + p.rowp);
            zz[0] = z4.x; zz[1] = z4.y; zz[2] = z4.z; zz[3] = z4.w;
            nn[0] = n4.x; nn[1] = n4.y; nn[2] = n4.z; nn[3] = n4.w;
        }
        float g[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {       // the entry's contribution = the row's gradient (0 + contribution)
            const int j = q * 4 + t;
            float a = 0.f;
            if (j < k) {
                const float ej = XV ? __fmul_rn(v[t], x) : v[t];
                a = __fsub_rn(__fmul_rn(d, Sq[t]), __fmul_rn(d, ej));
                if (XV) a = __fmul_rn(a, x);
            } else if (j == k) {
                a = XV ? __fmul_rn(d, x) : d;
            }
            g[t] = __fadd_rn(0.f, a);
            o[t] = v[t];
        }
        if (MODE == 2) {
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (q * 4 + t <= k) {
                    o[t] = fmb::ftrl_update(v[t], g[t], zz[t], nn[t], p.lr, p.ftrl.beta, p.ftrl.l1, p.ftrl.l2);
                    moved = true;
                }
        } else if (MODE == 1) {
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (q * 4 + t <= k) { o[t] = __fmaf_rn(g[t], -p.lr, v[t]); moved |= __float_as_int(o[t]) != __float_as_int(v[t]); }
        } else {
            // Adam: the window test on all four coordinates without a branch, then -- rarely -- the rest (the quarter-ulp
            // shortcut and the full pipeline) for the coordinates it did not settle.  One divergent region per item
            // instead of two per coordinate.
            unsigned need = 0;
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                float w;
                const bool ok = fmb::adam1_window(v[t], g[t], p.astep, w);
                if (q * 4 + t <= k) { if (ok) o[t] = w; else need |= 1u << t; }
            }
            if (need) {
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    if ((need >> t) & 1u) o[t] = fmb::adam1_rest(v[t], g[t], p.astep, fmb::adam1_in_domain(g[t], p.astep));
            }
#pragma unroll
            for (int t = 0; t < 4; ++t) moved |= __float_as_int(o[t]) != __float_as_int(v[t]);
        }
        if (moved) *reinterpret_cast<float4*>(p.table + (size_t)ids_s[ef] * p.rowp + q * 4) = make_float4(o[0], o[1], o[2], o[3]);
        if (MODE == 2) {
            *reinterpret_cast<float4*>(zrow) = make_float4(zz[0], zz[1], zz[2], zz[3]);
            *reinterpret_cast<float4*>(zrow + p.rowp) = make_float4(nn[0], nn[1], nn[2], nn[3]);
        }
    }
    FMB_TS(5);
    // phase 4b: rows hit several times: stage the entry's contribution at its sorted position (run kernel sums them)
    for (int it = threadIdx.x; it < ((p.dbg & 2) ? 0 : nm * cu); it += blockDim.x) {
        const int li = fmb_div_by_magic((unsigned)it, p.mcu), q = it - li * cu;
        const int ef = multi_s[li];
        const int s = fmb_div_by_magic((unsigned)ef, p.mF);
        const float x = XV ? x_s[ef] : 1.0f, d = d_s[s];
        const float4 S4 = *reinterpret_cast<const float4*>(S_s + s * rp + q * 4);
        const float4 v4 = *reinterpret_cast<const float4*>(rows_s + (size_t)ef * rp + q * 4);
        const float Sq[4] = {S4.x, S4.y, S4.z, S4.w};
        const float v[4] = {v4.x, v4.y, v4.z, v4.w};
        float* g = p.G + (size_t)(q * 4) * p.Npad + (pos_s[ef] & 0x7fffffffu);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int j = q * 4 + t;
            if (j < k) {
                const float ej = XV ? __fmul_rn(v[t], x) : v[t];
                float a = __fsub_rn(__fmul_rn(d, Sq[t]), __fmul_rn(d, ej));
                if (XV) a = __fmul_rn(a, x);
                g[(size_t)t * p.Npad] = a;
            } else if (j == k) {
                g[(size_t)t * p.Npad] = XV ? __fmul_rn(d, x) : d;
            }
        }
    }
    FMB_TS(6);
}

// posflag[perm[i]] = i | (row of sorted position i is hit more than once ? 0x80000000 : 0); optionally the list of the
// runs of >= 2 entries {first position, key, entries of the run among its first 32 positions, 0} and their number
// (*run_count zeroed by the caller).  Used behind the generic sort; the per-field sorts do this in their own tail
// (radix_sort.cu sort_tail).
__global__ void __launch_bounds__(256) pos_flags_kernel(const int32_t* __restrict__ skeys, const int32_t* __restrict__ perm,
                                                        int64_t N, uint32_t* __restrict__ posflag, int4* __restrict__ run_list,
                                                        uint32_t* __restrict__ run_count, int cap) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    int32_t key = -1;
    bool start = false;
    if (i < N) {
        key = __ldg(skeys + i);
        const int32_t kprev = i > 0 ? __ldg(skeys + i - 1) : -1;
        const int32_t knext = i + 1 < N ? __ldg(skeys + i + 1) : -1;
        const bool multi = key == kprev || key == knext;
        start = multi && key != kprev;
        posflag[__ldg(perm + i)] = (uint32_t)i | (multi ? 0x80000000u : 0u);
    }
    if (!run_list) return;
    const unsigned m = __ballot_sync(0xffffffffu, start);
    if (!m) return;
    // long runs (>= 128 entries) are listed downwards from the end of the segment and counted in run_count[1]
    const bool lng = start && i + 127 < N && __ldg(skeys + i + 127) == key;
    const unsigned ml = __ballot_sync(0xffffffffu, lng), ms = m & ~ml;
    const int lane = threadIdx.x & 31;
    uint32_t base = 0, basel = 0;
    if (ms) { const int leader = __ffs(ms) - 1; if (lane == leader) base = atomicAdd(run_count, (uint32_t)__popc(ms)); base = __shfl_sync(0xffffffffu, base, leader); }
    if (ml) { const int leader = __ffs(ml) - 1; if (lane == leader) basel = atomicAdd(run_count + 1, (uint32_t)__popc(ml)); basel = __shfl_sync(0xffffffffu, basel, leader); }
    if (start) {
        int n0 = 1;
        bool more = true;
        for (int c = 0; c < 4 && more; ++c) {          // eight keys per round trip
            int32_t kk[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) { const int64_t q = i + 1 + c * 8 + u; kk[u] = q < N ? __ldg(skeys + q) : -1; }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (more && c * 8 + u < 31 && kk[u] == key) ++n0; else more = false;
            }
        }
        const uint32_t lt = (1u << lane) - 1u;
        const int4 e4 = make_int4((int)i, key, n0, lng ? 1 : 0);
        if (lng) run_list[(size_t)cap - 1 - (basel + __popc(ml & lt))] = e4;
        else run_list[base + __popc(ms & lt)] = e4;
    }
}

static int ilog2_ceil(int x) { int l = 0; while ((1 << l) < x) ++l; return l; }

}  // namespace

static int g_step_dbg = 0;
static long long* g_step_tdbg = nullptr;
FMB_API void fmb_debug_set_step_timestamps(long long* dev) { g_step_tdbg = dev; }
// debug hook (not in the public header): timing attribution of the fused kernel's phases
FMB_API void fmb_debug_set_step_flags(int f) { g_step_dbg = f; }

// host-side handle of the fused kernel, for graph-node identification in session.cu (arguments 0..3 are ids, xv, y, posflag)
typedef void (*fused_fn_t)(const int32_t*, const float*, const float*, const uint32_t*, StepParams);
static fused_fn_t fused_fn(int cu, bool xv, int mode) {
#define FMB_FUSED_ROW(C, X) {fm_step_fused_kernel<C, X, 0>, fm_step_fused_kernel<C, X, 1>, fm_step_fused_kernel<C, X, 2>, \
                             fm_step_fused_kernel<C, X, 3>}
    static const fused_fn_t tab[2][2][4] = {{FMB_FUSED_ROW(0, false), FMB_FUSED_ROW(0, true)},
                                            {FMB_FUSED_ROW(3, false), FMB_FUSED_ROW(3, true)}};
#undef FMB_FUSED_ROW
    return tab[cu == 3][xv][mode];
}
// is `fn` one of the fused kernel's instantiations?  (graph-node identification in session.cu)
FMB_API int fmb_is_fused_kernel_fn(const void* fn) {
    for (int c = 0; c < 2; ++c)
        for (int x = 0; x < 2; ++x)
            for (int m = 0; m < 4; ++m)
                if (fn == (const void*)fused_fn(c ? 3 : 0, x != 0, m)) return 1;
    return 0;
}
FMB_API const void* fmb_pos_flags_kernel_fn(void) { return (const void*)pos_flags_kernel; }

// per-entry sorted position + multi-hit flag from the stable sort's output (fmb_sort_fields / fmb_sort_segment);
// _ex: also the run list for fmb_fm_backward_runs_list, as ONE segment (rl->nseg == 1, seg_cap >= N/2) whose counters
// rl->seg_count[0..1] (short, long runs) the caller zeroes beforehand (this kernel appends with atomics; the per-field
// sorts need neither)
struct fmb_runlist_t { int32_t* entries; uint32_t* seg_count; int nseg, seg_cap; };   // include/fmb200.h
FMB_API int fmb_pos_flags_ex(const int32_t* sorted_keys, const int32_t* perm, int64_t N, uint32_t* posflag,
                             const fmb_runlist_t* rl, cudaStream_t stream) {
    FMB_CHECK_ARG(sorted_keys && perm && posflag && N > 0 && N < ((int64_t)1 << 31), "fmb_pos_flags: bad arguments");
    FMB_CHECK_ARG(!rl || (rl->entries && rl->seg_count && rl->nseg == 1 && rl->seg_cap >= N / 2),
                  "fmb_pos_flags: the run list must be one segment of at least N/2 entries");
    int32_t* run_list = rl ? rl->entries : nullptr;
    uint32_t* run_count = rl ? rl->seg_count : nullptr;
    pos_flags_kernel<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(sorted_keys, perm, N, posflag,
                                                                      reinterpret_cast<int4*>(run_list), run_count, rl ? rl->seg_cap : 0);
    FMB_CHECK_LAUNCH("pos_flags_kernel");
    return FMB_OK;
}
FMB_API int fmb_pos_flags(const int32_t* sorted_keys, const int32_t* perm, int64_t N, uint32_t* posflag,
                          cudaStream_t stream) {
    return fmb_pos_flags_ex(sorted_keys, perm, N, posflag, nullptr, stream);
}

// Forward + loss + single-hit row updates + staging of multi-hit contributions (see file header).
//   posflag [B*F]: output of fmb_pos_flags for THIS batch's ids;  G: workspace of fmb_bwd_workspace_bytes(B*F, k)
//   bytes, handed to fmb_fm_backward_runs afterwards;  delta/lossv [B]: per-sample gradient and loss (inputs of
//   fmb_finish_step).  mode as in fmb_fm_backward_update.
struct fmb_ftrl_t { float* zn; float* bias_zn; float beta, l1, l2; };   // include/fmb200.h
struct fmb_adagrad_t { float* sums; float* bias_sum; float* mlp_sums; float eps; };   // include/fmb200.h

FMB_API int fmb_fm_step_fused_ex(const int32_t* ids, const float* xv, const float* y, float* table, const float* bias,
                                 const uint32_t* posflag, int B, int F, int k, int loss_kind, float lr, int mode,
                                 const fmb_ftrl_t* ftrl, float* delta, float* lossv, void* ws, size_t ws_bytes,
                                 cudaStream_t stream) {
    FMB_CHECK_ARG(ids && y && table && bias && posflag && delta && lossv && ws, "fmb_fm_step_fused: null pointer");
    FMB_CHECK_ARG(B > 0 && F > 0 && F < 512 && k > 0 && k <= 124, "fmb_fm_step_fused: bad shape B=%d F=%d k=%d", B, F, k);
    FMB_CHECK_ARG(loss_kind == 0 || loss_kind == 1, "fmb_fm_step_fused: unknown loss kind %d", loss_kind);
    FMB_CHECK_ARG(mode == 0 || mode == 1 || (mode == 2 && ftrl && ftrl->zn) ||
                  (mode == 3 && ftrl && reinterpret_cast<const fmb_adagrad_t*>(ftrl)->sums),
                  "fmb_fm_step_fused: unknown update mode %d (mode 2 needs the FTRL state, mode 3 the Adagrad state)", mode);
    const int64_t N = (int64_t)B * F;
    if (ws_bytes < fmb_bwd_workspace_bytes(N, k)) { fmb_set_error("fmb_fm_step_fused: workspace too small"); return FMB_ERR_WS; }
    StepParams p;
    p.table = table; p.bias = bias;
    p.B = B; p.F = F; p.k = k; p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4);
    p.cu = (k + 1 + 3) / 4; p.ql_log = ilog2_ceil(p.cu); p.jl_log = ilog2_ceil(p.kp4);
    p.mF = fmb_div_magic((unsigned)F); p.mcu = fmb_div_magic((unsigned)p.cu);
    p.loss_kind = loss_kind; p.mode = mode; p.lr = lr; p.astep = -(lr / 0.1f);
    p.delta = delta; p.lossv = lossv;
    p.G = (float*)ws; p.Npad = (N + 3) / 4 * 4 + 64;
    p.dbg = g_step_dbg;
    p.ftrl.zn = nullptr; p.ftrl.bias_zn = nullptr; p.ftrl.beta = p.ftrl.l1 = p.ftrl.l2 = 0.f;
    if (mode == 2) { p.ftrl.zn = ftrl->zn; p.ftrl.bias_zn = ftrl->bias_zn; p.ftrl.beta = ftrl->beta; p.ftrl.l1 = ftrl->l1; p.ftrl.l2 = ftrl->l2; }
    if (mode == 3) { const fmb_adagrad_t* a = reinterpret_cast<const fmb_adagrad_t*>(ftrl); p.ada.sums = a->sums; p.ada.bias_sum = a->bias_sum; p.ada.eps = a->eps; }
    p.tdbg = g_step_tdbg;
    int SB = 256 >> p.jl_log;
    if (SB < 4) SB = 4;
    if (SB > 32) SB = 32;
    auto bytes = [&](int sb) {
        return sizeof(float) * ((size_t)sb * F * p.cu * 4 + (size_t)4 * sb * F + (size_t)sb * k + (size_t)sb * p.cu * 4 + sb);
    };
    while (SB > 1 && bytes(SB) > 48 * 1024) SB >>= 1;
    // at least ~6 tiles per SM when the batch allows it: the tiles of an SM are then in different phases (gather, reduce,
    // update) at any time and the 148 SMs finish together (8 192 samples: 1 024 tiles of 8 instead of 512 of 16, measured
    // 64 instead of 75 us per step, profiles/r2_sweep_tile.txt)
    // ... and 8-sample tiles at ANY batch size: 20.7 KB per CTA keeps 8 CTAs (64 warps) per SM resident instead of 5 with
    // 16-sample tiles; the kernel is latency-bound (55 % "no eligible warp" at B = 65 536 with 16-sample tiles,
    // profiles/r2_final3_fused_ncu_summary.txt): measured 158.0 vs 164.1 us per launch and 363 vs 391 us per step there
    while (SB > 8) SB >>= 1;
    {   // experiment knob: FMB_STEP_SB caps the samples per tile
        static int cap = -1;
        if (cap < 0) { const char* e = getenv("FMB_STEP_SB"); cap = e ? atoi(e) : 0; }
        if (cap > 0 && SB > cap) SB = cap;
    }
    FMB_CHECK_ARG(bytes(SB) <= 200 * 1024, "fmb_fm_step_fused: F*k too large for one sample tile (F=%d k=%d: %zu bytes > 200 KB)",
                  F, k, bytes(SB));
    p.SB = SB;
    const fused_fn_t fn = fused_fn(p.cu, xv != nullptr, mode);
    if (bytes(SB) > 48 * 1024) cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    fn<<<(B + SB - 1) / SB, 256, bytes(SB), stream>>>(ids, xv, y, posflag, p);
    FMB_CHECK_LAUNCH("fm_step_fused_kernel");
    return FMB_OK;
}

FMB_API int fmb_fm_step_fused(const int32_t* ids, const float* xv, const float* y, float* table, const float* bias,
                              const uint32_t* posflag, int B, int F, int k, int loss_kind, float lr, int mode,
                              float* delta, float* lossv, void* ws, size_t ws_bytes, cudaStream_t stream) {
    return fmb_fm_step_fused_ex(ids, xv, y, table, bias, posflag, B, F, k, loss_kind, lr, mode, nullptr, delta, lossv, ws,
                                ws_bytes, stream);
}
