// shard3.cu -- the row-sharded multi-GPU FM step (SURVEY.md 8e; BASELINE.json configs[4]) as ONE kernel per step.
//
// sharded.cu runs a step as three dependent kernels per rank -- partial forward (gathers the owned rows), combine, backward
// (gathers the owned rows AGAIN) -- with a kernel-wide epoch flag between them: 139 us of kernels + 75 us of waits at 8 GPUs
// against 41 us for the whole single-GPU step.  Here a CTA owns a TILE of SB consecutive samples of one source rank and keeps
// the rows it owns for them in shared memory across both exchanges:
//
//   P0  ids of the tile (coalesced rows of the transposed ids), ownership test, compact list of the owned entries in
//       (sample, field) order, their sorted positions / multi-hit flags from the owner sort (one step ahead)
//   P1  gather the owned rows (cp.async, 16 B per request, all in flight)
//   P2  per sample: S, Q, first over the owned fields in field order                 (arithmetic of shard_partial_forward)
//   P3  store the tile's partials into the SAMPLE OWNER's recv, publish the tile's flag there      (peer stores over NVLink)
//   P4  (tiles of my own samples) wait for the G partials of the tile, fold in owner order, logit, loss, delta
//       (arithmetic of shard_combine), store the context rows into every rank's ctx_all, publish the tile's flag everywhere
//   P5  wait for the tile's context
//   P6  rows hit once in the global batch: update from the shared-memory copy; the others: stage the contribution at the
//       entry's sorted position for the run kernel                       (arithmetic of fm_bwd_entry1 / fm_step_fused)
//
// followed by the run kernel (fm_backward.cu) and the bias step.  Flags are per TILE (uint32 epochs in symmetric memory,
// never reset): a tile waits only for the tiles that hold the same samples on the other ranks, not for whole kernels.
// Progress: tile t needs tile t of every rank to have STARTED; CTAs are dispatched in blockIdx order, so the resident
// window of every rank covers the same tiles.  Every wait is bounded and raises the error word instead of hanging.
// Same values in the same order as sharded.cu's path: results are bit-identical to it (tests/test_sharded3.py).
#include "fmb_common.cuh"
#include <cstdlib>

namespace {

struct PeerPtrs3 { void* p[8]; };

struct Step3Params {
    const int32_t* idsT_all;     // [G][F][B]
    float* table;                // local rows [R_local + 1][rowp]
    const float* bias;
    const float* y;              // [B] labels of MY samples
    const uint32_t* posflag;     // [F][G*B]: sorted position | multi-hit flag of the entries this rank owns
    int G, glog, me, B, F, k, rowp, kp4, cu, PW, CW;
    int SB, sb_log, cap_e, T, Tl, jl_log;
    uint32_t mF, mcu;
    int loss_kind, mode;
    float lr, astep;
    float* Gst;                  // [k+1][Npad] staged contributions
    int64_t Npad;
    PeerPtrs3 recv, ctx, tflags; // rank r's recv [G][B][PW], ctx_all [G*B][CW], tile flags uint32 [2*T]
    const float* recv_local;
    const float* ctx_local;
    const uint32_t* tflags_local;
    const uint32_t* epoch;       // this step's epoch is *epoch + 1 (bumped by shard3_bump_kernel behind the step)
    int* error;                  // 16 + phase on a time-out, 32 on a tile's entry-capacity overflow
    long long* tdbg;             // debug only: per-tile phase timestamps [T][8] (globaltimer ns), else NULL
};

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
    unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;\n" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ bool wait_flag(const uint32_t* f, uint32_t e) {
    for (long long spin = 0; spin < (1ll << 24); ++spin) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(f) : "memory");
        if ((int32_t)(v - e) >= 0) return true;
        if (spin > 64) __nanosleep(64);
    }
    return false;
}

template <int CU>
__global__ void __launch_bounds__(256, 7) shard_step_fused_kernel(Step3Params p) {
    extern __shared__ __align__(16) float smem[];
    const int F = p.F, k = p.k, SB = p.SB, kp4 = p.kp4, PW = p.PW, CW = p.CW, cap = p.cap_e;
    constexpr int rp = CU * 4;
    float* rows_s = smem;                                           // [cap][rp]; P0: the tile's ids [F][SB+1]
    int32_t* sid = reinterpret_cast<int32_t*>(smem);
    float* ctx_s = rows_s + (size_t)cap * rp;                       // [SB][CW] context rows of the tile's samples
    int32_t* lrow_s = reinterpret_cast<int32_t*>(ctx_s + SB * CW);  // [cap] local row
    uint32_t* pos_s = reinterpret_cast<uint32_t*>(lrow_s + cap);    // [cap] sorted position | multi-hit flag
    uint16_t* ent_s = reinterpret_cast<uint16_t*>(pos_s + cap);     // [cap] sample << 8 | field
    uint16_t* list_s = ent_s + cap;                                 // [cap] rows hit once from the front, the others from the back
    uint16_t* start_s = list_s + cap;                               // [SB + 1] first entry of every sample
    uint16_t* cnt_s = start_s + SB + 2;                             // [niter + 1]
    __shared__ int n_single, n_multi, n_ent;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = blockIdx.x, o = t % p.G, tl = t / p.G;            // sample owner of the tile, tile index among its tiles
    const int b0 = tl * SB;                                         // first sample (local index on rank o)
    const uint32_t e_now = *p.epoch + 1u;
    const int64_t GB = (int64_t)p.G * p.B;
    if (threadIdx.x == 0) { n_single = 0; n_multi = 0; }
#define S3_TS(i) do { if (p.tdbg && threadIdx.x == 0) { unsigned long long t_; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_)); p.tdbg[(size_t)blockIdx.x * 8 + (i)] = (long long)t_; } } while (0)
    S3_TS(0);

    // ---- P0a: the tile's ids, coalesced rows of idsT_all[o]
    {
        const int32_t* slab = p.idsT_all + (size_t)o * F * p.B + b0;
        for (int i = threadIdx.x; i < F * SB; i += 256) {
            const int f = i >> p.sb_log, s = i & (SB - 1);
            sid[f * (SB + 1) + s] = __ldg(slab + (size_t)f * p.B + s);
        }
    }
    __syncthreads();
    // ---- P0b: ownership, counted per 32 (sample, field) pairs in sample-major order
    const int npairs = SB * F, niter = (npairs + 31) >> 5;
    const uint32_t lt = (1u << lane) - 1u;
    for (int it = warp; it < niter; it += 8) {
        const int i = it * 32 + lane;
        bool own = false;
        if (i < npairs) {
            const int s = fmb_div_by_magic((unsigned)i, p.mF), f = i - s * F;
            own = (sid[f * (SB + 1) + s] & (p.G - 1)) == p.me;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, own);
        if (lane == 0) cnt_s[it] = (uint16_t)__popc(bal);
    }
    __syncthreads();
    if (warp == 0) {                                                // exclusive scan of the counts
        int carry = 0;
        for (int c0 = 0; c0 < niter; c0 += 32) {
            const int v = c0 + lane < niter ? (int)cnt_s[c0 + lane] : 0;
            int inc = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= d) inc += u; }
            if (c0 + lane < niter) cnt_s[c0 + lane] = (uint16_t)(carry + inc - v);
            carry += __shfl_sync(0xffffffffu, inc, 31);
        }
        if (lane == 0) {
            if (carry > cap) { atomicExch(p.error, 32); carry = cap; }
            n_ent = carry;
            start_s[SB] = (uint16_t)carry;
        }
    }
    __syncthreads();
    // ---- P0c: the entry list in (sample, field) order; sorted positions; lists of the rows hit once / several times
    for (int it = warp; it < niter; it += 8) {
        const int i = it * 32 + lane;
        bool own = false;
        int s = 0, f = 0;
        int32_t gid = 0;
        if (i < npairs) {
            s = fmb_div_by_magic((unsigned)i, p.mF); f = i - s * F;
            gid = sid[f * (SB + 1) + s];
            own = (gid & (p.G - 1)) == p.me;
        }
        const unsigned bal = __ballot_sync(0xffffffffu, own);
        const int idx = (int)cnt_s[it] + __popc(bal & lt);
        if (i < npairs && f == 0) start_s[s] = (uint16_t)min(idx, cap);
        uint32_t pf = 0;
        const bool keep = own && idx < cap;
        if (keep) pf = __ldg(p.posflag + (size_t)f * GB + (size_t)o * p.B + b0 + s);
        const unsigned ms = __ballot_sync(0xffffffffu, keep && !(pf >> 31));
        const unsigned mm = __ballot_sync(0xffffffffu, keep && (pf >> 31));
        int bs = 0, bm = 0;
        if (lane == 0) { bs = atomicAdd(&n_single, __popc(ms)); bm = atomicAdd(&n_multi, __popc(mm)); }
        bs = __shfl_sync(0xffffffffu, bs, 0);
        bm = __shfl_sync(0xffffffffu, bm, 0);
        if (keep) {
            lrow_s[idx] = gid >> p.glog;
            ent_s[idx] = (uint16_t)((s << 8) | f);
            pos_s[idx] = pf;
            if (pf >> 31) list_s[cap - 1 - (bm + __popc(mm & lt))] = (uint16_t)idx;
            else list_s[bs + __popc(ms & lt)] = (uint16_t)idx;
        }
    }
    __syncthreads();
    S3_TS(1);
    const int ne = n_ent;
    // ---- P1: gather the owned rows (the ids are dead: rows_s takes their place)
    {
        const int q = threadIdx.x & 3;
        if (q < CU)
            for (int idx = threadIdx.x >> 2; idx < ne; idx += 64)
                cp_async16(rows_s + (size_t)idx * rp + q * 4, p.table + (size_t)lrow_s[idx] * p.rowp + q * 4);
        asm volatile("cp.async.commit_group;\n" ::);
        asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    }
    __syncthreads();
    S3_TS(2);
    // ---- P2 + P3: partial sums over the owned fields in field order, stored straight into recv of the samples' owner
    // (the lanes of a sample write 4*(k+1) contiguous bytes each for S and Q); then the tile's flag there
    const int jl = 1 << p.jl_log, j = threadIdx.x & (jl - 1);
    for (int s = threadIdx.x >> p.jl_log; s < SB; s += 256 >> p.jl_log) {
        float* out = static_cast<float*>(p.recv.p[o]) + ((size_t)p.me * p.B + b0 + s) * PW;
        float S = 0.f, Q = 0.f;
        if (j <= k) {
            const int u0 = start_s[s], u1 = start_s[s + 1];
            for (int u = u0; u < u1; ++u) {
                const float e = rows_s[(size_t)u * rp + j];       // x == 1
                S = __fadd_rn(S, e);
                Q = __fadd_rn(Q, __fmul_rn(e, e));
            }
        }
        // 16-byte stores (4-byte stores over NVLink made this phase 11 us): lane 4q collects components 4q..4q+3 of S and
        // of Q from its neighbours; padding components (k <= j < kp4) are zero; lane k holds the first-order sum
        const float first = __shfl_sync(0xffffffffu, S, (lane & ~(jl - 1)) + k);
        const float Sv = j < k ? S : 0.f, Qv = j < k ? Q : 0.f;
        const float S1 = __shfl_down_sync(0xffffffffu, Sv, 1), S2 = __shfl_down_sync(0xffffffffu, Sv, 2), S3 = __shfl_down_sync(0xffffffffu, Sv, 3);
        const float Q1 = __shfl_down_sync(0xffffffffu, Qv, 1), Q2 = __shfl_down_sync(0xffffffffu, Qv, 2), Q3 = __shfl_down_sync(0xffffffffu, Qv, 3);
        if ((j & 3) == 0 && j < kp4) {
            *reinterpret_cast<float4*>(out + j) = make_float4(Sv, S1, S2, S3);
            *reinterpret_cast<float4*>(out + kp4 + j) = make_float4(Qv, Q1, Q2, Q3);
        }
        if (j == 1) *reinterpret_cast<float4*>(out + 2 * kp4) = make_float4(first, 0.f, 0.f, 0.f);
    }
    __syncthreads();
    // release at system scope: the barrier orders the CTA's stores before thread 0's release (no separate fence.sc.sys)
    if (threadIdx.x == 0) st_release_sys(static_cast<uint32_t*>(p.tflags.p[o]) + (size_t)p.me * p.Tl + tl, e_now);
    S3_TS(3);
    // ---- P4: my own samples: fold the G partials in owner order, logit, loss, delta; context to every rank
    if (o == p.me) {
        if ((int)threadIdx.x < p.G)
            if (!wait_flag(p.tflags_local + (size_t)threadIdx.x * p.Tl + tl, e_now)) atomicExch(p.error, 16 + 4);
        __syncthreads();
        for (int s = threadIdx.x >> p.jl_log; s < SB; s += 256 >> p.jl_log) {
            const float* r0 = p.recv_local + (size_t)(b0 + s) * PW;
            const size_t ostride = (size_t)p.B * PW;
            float bi = 0.f, sf = 0.f;
            if (j < kp4) {
                float Sj = 0.f, Qj = 0.f;
                for (int g = 0; g < p.G; ++g) {
                    Sj = __fadd_rn(Sj, __ldcg(r0 + g * ostride + j));
                    Qj = __fadd_rn(Qj, __ldcg(r0 + g * ostride + kp4 + j));
                }
                ctx_s[s * CW + j] = Sj;
                bi = __fmul_rn(__fsub_rn(__fmul_rn(Sj, Sj), Qj), 0.5f);
            } else if (j == kp4) {
                for (int g = 0; g < p.G; ++g) sf = __fadd_rn(sf, __ldcg(r0 + g * ostride + 2 * kp4));
            }
            // sum_j bi_j in ATen's order: every lane of the sample's group walks the same sequence (the loop shape depends
            // on k only), reading component jj from the lane that holds it
            const int gbase = lane & ~(jl - 1);
            const float sum_bi = fmb::aten_row_sum_small([&](int jj) { return __shfl_sync(0xffffffffu, bi, gbase + jj); }, k);
            const float sum_first = __shfl_sync(0xffffffffu, sf, gbase + kp4);
            if (j == 0) {
                const int b = b0 + s;
                const float z = __fadd_rn(__fadd_rn(sum_first, sum_bi), __ldg(p.bias));
                float lossv, d;   // sample b of rank `me` is element me*B + b of the global batch (torch.sigmoid is position-dependent)
                fmb::bce_logits_value_grad(p.loss_kind, z, p.y[b], p.me * p.B + b, p.G * p.B, lossv, d);
                float* c = ctx_s + s * CW + kp4;
                c[0] = d; c[1] = lossv; c[2] = z; c[3] = 0.f;
            }
        }
        __syncthreads();
        const int n4 = SB * CW / 4;
        const size_t o4 = ((size_t)p.me * p.B + b0) * CW / 4;
        for (int i = threadIdx.x; i < n4; i += 256) {
            const float4 v = reinterpret_cast<const float4*>(ctx_s)[i];
            for (int r = 0; r < p.G; ++r) static_cast<float4*>(p.ctx.p[r])[o4 + i] = v;
        }
        __syncthreads();
        if ((int)threadIdx.x < p.G) st_release_sys(static_cast<uint32_t*>(p.tflags.p[threadIdx.x]) + p.T + t, e_now);
    }
    S3_TS(4);
    // ---- P5: the tile's context (S, delta) from the samples' owner
    if (threadIdx.x == 0)
        if (!wait_flag(p.tflags_local + p.T + t, e_now)) atomicExch(p.error, 16 + 5);
    __syncthreads();
    if (o != p.me) {
        const int n4 = SB * CW / 4;
        const float4* src = reinterpret_cast<const float4*>(p.ctx_local + ((size_t)o * p.B + b0) * CW);
        for (int i = threadIdx.x; i < n4; i += 256) reinterpret_cast<float4*>(ctx_s)[i] = __ldcg(src + i);
        __syncthreads();
    }
    S3_TS(5);
    // ---- P6a: rows hit once in the global batch: gradient = 0 + contribution, update from the shared-memory copy
    const int ns = n_single, nm = n_multi;
    for (int it = threadIdx.x; it < ns * CU; it += 256) {
        const int li = it / CU, q = it - li * CU;
        const int idx = list_s[li];
        const int s = ent_s[idx] >> 8;
        const float d = ctx_s[s * CW + kp4];
        if (d == 0.0f) continue;       // exact: every gradient is +0 and both update rules return p (fm_step.cu, phase 4a)
        const float4 v4 = *reinterpret_cast<const float4*>(rows_s + (size_t)idx * rp + q * 4);
        float4 S4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q * 4 < kp4) S4 = *reinterpret_cast<const float4*>(ctx_s + s * CW + q * 4);
        const float Sq[4] = {S4.x, S4.y, S4.z, S4.w};
        const float v[4] = {v4.x, v4.y, v4.z, v4.w};
        float o4[4];
        bool moved = false;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int jj = q * 4 + u;
            float a = 0.f;
            if (jj < k) a = __fsub_rn(__fmul_rn(d, Sq[u]), __fmul_rn(d, v[u]));
            else if (jj == k) a = d;
            const float g = __fadd_rn(0.f, a);
            o4[u] = jj <= k ? fmb::apply_update_a(v[u], g, p.lr, p.astep, p.mode) : v[u];
            moved |= __float_as_int(o4[u]) != __float_as_int(v[u]);
        }
        if (moved) *reinterpret_cast<float4*>(p.table + (size_t)lrow_s[idx] * p.rowp + q * 4) = make_float4(o4[0], o4[1], o4[2], o4[3]);
    }
    // ---- P6b: the others: contribution at the entry's sorted position (the run kernel sums each run in sample order)
    for (int it = threadIdx.x; it < nm * CU; it += 256) {
        const int li = it / CU, q = it - li * CU;
        const int idx = list_s[cap - 1 - li];
        const int s = ent_s[idx] >> 8;
        const float d = ctx_s[s * CW + kp4];
        const float4 v4 = *reinterpret_cast<const float4*>(rows_s + (size_t)idx * rp + q * 4);
        float4 S4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (q * 4 < kp4) S4 = *reinterpret_cast<const float4*>(ctx_s + s * CW + q * 4);
        const float Sq[4] = {S4.x, S4.y, S4.z, S4.w};
        const float v[4] = {v4.x, v4.y, v4.z, v4.w};
        float* g = p.Gst + (size_t)(q * 4) * p.Npad + (pos_s[idx] & 0x7fffffffu);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int jj = q * 4 + u;
            if (jj < k) g[(size_t)u * p.Npad] = __fsub_rn(__fmul_rn(d, Sq[u]), __fmul_rn(d, v[u]));
            else if (jj == k) g[(size_t)u * p.Npad] = d;
        }
    }
    S3_TS(6);
}

__global__ void shard3_bump_kernel(uint32_t* epoch) { *epoch += 1u; }

static long long* g_s3_tdbg = nullptr;
static int ilog2_exact3(int x) { int l = 0; while ((1 << l) < x) ++l; return (1 << l) == x ? l : -1; }
static int ilog2_ceil3(int x) { int l = 0; while ((1 << l) < x) ++l; return l; }
static int64_t npad3(int64_t N) { return (N + 3) / 4 * 4 + 64; }   // == bwd_npad (fm_backward.cu)

}  // namespace

extern "C" size_t fmb_bwd_workspace_bytes(int64_t, int);
// debug hook (not in the public header): per-tile phase timestamps of the fused sharded step
FMB_API void fmb_debug_set_shard3_timestamps(long long* dev) { g_s3_tdbg = dev; }

// tile geometry of the fused sharded step: samples per tile (8 per rank: every rank's tile holds ~8*F owned entries whatever
// G is), tiles per step, tile-flag words (2 * tiles, uint32, zero-initialised, in peer-mapped memory).  0 when the shape is
// not supported by this path (G a power of two <= 8, B a multiple of 8*G, k + 1 <= 12 floats per row chunked by 3, F <= 255).
FMB_API int fmb_shard3_tiles(int G, int B, int F, int k) {
    if (G < 1 || G > 8 || ilog2_exact3(G) < 0 || B <= 0 || B % (8 * G) != 0 || F < 1 || F > 255 || k < 1 || k > 15) return 0;
    if ((int64_t)G * B > 65536) return 0;
    return (int)((int64_t)G * B / (8 * G));
}

// One step of the row-sharded FM (update_embedding over the global batch of G*B samples), fused: see the file header.
//   idsT_all [G][F][B] (this batch, every rank's slab landed), posflag [F][G*B] + the owner sort's workspace contract
//   (fmb_shard_sort_fields_pf with the same cap), y [B] my labels, ws = staging of fmb_bwd_workspace_bytes(F*cap, k) bytes
//   (handed to fmb_fm_backward_runs_list afterwards).  recv / ctx / tflags: HOST arrays of G device pointers (entry r = where
//   this device maps rank r's buffer); *_local = my own copies; epoch_dev: uint32 step counter in ordinary device memory
//   (fmb_shard3_bump increments it behind the step); error_dev: see Step3Params.
FMB_API int fmb_shard3_step(const int32_t* idsT_all, float* table_local, const float* bias, const float* y,
                            const uint32_t* posflag, int G, int me, int B, int F, int k, int cap, int loss_kind, float lr,
                            int mode, void* ws, size_t ws_bytes, void* const* recv_peers, void* const* ctx_peers,
                            void* const* tflag_peers, const float* recv_local, const float* ctx_local,
                            const uint32_t* tflags_local, const uint32_t* epoch_dev, int* error_dev, cudaStream_t stream) {
    FMB_CHECK_ARG(idsT_all && table_local && bias && y && posflag && ws && recv_peers && ctx_peers && tflag_peers && recv_local &&
                  ctx_local && tflags_local && epoch_dev && error_dev, "fmb_shard3_step: null pointer");
    const int T = fmb_shard3_tiles(G, B, F, k);
    FMB_CHECK_ARG(T > 0 && me >= 0 && me < G && cap > 0, "fmb_shard3_step: unsupported shape G=%d B=%d F=%d k=%d", G, B, F, k);
    FMB_CHECK_ARG(mode == 0 || mode == 1, "fmb_shard3_step: unknown update mode %d", mode);
    const int64_t N = (int64_t)F * cap;
    if (ws_bytes < fmb_bwd_workspace_bytes(N, k)) { fmb_set_error("fmb_shard3_step: workspace too small"); return FMB_ERR_WS; }
    Step3Params p;
    memset(&p, 0, sizeof(p));
    p.idsT_all = idsT_all; p.table = table_local; p.bias = bias; p.y = y; p.posflag = posflag;
    p.G = G; p.glog = ilog2_exact3(G); p.me = me; p.B = B; p.F = F; p.k = k;
    p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4); p.cu = (k + 1 + 3) / 4;
    p.PW = 2 * p.kp4 + 4; p.CW = p.kp4 + 4;
    p.SB = 8 * G; p.sb_log = ilog2_exact3(p.SB); p.T = T; p.Tl = T / G; p.jl_log = ilog2_ceil3(p.kp4 + 1);
    // entry capacity of a tile.  A tile holds 8*F owned entries on average whatever G is; the worst case is SB*F (every
    // entry of the tile owned by this rank).  When the worst case fits the shared memory of 7 resident CTAs per SM it is
    // used; otherwise 1.4x the mean + 16 (FMB_SHARD3_CAP overrides): ids whose hot rows concentrate on one rank beyond that
    // raise error 32 (check_exchange) instead of training on silently -- the three-kernel path has no such limit.
    const int niter = (p.SB * F + 31) / 32;
    auto smem_of = [&](int cap_e) {
        return (size_t)cap_e * p.cu * 16 + (size_t)p.SB * p.CW * 4 + (size_t)cap_e * (4 + 4 + 2 + 2) + (size_t)(p.SB + 2 + niter + 2) * 2 + 16;
    };
    {
        const int full = (p.SB * F + 15) / 16 * 16;
        static int forced = -1;
        if (forced < 0) { const char* e = getenv("FMB_SHARD3_CAP"); forced = e ? atoi(e) : 0; }
        if (forced > 0) p.cap_e = (forced + 15) / 16 * 16;
        else if (smem_of(full) <= 32000) p.cap_e = full;
        else p.cap_e = (8 * F * 7 / 5 + 16 + 15) / 16 * 16;
        if (p.cap_e > full) p.cap_e = full;
        const int need = (F * (p.SB + 1) + p.cu * 4 - 1) / (p.cu * 4);   // the tile's ids must fit where the rows go
        if (p.cap_e < need) p.cap_e = (need + 15) / 16 * 16;
    }
    p.mF = fmb_div_magic((unsigned)F); p.mcu = fmb_div_magic((unsigned)p.cu);
    p.loss_kind = loss_kind; p.mode = mode; p.lr = lr; p.astep = -(lr / 0.1f);
    p.Gst = (float*)ws; p.Npad = npad3(N);
    for (int r = 0; r < 8; ++r) {
        p.recv.p[r] = r < G ? recv_peers[r] : nullptr; p.ctx.p[r] = r < G ? ctx_peers[r] : nullptr;
        p.tflags.p[r] = r < G ? tflag_peers[r] : nullptr;
        if (r < G && !(p.recv.p[r] && p.ctx.p[r] && p.tflags.p[r])) { fmb_set_error("fmb_shard3_step: peer pointer %d is null", r); return FMB_ERR_ARG; }
    }
    p.recv_local = recv_local; p.ctx_local = ctx_local; p.tflags_local = tflags_local; p.epoch = epoch_dev; p.error = error_dev;
    p.tdbg = g_s3_tdbg;
    const size_t smem = smem_of(p.cap_e);
    FMB_CHECK_ARG(smem <= 200 * 1024, "fmb_shard3_step: tile too large for shared memory");
    void (*fn)(Step3Params) = nullptr;
    switch (p.cu) {
        case 1: fn = shard_step_fused_kernel<1>; break;
        case 2: fn = shard_step_fused_kernel<2>; break;
        case 3: fn = shard_step_fused_kernel<3>; break;
        default: fn = shard_step_fused_kernel<4>; break;
    }
    if (smem > 48 * 1024) cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    fn<<<T, 256, smem, stream>>>(p);
    FMB_CHECK_LAUNCH("shard_step_fused_kernel");
    return FMB_OK;
}

// the step counter of fmb_shard3_step: +1, on the stream, behind the step
FMB_API int fmb_shard3_bump(uint32_t* epoch_dev, cudaStream_t stream) {
    FMB_CHECK_ARG(epoch_dev, "fmb_shard3_bump: null pointer");
    shard3_bump_kernel<<<1, 1, 0, stream>>>(epoch_dev);
    FMB_CHECK_LAUNCH("shard3_bump_kernel");
    return FMB_OK;
}
