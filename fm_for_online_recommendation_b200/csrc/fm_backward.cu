// fm_backward.cu -- sparse embedding gradient as a deterministic segmented reduce over the sorted
// (row id, entry) list, fused with the per-row parameter update.
//
// Replaces autograd + 2F dense `embedding_dense_backward` + the dense `Adam.step` over all rows
// (models/models_online_deep/fm_adam.py:56-69, deepfm_adam.py:91-117; SURVEY.md 8a A6/A12): only
// the rows a batch touches are read and written.  Per entry (b, f) of row r:
//     e_j   = V_r[j] * x                                     (deepfm_adam.py:60)
//     g_e_j = (g*S_b[j]) - (g*e_j)      g = delta_b (FM scalar path) and/or gvec_b[j] (MLP path)
//     grad V_r[j] += g_e_j * x ;  grad w_r += delta_b * x    summed IN SAMPLE ORDER per row
// then one update per row (fresh-Adam sign step or SGD).  No float atomics anywhere.
//
// Two kernels over the sorted list:
//   fm_bwd_entry_kernel : one 4-lane group per entry (one lane per 16-byte chunk of the row).  A row
//       hit by a single entry of the batch (the common case in large fields) is updated right here
//       from registers; entries of rows hit several times write their contribution to a staging
//       buffer G (L2-resident).
//   fm_bwd_runs_kernel  : one warp per 32 sorted positions finds the runs (>= 2 entries) that START
//       there and sums each run left to right, one lane per component -- the first 32 entries straight
//       from G, longer runs through a 4-stage bulk-copy (TMA) ring in shared memory so the serial fp32
//       chain (the only part that cannot be parallelised without changing the rounding) never waits on L2.
// G is component-major ([component][position], SoA): a lane's chain reads ITS component of consecutive
// entries, so the ring holds one contiguous row per lane and the chain consumes 4 entries per LDS.128
// (the entry-major layout cost one LDS.32 per entry: 64 instructions per 32 entries, 10.6 cycles per entry
// measured with clock64; the add chain itself is 4).
#include "fmb_common.cuh"
#include <cstdlib>
#include <cstring>
#include <cuda.h>   // CUtensorMap (the encoder is fetched through cudaGetDriverEntryPoint: no libcuda link)

namespace {

struct BwdParams {
    const int32_t* skeys;
    const int32_t* perm;
    int64_t N;
    const float* xv;
    float* table;
    int F, k, rowp, kp4;
    int cu;               // 16-byte chunks per row that hold data: ceil((k+1)/4)
    int ql_log;           // log2(lanes per entry), 2^ql_log >= cu
    unsigned long long fmagic;  // ceil(2^fshift / F): b = (e * fmagic) >> fshift, exact for e < N (2^fshift > N*F)
    int fshift;
    const float* S;
    const float* gs;
    int use_fm2;
    const float* gvec;
    float lr;
    int mode;
    int s_pitch;          // row pitch of S / gvec in floats (kp4 unless they live in a gathered context)
    int gs_stride;        // stride of gs in floats
    int32_t key_limit;    // keys >= key_limit are padding (sharded path) and are skipped
    float* G;             // [k+1 (+k)][Npad] staged contributions, component-major: rows 0..k chain A (or the only
                          // chain), rows k+1..2k chain B when both gradient paths are live
    int64_t Npad;         // row pitch of G (positions, multiple of 4, >= N + 64)
    long long* dbg;       // optional per-run timing records (debug builds of bench only), else NULL
    float astep;          // -(lr/0.1f): Adam step size, computed once on the host (same IEEE division)
    // multi-GPU (csrc/shard2.cu): shard_G > 0 = do not update, store the run's partial gradient into the inbox of the
    // row's owner (key % G) at slot [shard_me][position of the run's first entry]
    union {                // the update rule's per-coordinate state (same size as the FTRL state alone)
        fmb::FtrlState ftrl;   // mode 2 only
        fmb::AdagradState ada; // mode 3 only
    };
    int min_run1;          // 1: rows hit once are summed (0 + g) and updated here too (AFM path: nothing updates them earlier)
    float* inbox[8];
    int shard_G, shard_me;
    int64_t shard_N;
    // run-list mode (fm_bwd_runs_kernel<true>): the runs of >= 2 entries as {first sorted position, key, entries among
    // the first 32 positions that belong to the run (2..32), 0}, in any order, in one segment per producer CTA (no global
    // counter, nothing to zero) -- written one step ahead by the sort (radix_sort.cu / fm_step.cu pos_flags_kernel)
    const int4* run_list;          // [run_nseg][run_cap] entries, segment g holds run_segc[g] of them
    const uint32_t* run_segc;
    int run_nseg, run_cap;
    int pdl;                       // 1: launched as a programmatic dependent of the kernel that stages G
};

// update of coordinate c of row `key` from its summed gradient: modes 0 / 1 in registers, mode 3 (Adagrad: ADA, an
// instantiation of its own so that the others stay as they are) also reads and writes the coordinate's sum
template <bool ADA>
__device__ __forceinline__ float row_update(const BwdParams& p, float old, float g, int32_t key, int c) {
    if (ADA) {
        float* sp = p.ada.sums + (size_t)key * p.rowp + c;
        float sv = *sp;
        const float o = fmb::adagrad_update(old, g, sv, p.lr, p.ada.eps);
        *sp = sv;
        return o;
    }
    return fmb::apply_update_a(old, g, p.lr, p.astep, p.mode);
}

// ---------------------------------------------------------------------------------------------
template <bool ADA>
__global__ void __launch_bounds__(256) fm_bwd_entry_kernel(BwdParams p) {
    const int q = threadIdx.x & ((1 << p.ql_log) - 1);
    const int64_t i = (int64_t)blockIdx.x * (256 >> p.ql_log) + (threadIdx.x >> p.ql_log);
    if (i >= p.N || q >= p.cu) return;
    const int32_t key = __ldg(p.skeys + i);
    if (key >= p.key_limit) return;
    const int32_t kprev = i > 0 ? __ldg(p.skeys + i - 1) : -1;
    const int32_t knext = i + 1 < p.N ? __ldg(p.skeys + i + 1) : -1;
    const int32_t e = __ldg(p.perm + i);
    const int b = (int)(((unsigned long long)(unsigned)e * p.fmagic) >> p.fshift);
    const float x = p.xv ? __ldg(p.xv + e) : 1.0f;
    const float d = __ldg(p.gs + (size_t)b * p.gs_stride);
    float* rowptr = p.table + (size_t)key * p.rowp + q * 4;
    const float4 v4 = *reinterpret_cast<const float4*>(rowptr);
    float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), g4 = s4;
    if (q * 4 < p.kp4) {
        s4 = __ldg(reinterpret_cast<const float4*>(p.S + (size_t)b * p.s_pitch + q * 4));
        if (p.gvec) g4 = __ldg(reinterpret_cast<const float4*>(p.gvec + (size_t)b * p.s_pitch + q * 4));
    }
    const float v[4] = {v4.x, v4.y, v4.z, v4.w}, s[4] = {s4.x, s4.y, s4.z, s4.w}, g[4] = {g4.x, g4.y, g4.z, g4.w};
    const bool two = p.use_fm2 && p.gvec;
    float a[4], c[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int j = q * 4 + t;
        a[t] = 0.f; c[t] = 0.f;
        if (j < p.k) {
            const float ej = __fmul_rn(v[t], x);
            if (p.use_fm2) a[t] = __fmul_rn(__fsub_rn(__fmul_rn(d, s[t]), __fmul_rn(d, ej)), x);
            if (p.gvec) c[t] = __fmul_rn(__fsub_rn(__fmul_rn(g[t], s[t]), __fmul_rn(g[t], ej)), x);
        } else if (j == p.k) {
            a[t] = __fmul_rn(d, x);
        }
    }
    if (key != kprev && key != knext) {
        // the only entry of its row: sum = 0 + contribution; update from registers
        float o[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int j = q * 4 + t;
            if (j < p.k) {
                const float gr = two ? __fadd_rn(__fadd_rn(0.f, a[t]), __fadd_rn(0.f, c[t]))
                                     : __fadd_rn(0.f, p.gvec ? c[t] : a[t]);
                o[t] = row_update<ADA>(p, v[t], gr, key, j);
            } else if (j == p.k) {
                o[t] = row_update<ADA>(p, v[t], __fadd_rn(0.f, a[t]), key, j);
            } else {
                o[t] = v[t];
            }
        }
        *reinterpret_cast<float4*>(rowptr) = make_float4(o[0], o[1], o[2], o[3]);
    } else {
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int j = q * 4 + t;
            if (j > p.k) continue;
            if (two) {
                p.G[(size_t)j * p.Npad + i] = a[t];
                if (j < p.k) p.G[(size_t)(p.k + 1 + j) * p.Npad + i] = c[t];
            } else {
                p.G[(size_t)j * p.Npad + i] = (p.gvec && j < p.k) ? c[t] : a[t];
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Thread-per-entry version for rows of at most 4 chunks (k <= 15): the per-entry bookkeeping (three key
// loads, permutation, sample index, delta, feature value) is paid once per entry instead of once per
// 16-byte chunk, which is what made the lane-per-chunk kernel instruction-bound (75 % issue utilisation,
// ~450 instructions per lane: profiles/r1g).  Row and S reads are random per entry either way.
template <int CU, bool ADA>
__global__ void __launch_bounds__(256) fm_bwd_entry1_kernel(BwdParams p) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= p.N) return;
    const int32_t key = __ldg(p.skeys + i);
    if (key >= p.key_limit) return;
    const int32_t kprev = i > 0 ? __ldg(p.skeys + i - 1) : -1;
    const int32_t knext = i + 1 < p.N ? __ldg(p.skeys + i + 1) : -1;
    const int32_t e = __ldg(p.perm + i);
    const int b = (int)(((unsigned long long)(unsigned)e * p.fmagic) >> p.fshift);
    const float x = p.xv ? __ldg(p.xv + e) : 1.0f;
    const float d = __ldg(p.gs + (size_t)b * p.gs_stride);
    float* rowptr = p.table + (size_t)key * p.rowp;
    float v[CU * 4], s[CU * 4], g[CU * 4];
#pragma unroll
    for (int q = 0; q < CU; ++q) {
        const float4 v4 = *reinterpret_cast<const float4*>(rowptr + q * 4);
        v[q * 4] = v4.x; v[q * 4 + 1] = v4.y; v[q * 4 + 2] = v4.z; v[q * 4 + 3] = v4.w;
        float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), g4 = s4;
        if (q * 4 < p.kp4) {
            s4 = __ldg(reinterpret_cast<const float4*>(p.S + (size_t)b * p.s_pitch + q * 4));
            if (p.gvec) g4 = __ldg(reinterpret_cast<const float4*>(p.gvec + (size_t)b * p.s_pitch + q * 4));
        }
        s[q * 4] = s4.x; s[q * 4 + 1] = s4.y; s[q * 4 + 2] = s4.z; s[q * 4 + 3] = s4.w;
        g[q * 4] = g4.x; g[q * 4 + 1] = g4.y; g[q * 4 + 2] = g4.z; g[q * 4 + 3] = g4.w;
    }
    const bool two = p.use_fm2 && p.gvec;
    const bool single = key != kprev && key != knext;
    float o[CU * 4], o2[CU * 4];
#pragma unroll
    for (int j = 0; j < CU * 4; ++j) {
        float a = 0.f, c = 0.f;
        if (j < p.k) {
            const float ej = __fmul_rn(v[j], x);
            if (p.use_fm2) a = __fmul_rn(__fsub_rn(__fmul_rn(d, s[j]), __fmul_rn(d, ej)), x);
            if (p.gvec) c = __fmul_rn(__fsub_rn(__fmul_rn(g[j], s[j]), __fmul_rn(g[j], ej)), x);
        } else if (j == p.k) {
            a = __fmul_rn(d, x);
        }
        if (single) {
            // the only entry of its row: sum = 0 + contribution; update from registers
            if (j < p.k) {
                const float gr = two ? __fadd_rn(__fadd_rn(0.f, a), __fadd_rn(0.f, c)) : __fadd_rn(0.f, p.gvec ? c : a);
                o[j] = row_update<ADA>(p, v[j], gr, key, j);
            } else if (j == p.k) {
                o[j] = row_update<ADA>(p, v[j], __fadd_rn(0.f, a), key, j);
            } else {
                o[j] = v[j];
            }
        } else {
            o[j] = two ? a : ((p.gvec && j < p.k) ? c : a);
            o2[j] = c;
        }
    }
    if (single) {
#pragma unroll
        for (int q = 0; q < CU; ++q)
            *reinterpret_cast<float4*>(rowptr + q * 4) = make_float4(o[q * 4], o[q * 4 + 1], o[q * 4 + 2], o[q * 4 + 3]);
    } else {
#pragma unroll
        for (int j = 0; j < CU * 4; ++j) {
            if (j > p.k) continue;
            p.G[(size_t)j * p.Npad + i] = o[j];          // adjacent threads = adjacent positions: coalesced
            if (two && j < p.k) p.G[(size_t)(p.k + 1 + j) * p.Npad + i] = o2[j];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Ring geometry (template parameters of the run kernel): RING_SE entries per stage, RING_NS stages.  The short-run
// launches use 64 x 4; the launch that takes the LONG runs of the run list (>= 128 entries: the hot rows of the small
// fields, ~180 of a Criteo-shaped batch's 1 900 runs but its whole critical path) uses 128 x 4 and starts the ring at the
// run's first entry: the per-stage costs (mbarrier wait, TMA issue by lane 0, loop control: ~460 cycles) were 7 of the 16
// cycles per entry with 64-entry stages, and the 32-entry direct part in front of the ring cost another 3 600 cycles.
// RING_SEP = RING_SE + 4 floats per lane row of a stage = inner box of the tensor-map copy.  TMA needs
                                       // 16-byte aligned row starts, so a stage starts up to 3 entries early (`mis`);
                                       // the pitch of 4 banks per lane also makes the LDS.128 conflict-free

// ---- mbarrier + TMA helpers -------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"((unsigned)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
// bounded wait: returns false if the phase never completed (never expected; avoids hanging the GPU)
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, unsigned parity) {
    const unsigned a = (unsigned)__cvta_generic_to_shared(bar);
    for (int spin = 0; spin < (1 << 20); ++spin) {
        unsigned ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
        if (ok) return true;
    }
    return false;
}
// 2-D tiled TMA: box [rows][RING_SEP entries] of the component-major staging buffer, starting at (entry x, row y)
__device__ __forceinline__ void tma_g2s_2d(void* smem_dst, const CUtensorMap* tmap, int x, int y, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n" ::"r"(
            (unsigned)__cvta_generic_to_shared(smem_dst)),
        "l"(tmap), "r"(x), "r"(y), "r"((unsigned)__cvta_generic_to_shared(bar))
        : "memory");
}

// LIST = false: one warp per 32 sorted positions, handling the runs that start there (the tower `fit` path, the AFM path and
// the sharded paths: the run list does not exist there).  LIST = true: one warp per entry of the run list, grid-strided:
// the ~2 000 runs of a Criteo-shaped batch are then all in flight at once, where the position-major mapping packed them
// into the first third of the grid (the small fields sort first) and needed two waves of CTAs for them (17 -> 9 us).
// bid / nblocks: this CTA's index among the CTAs running this body, and their number (the run-list launch runs two bodies:
// its first CTAs take the long runs, the others the short ones).  segb_off: offset (floats) of the segment-count prefix in
// dynamic shared memory.  warps_per_block: working warps (the CTA's other warps only help with the prefix).
template <bool LIST, int RING_SE, int RING_NS, bool LONGM, bool ADA>
__device__ __forceinline__ void runs_body(const CUtensorMap& gmap, const BwdParams& p, int warps_per_block, int warp_f, int accs_n,
                                          int ring_comps, unsigned bid, unsigned nblocks, int segb_off) {
    constexpr int RING_SEP = RING_SE + 4;
    extern __shared__ __align__(128) float smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t P0 = ((int64_t)bid * warps_per_block + wib) * 32;
    if (!LIST && P0 >= p.N) return;
    const bool two = p.use_fm2 && p.gvec;
    const int kc = p.k + 1;
    const int nv = kc + (two ? p.k : 0);          // virtual lanes: chain A comps, then chain B comps
    const int stage_f = (ring_comps * RING_SEP + 31) & ~31;   // stages stay 128-byte aligned (TMA destination)
    float* ring = smem + (size_t)wib * warp_f;    // [NS][ring_comps][SEP]
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + RING_NS * stage_f);   // [NS] mbarriers
    float* accs = reinterpret_cast<float*>(bars + RING_NS);                   // [accs_n + 32]

    int32_t k0 = -2, k1 = -2;
    unsigned todo = 0;
    uint32_t lr = 0, ln = 0, lstep = 0;           // LIST: next run of this warp, number of runs, stride
    // exclusive prefix of the segment counts, behind the warps' rings in dynamic shared memory: [run_nseg + 1]
    uint32_t* seg_base = reinterpret_cast<uint32_t*>(smem + segb_off);
    if (LIST) {
        lr = bid * warps_per_block + wib;
        lstep = nblocks * warps_per_block;
        // every CTA scans the segment counts itself (a few hundred words, one L2 round trip -- the same latency as the
        // single global counter it replaces, but no atomics in the producers and no memset in front of them)
        // (the long runs' counts follow the short runs' in run_segc; their entries grow downwards from each segment's end)
        for (int g = threadIdx.x; g < p.run_nseg; g += blockDim.x) seg_base[g] = __ldg(p.run_segc + (LONGM ? p.run_nseg : 0) + g);
        __syncthreads();
        if (wib == 0) {
            uint32_t carry = 0;
            for (int b0 = 0; b0 < p.run_nseg; b0 += 32) {
                const uint32_t v = b0 + lane < p.run_nseg ? seg_base[b0 + lane] : 0u;
                uint32_t inc = v;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
                if (b0 + lane < p.run_nseg) seg_base[b0 + lane] = carry + inc - v;
                carry += __shfl_sync(0xffffffffu, inc, 31);
            }
            if (lane == 0) seg_base[p.run_nseg] = carry;
        }
        __syncthreads();
        const uint32_t total = seg_base[p.run_nseg];
        ln = total;
        if (wib >= warps_per_block) return;
        // launched with programmatic stream serialization behind the fused kernel (session.cu): everything above only
        // reads the sort's outputs; the staged contributions and the rows are complete once the fused grid has finished
        if (p.pdl) asm volatile("griddepcontrol.wait;\n" ::: "memory");
    } else {
        // keys of this warp's 32 positions and of the 32 after them (one memory latency for both)
        const int64_t pos = P0 + lane;
        k0 = pos < p.N ? __ldg(p.skeys + pos) : -2;
        k1 = pos + 32 < p.N ? __ldg(p.skeys + pos + 32) : -2;
        int32_t prev = __shfl_up_sync(0xffffffffu, k0, 1);
        int32_t next = __shfl_down_sync(0xffffffffu, k0, 1);
        const int32_t k1_0 = __shfl_sync(0xffffffffu, k1, 0);
        if (lane == 0) prev = P0 > 0 ? __ldg(p.skeys + P0 - 1) : -1;
        if (lane == 31) next = k1_0;
        // runs (>= 2 entries) that START inside these 32 positions
        todo = __ballot_sync(0xffffffffu, pos < p.N && k0 >= 0 && k0 < p.key_limit && k0 != prev && (k0 == next || p.min_run1));
    }
    bool bars_ready = false;
    unsigned phase = 0;  // bit st = parity to wait for on bars[st]

    while (LIST ? lr < ln : todo != 0) {
        int64_t s;
        int32_t key;
        int n0;
        if (LIST) {
            int lo = 0, hi = p.run_nseg;              // largest segment with seg_base[seg] <= lr
            while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (seg_base[mid] <= lr) lo = mid; else hi = mid; }
            const uint32_t idx = lr - seg_base[lo];
            const int4 e = __ldg(p.run_list + (size_t)lo * p.run_cap + (LONGM ? (uint32_t)p.run_cap - 1u - idx : idx));
            lr += lstep;
            s = e.x; key = e.y; n0 = e.z;
        } else {
            const int bit = __ffs(todo) - 1;
            todo &= todo - 1;
            s = P0 + bit;
            key = __shfl_sync(0xffffffffu, k0, bit);
            // leading matches among the first 32 entries of the run (keys are already in registers)
            const int t = bit + lane;
            const int32_t ka = __shfl_sync(0xffffffffu, k0, t & 31);
            const int32_t kb = __shfl_sync(0xffffffffu, k1, t & 31);
            const unsigned mm = __ballot_sync(0xffffffffu, (t < 32 ? ka : kb) == key);
            n0 = (mm == 0xffffffffu) ? 32 : __ffs(~mm) - 1;
        }
        long long t_start = 0, t_direct = 0, t_ring = 0, c_wait = 0, c_cons = 0, c_issue = 0;
        if (p.dbg) t_start = clock64();
        int run_len = 0;
        // long run: probe its extent.  Keys are sorted, so "key at the end of 32-entry block b still matches"
        // is a prefix property: one load per lane covers the next 1024 entries.
        int32_t probe = -2;
        const int64_t ring0 = LONGM ? s : s + 32;     // first entry that goes through the ring
        if (LONGM) n0 = 0;                            // no direct part
        const bool ringed = LONGM || n0 == 32;
        if (ringed) { const int64_t q = ring0 + 32 * (int64_t)(lane + 1) - 1; probe = q < p.N ? __ldg(p.skeys + q) : -2; }
        if (ringed && !bars_ready) {
            if (lane == 0) {
                for (int st = 0; st < RING_NS; ++st) mbar_init(bars + st, 1);
                asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
            }
            __syncwarp();
            bars_ready = true;
        }

        for (int v0 = 0; v0 < nv; v0 += 32) {  // one pass per group of 32 (buffer, component) lanes
            const int vl = v0 + lane;
            const bool active = vl < nv;
            const bool isB = vl >= kc;
            const int comp = isB ? vl - kc : vl;
            // this lane's component row of the staging buffer
            const float* src = p.G + (size_t)(active ? vl : 0) * p.Npad;   // chain B rows follow chain A's (comp unused)
            (void)isB; (void)comp;
            // the row's old value is needed only at the very end: fetch it now, off the critical path
            float pold = 0.f;
            if (v0 == 0 && lane < kc && !p.shard_G) pold = p.table[(size_t)key * p.rowp + lane];
            // direct part: up to 32 entries straight from G, all loads in flight at once
            float acc = 0.f;
            {
                const float* sp = src + s;
                float tv[16], tw[16];
#pragma unroll
                for (int u = 0; u < 16; ++u) tv[u] = (active && u < n0) ? __ldg(sp + u) : 0.f;
#pragma unroll
                for (int u = 0; u < 16; ++u) tw[u] = (active && 16 + u < n0) ? __ldg(sp + 16 + u) : 0.f;
#pragma unroll
                for (int u = 0; u < 16; ++u)
                    if (u < n0) acc = __fadd_rn(acc, tv[u]);
#pragma unroll
                for (int u = 0; u < 16; ++u)
                    if (16 + u < n0) acc = __fadd_rn(acc, tw[u]);
            }
            if (p.dbg) t_direct = clock64();
            run_len = n0;
            if (ringed) {
                // stream the rest in windows of up to 1024 entries: [c0, c0 + wlen); every stage's copy starts `mis`
                // entries early (windows and stages are multiples of 4 entries, so `mis` is the same for all of them)
                int64_t c0 = ring0;
                const int mis = (int)(c0 & 3);
                int32_t pr = probe;
                bool ok = true;
                while (ok) {
                    const unsigned pm = __ballot_sync(0xffffffffu, pr == key);
                    const int full = (pm == 0xffffffffu) ? 32 : __ffs(~pm) - 1;   // full 32-entry blocks
                    int part = 0;
                    if (full < 32) {
                        const int64_t q = c0 + 32 * (int64_t)full + lane;
                        const unsigned m3 = __ballot_sync(0xffffffffu, q < p.N && __ldg(p.skeys + q) == key);
                        part = (m3 == 0xffffffffu) ? 32 : __ffs(~m3) - 1;
                    }
                    const int wlen = 32 * full + part;
                    const int T = (wlen + RING_SE - 1) / RING_SE;
                    // ONE tensor-map copy per stage: rows v0 .. v0+ring_comps-1 (rows past the last one are zero
                    // filled), RING_SEP entries from the 16-byte aligned position at or before the stage's first entry
                    auto issue = [&](int tstage) {
                        if (lane == 0) {
                            const int st = tstage & (RING_NS - 1);
                            mbar_expect_tx(bars + st, (unsigned)(ring_comps * RING_SEP * 4));
                            tma_g2s_2d(ring + (size_t)st * stage_f, &gmap, (int)(c0 - mis + RING_SE * (int64_t)tstage), v0, bars + st);
                        }
                    };
                    for (int ts = 0; ts < T && ts < RING_NS; ++ts) issue(ts);
                    // next window's probe (only needed when this window is completely full)
                    int32_t pr_next = -2;
                    if (full == 32) { const int64_t q = c0 + 1024 + 32 * (int64_t)(lane + 1) - 1; pr_next = q < p.N ? __ldg(p.skeys + q) : -2; }
                    for (int ts = 0; ts < T; ++ts) {
                        const int st = ts & (RING_NS - 1);
                        long long w0 = 0;
                        if (p.dbg) w0 = clock64();
                        if (!mbar_wait(bars + st, (phase >> st) & 1u)) { ok = false; break; }
                        phase ^= 1u << st;
                        long long w1 = 0;
                        if (p.dbg) { w1 = clock64(); c_wait += w1 - w0; }
                        const int n = min(RING_SE, wlen - RING_SE * ts);
                        if (active) {
                            const float4* b4 = reinterpret_cast<const float4*>(ring + (size_t)st * stage_f + lane * RING_SEP);
                            if (n == RING_SE) {        // full stage: entries [mis, mis + SE) of the lane's row = part of quad
                                                       // 0, quads 1 .. SE/4-1, part of quad SE/4; 16 LDS.128 in flight at a
                                                       // time, then the bare add chain
                                {
                                    const float4 q = b4[0];
                                    if (mis == 0) acc = __fadd_rn(acc, q.x);
                                    if (mis <= 1) acc = __fadd_rn(acc, q.y);
                                    if (mis <= 2) acc = __fadd_rn(acc, q.z);
                                    acc = __fadd_rn(acc, q.w);
                                }
#pragma unroll
                                for (int c = 0; c < RING_SE / 64; ++c) {
                                    constexpr int last = RING_SE / 64 - 1;
                                    const int nq = c == last ? 15 : 16;
                                    float4 tv[16];
#pragma unroll
                                    for (int u = 0; u < 16; ++u) if (u < nq) tv[u] = b4[1 + 16 * c + u];
#pragma unroll
                                    for (int u = 0; u < 16; ++u)
                                        if (u < nq) {
                                            acc = __fadd_rn(acc, tv[u].x); acc = __fadd_rn(acc, tv[u].y);
                                            acc = __fadd_rn(acc, tv[u].z); acc = __fadd_rn(acc, tv[u].w);
                                        }
                                }
                                {
                                    const float4 q = b4[RING_SE / 4];
                                    if (mis >= 1) acc = __fadd_rn(acc, q.x);
                                    if (mis >= 2) acc = __fadd_rn(acc, q.y);
                                    if (mis >= 3) acc = __fadd_rn(acc, q.z);
                                }
                            } else {
                                const int end = mis + n;   // entries [mis, end) of this lane's row
                                int e = 0;
                                if (mis) {                 // first, partial quad
                                    const float4 q = b4[0];
                                    if (mis <= 1 && 1 < end) acc = __fadd_rn(acc, q.y);
                                    if (mis <= 2 && 2 < end) acc = __fadd_rn(acc, q.z);
                                    if (3 < end) acc = __fadd_rn(acc, q.w);
                                    e = 4;
                                }
#pragma unroll 1
                                for (; e + 4 <= end; e += 4) {
                                    const float4 q = b4[e >> 2];
                                    acc = __fadd_rn(acc, q.x); acc = __fadd_rn(acc, q.y);
                                    acc = __fadd_rn(acc, q.z); acc = __fadd_rn(acc, q.w);
                                }
                                if (e < end) {             // last, partial quad
                                    const float4 q = b4[e >> 2];
                                    acc = __fadd_rn(acc, q.x);
                                    if (e + 1 < end) acc = __fadd_rn(acc, q.y);
                                    if (e + 2 < end) acc = __fadd_rn(acc, q.z);
                                }
                            }
                        }
                        __syncwarp();
                        long long w2 = 0;
                        if (p.dbg) { w2 = clock64(); c_cons += w2 - w1; }
                        if (ts + RING_NS < T) issue(ts + RING_NS);
                        if (p.dbg) c_issue += clock64() - w2;
                    }
                    run_len += wlen;
                    if (full < 32) break;
                    c0 += 1024;
                    pr = pr_next;
                }
            }
            if (p.dbg) t_ring = clock64();
            if (active) accs[vl] = acc;
            if (v0 == 0 && lane < kc) accs[accs_n + lane] = pold;
        }
        __syncwarp();
        // fold chain B into chain A and update the row (one lane per component)
        for (int c0 = 0; c0 < kc; c0 += 32) {
            const int c = c0 + lane;
            if (c < kc) {
                float gsum = accs[c];
                if (two && c < p.k) gsum = __fadd_rn(gsum, accs[kc + c]);
                if (p.shard_G) {
                    p.inbox[key % p.shard_G][((size_t)p.shard_me * p.shard_N + s) * 16 + c] = gsum;
                    continue;
                }
                float* addr = p.table + (size_t)key * p.rowp + c;
                const float old = c < 32 ? accs[accs_n + c] : *addr;
                if (ADA) {
                    float* sp = p.ada.sums + (size_t)key * p.rowp + c;
                    float sv = *sp;
                    *addr = fmb::adagrad_update(old, gsum, sv, p.lr, p.ada.eps);
                    *sp = sv;
                } else if (p.mode == 2) {
                    float* zp = p.ftrl.zn + (size_t)key * 2 * p.rowp + c;
                    float z = zp[0], n = zp[p.rowp];
                    *addr = fmb::ftrl_update(old, gsum, z, n, p.lr, p.ftrl.beta, p.ftrl.l1, p.ftrl.l2);
                    zp[0] = z; zp[p.rowp] = n;
                } else {
                    *addr = fmb::apply_update_a(old, gsum, p.lr, p.astep, p.mode);
                }
            }
        }
        __syncwarp();
        if (p.dbg && lane == 0 && run_len >= p.dbg[1]) {   // dbg[1] = shortest run to record
            const unsigned long long slot = atomicAdd((unsigned long long*)p.dbg, 1ULL);
            if (slot < 4000) {
                long long* r = p.dbg + 8 + slot * 8;
                unsigned long long gt; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt));
                r[0] = run_len; r[1] = (long long)gt - (clock64() - t_start) * 1000 / 1965; r[2] = t_direct - t_start; r[3] = t_ring - t_direct;
                r[4] = clock64() - t_ring; r[5] = c_issue; r[6] = c_wait; r[7] = c_cons;
            }
        }
    }
}

// position-major launch (tower fit, AFM, sharded paths).  ADA: update mode 3 (Adagrad)
template <bool ADA>
__global__ void __launch_bounds__(256, 2) fm_bwd_runs_kernel(const __grid_constant__ CUtensorMap gmap, BwdParams p, int warps_per_block, int warp_f,
                                                             int accs_n, int ring_comps) {
    runs_body<false, 64, 4, false, ADA>(gmap, p, warps_per_block, warp_f, accs_n, ring_comps, blockIdx.x, gridDim.x, 0);
}

// run-list launch: CTAs [0, nlong) take the long runs (>= 128 entries: 128-entry stages, ring from the first entry, wpl
// working warps), the others the short runs.  The long runs are the step's longest dependent chain, so their CTAs come
// first in the grid and are placed first; as two launches the second one waited for shared memory behind the first.
constexpr int LONG_SE = 128, LONG_NS = 4;
template <bool ADA>
__global__ void __launch_bounds__(256, 2) fm_bwd_runs_list_kernel(const __grid_constant__ CUtensorMap gmap_s, const __grid_constant__ CUtensorMap gmap_l,
                                                                  BwdParams p, int wps, int warp_f_s, int wpl, int warp_f_l, int accs_n,
                                                                  int ring_comps, unsigned nlong, int segb_off) {
    if (blockIdx.x < nlong) runs_body<true, LONG_SE, LONG_NS, true, ADA>(gmap_l, p, wpl, warp_f_l, accs_n, ring_comps, blockIdx.x, nlong, segb_off);
    else runs_body<true, 64, 4, false, ADA>(gmap_s, p, wps, warp_f_s, accs_n, ring_comps, blockIdx.x - nlong, gridDim.x - nlong, segb_off);
}

static int ilog2_ceil(int x) { int l = 0; while ((1 << l) < x) ++l; return l; }

}  // namespace

// workspace of fmb_fm_backward_update: the component-major contribution staging buffer (chain A rows, chain B rows)
static int64_t bwd_npad(int64_t N) { return (N + 3) / 4 * 4 + 64; }   // row pitch of G: multiple of 4, slack for
                                                                       // the bulk copies' rounded-up tails
FMB_API size_t fmb_bwd_workspace_bytes(int64_t N, int k) {
    const size_t rows = (size_t)((k + 1 + 3) / 4) * 4;
    return 2 * (((size_t)bwd_npad(N) * rows * 4 + 255) / 256 * 256) + 256;
}

static long long* g_runs_dbg = nullptr;
// debug hook (not in the public header): device buffer of 8 + 4000*8 int64 receiving per-run cycle counts
FMB_API void fmb_debug_set_runs_buffer(long long* dev) { g_runs_dbg = dev; }

// launches fm_bwd_runs_kernel over the staged contributions p.G (per-warp shared memory = ring + mbarriers + accumulators)
typedef CUresult (*EncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiled tensor_map_encoder() {
    static EncodeTiled encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && fn) encode = (EncodeTiled)fn;
    }
    return encode;
}

static int ring_warp_floats(int ring_comps, int accs_n, int SE, int NS, int* stage_f_out) {
    // ring (multiple of 128 B per warp) + NS mbarriers (8 B each) + accumulators + prefetched old row
    const int stage_f = fmb_round_up(ring_comps * (SE + 4), 32);
    if (stage_f_out) *stage_f_out = stage_f;
    return fmb_round_up(NS * stage_f + 2 * NS + accs_n + 32, 32);
}
// tensor map of the staging buffer: [nv rows][Npad] fp32, box = [ring_comps rows][SE + 4 entries]
static int ring_tensor_map(CUtensorMap* gmap, const BwdParams& p, int nv, int ring_comps, int SE) {
    EncodeTiled encode = tensor_map_encoder();
    if (!encode) { fmb_set_error("fmb_fm_backward_update: cuTensorMapEncodeTiled not available from the driver"); return FMB_ERR_CUDA; }
    const cuuint64_t gdim[2] = {(cuuint64_t)p.Npad, (cuuint64_t)nv};
    const cuuint64_t gstride[1] = {(cuuint64_t)p.Npad * 4};
    const cuuint32_t box[2] = {(cuuint32_t)(SE + 4), (cuuint32_t)ring_comps};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult cr = encode(gmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, p.G, gdim, gstride, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                               CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { fmb_set_error("fmb_fm_backward_update: cuTensorMapEncodeTiled failed (%d)", (int)cr); return FMB_ERR_CUDA; }
    return FMB_OK;
}

template <bool ADA>
static int launch_runs_t(BwdParams& p, bool two, cudaStream_t stream) {
    const int k = p.k;
    const int64_t N = p.N;
    const int nv = k + 1 + (two ? k : 0);
    const int accs_n = (nv + 3) / 4 * 4;
    const int ring_comps = nv < 32 ? nv : 32;
    const int warp_f = ring_warp_floats(ring_comps, accs_n, 64, 4, nullptr);
    int wpb = 8;
    while (wpb > 1 && (size_t)wpb * warp_f * 4 > 56 * 1024) wpb >>= 1;
    const size_t sm = (size_t)wpb * warp_f * 4;
    FMB_CHECK_ARG(sm <= 200 * 1024, "fmb_fm_backward_update: k too large for the run ring");
    const int64_t nwarps = (N + 31) / 32;
    const unsigned grid = (unsigned)((nwarps + wpb - 1) / wpb);
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(fm_bwd_runs_kernel<ADA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(fm_bwd_runs_list_kernel<ADA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr = true;
    }
    CUtensorMap gmap;
    int rc = ring_tensor_map(&gmap, p, nv, ring_comps, 64);
    if (rc) return rc;
    if (!p.run_list) {
        fm_bwd_runs_kernel<ADA><<<grid, 32 * wpb, sm, stream>>>(gmap, p, wpb, warp_f, accs_n, ring_comps);
        FMB_CHECK_LAUNCH("fm_bwd_runs_kernel");
        return FMB_OK;
    }
    // run-list launch.  Long-run CTAs: as many working warps as the short CTAs' shared memory holds with the deeper ring.
    CUtensorMap gmap_l;
    rc = ring_tensor_map(&gmap_l, p, nv, ring_comps, LONG_SE);
    if (rc) return rc;
    const int warp_f_l = ring_warp_floats(ring_comps, accs_n, LONG_SE, LONG_NS, nullptr);
    int wpl = (int)(sm / ((size_t)warp_f_l * 4));
    size_t smd = sm;
    if (wpl < 1) { wpl = 1; smd = (size_t)warp_f_l * 4; }
    if (wpl > wpb) wpl = wpb;
    FMB_CHECK_ARG(smd <= 200 * 1024, "fmb_fm_backward_update: k too large for the long-run ring");
    const size_t segb = (size_t)(p.run_nseg + 1 + 31) / 32 * 128;
    static int sms = 0;
    if (!sms) { int dev = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev); if (sms <= 0) sms = 148; }
    // short runs: as many CTAs as are resident at once beside the long-run CTAs, grid-strided over the list
    int per_sm = (int)((size_t)224 * 1024 / (smd + segb + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm * wpb > 32) per_sm = 32 / wpb;
    const unsigned nlong = (unsigned)sms;                                   // one long-run CTA per SM
    static int short_per_sm = -1;      // experiment knob FMB_RUNS_SHORT_PER_SM (default: one slot less than fit)
    if (short_per_sm < 0) { const char* e = getenv("FMB_RUNS_SHORT_PER_SM"); short_per_sm = e ? atoi(e) : 0; }
    unsigned nshort = (unsigned)(sms * (short_per_sm > 0 ? short_per_sm : (per_sm > 1 ? per_sm - 1 : 1)));
    if (nshort > grid) nshort = grid;
    if (p.pdl) {
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(nlong + nshort); cfg.blockDim = dim3(32 * wpb); cfg.dynamicSmemBytes = smd + segb; cfg.stream = stream;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        const cudaError_t le = cudaLaunchKernelEx(&cfg, fm_bwd_runs_list_kernel<ADA>, gmap, gmap_l, p, wpb, warp_f, wpl, warp_f_l, accs_n,
                                                  ring_comps, nlong, (int)(smd / 4));
        if (le != cudaSuccess) { fmb_set_error("fm_bwd_runs_list_kernel (programmatic launch): %s", cudaGetErrorString(le)); return FMB_ERR_CUDA; }
    } else {
        fm_bwd_runs_list_kernel<ADA><<<nlong + nshort, 32 * wpb, smd + segb, stream>>>(gmap, gmap_l, p, wpb, warp_f, wpl, warp_f_l, accs_n,
                                                                                 ring_comps, nlong, (int)(smd / 4));
    }
    FMB_CHECK_LAUNCH("fm_bwd_runs_list_kernel");
    return FMB_OK;
}
static int launch_runs(BwdParams& p, bool two, cudaStream_t stream) {
    return p.mode == 3 ? launch_runs_t<true>(p, two, stream) : launch_runs_t<false>(p, two, stream);
}

// A6 sparse backward + update (see file header).
//   sorted_keys/perm [N]: output of fmb_sort_segment / fmb_sort_fields over ids[B*F]; xv [B*F] or NULL
//   table [R,rowp] updated in place; S [B,kp4]; gs [B]; gvec [B,kp4] or NULL
//   use_fm2: the scalar gs also flows through Sum_j bi (FM / DeepFM logit); 0 for NFM
//   mode 0: fresh-Adam sign step (reference), 1: SGD
// _ex adds: n_entries = 1 + the largest entry index stored in perm (B*F; the sharded path passes
//   world*B*F), s_pitch / gs_stride (S, gvec and gs may live inside a gathered per-sample context),
//   key_limit (sorted keys >= key_limit are padding and are skipped).
// _rl: with the run list of the sorted keys (nullable; fmb_shard_sort_fields_rl / fmb_sort_fields_ex) the run kernel starts
// one warp per run, the long runs first (the owner-side chains of the sharded step are G*B/rows long)
struct fmb_runlist_t { int32_t* entries; uint32_t* seg_count; int nseg, seg_cap; };   // include/fmb200.h
struct fmb_adagrad_t { float* sums; float* bias_sum; float* mlp_sums; float eps; };   // include/fmb200.h
// _rl_ex: update mode 3 (Adagrad) needs `ada` (the table's sums); NULL otherwise
FMB_API int fmb_fm_backward_update_rl_ex(const int32_t* sorted_keys, const int32_t* perm, int64_t N, int64_t n_entries,
                                         const float* xv, float* table, int F, int k, const float* S, int s_pitch,
                                         const float* gs, int gs_stride, int use_fm2, const float* gvec,
                                         int32_t key_limit, float lr, int mode, const fmb_adagrad_t* ada,
                                         const fmb_runlist_t* rl, void* ws, size_t ws_bytes, cudaStream_t stream) {
    FMB_CHECK_ARG(!rl || (rl->entries && rl->seg_count && rl->nseg >= 1 && rl->nseg <= 2048 && rl->seg_cap >= 1),
                  "fmb_fm_backward_update: bad run list");
    FMB_CHECK_ARG(sorted_keys && perm && table && S && gs && ws, "fmb_fm_backward_update: null pointer");
    FMB_CHECK_ARG(N > 0 && F > 0 && F < 512 && k > 0 && k <= 124, "fmb_fm_backward_update: bad shape N=%lld F=%d k=%d (need F < 512, k <= 124)",
                  (long long)N, F, k);
    FMB_CHECK_ARG(mode == 0 || mode == 1 || (mode == 3 && ada && ada->sums),
                  "fmb_fm_backward_update: unknown update mode %d (mode 3 needs the Adagrad state)", mode);
    FMB_CHECK_ARG(use_fm2 || gvec, "fmb_fm_backward_update: neither gradient path enabled");
    FMB_CHECK_ARG(n_entries > 0 && n_entries < ((int64_t)1 << 31), "fmb_fm_backward_update: n_entries out of range");
    if (ws_bytes < fmb_bwd_workspace_bytes(N, k)) { fmb_set_error("fmb_fm_backward_update: workspace too small"); return FMB_ERR_WS; }
    BwdParams p;
    memset(&p, 0, sizeof(p));
    p.skeys = sorted_keys; p.perm = perm; p.N = N; p.xv = xv; p.table = table;
    p.F = F; p.k = k; p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4);
    p.cu = (k + 1 + 3) / 4; p.ql_log = ilog2_ceil(p.cu);
    {
        int bn = 0, bf = 0;
        while (((int64_t)1 << bn) < n_entries) ++bn;
        while ((1 << bf) <= F) ++bf;
        p.fshift = bn + bf;  // 2^fshift > n_entries*F, and e*fmagic < 2^(2*bn+2) <= 2^64
        p.fmagic = ((1ULL << p.fshift) + (unsigned long long)F - 1) / (unsigned long long)F;
    }
    p.S = S; p.gs = gs; p.use_fm2 = use_fm2; p.gvec = gvec; p.lr = lr; p.mode = mode;
    p.s_pitch = s_pitch; p.gs_stride = gs_stride; p.key_limit = key_limit;
    p.astep = -(lr / 0.1f);
    if (mode == 3) { p.ada.sums = ada->sums; p.ada.bias_sum = ada->bias_sum; p.ada.eps = ada->eps; }
    p.dbg = g_runs_dbg;
    p.Npad = bwd_npad(N);
    p.G = (float*)ws;
    const bool two = use_fm2 && gvec;
    const unsigned grid1 = (unsigned)((N + 255) / 256);
    if (mode == 3) {
        switch (p.cu) {
            case 1: fm_bwd_entry1_kernel<1, true><<<grid1, 256, 0, stream>>>(p); break;
            case 2: fm_bwd_entry1_kernel<2, true><<<grid1, 256, 0, stream>>>(p); break;
            case 3: fm_bwd_entry1_kernel<3, true><<<grid1, 256, 0, stream>>>(p); break;
            case 4: fm_bwd_entry1_kernel<4, true><<<grid1, 256, 0, stream>>>(p); break;
            default: {
                const int epb = 256 >> p.ql_log;
                fm_bwd_entry_kernel<true><<<(unsigned)((N + epb - 1) / epb), 256, 0, stream>>>(p);
            }
        }
    } else {
        switch (p.cu) {
            case 1: fm_bwd_entry1_kernel<1, false><<<grid1, 256, 0, stream>>>(p); break;
            case 2: fm_bwd_entry1_kernel<2, false><<<grid1, 256, 0, stream>>>(p); break;
            case 3: fm_bwd_entry1_kernel<3, false><<<grid1, 256, 0, stream>>>(p); break;
            case 4: fm_bwd_entry1_kernel<4, false><<<grid1, 256, 0, stream>>>(p); break;
            default: {
                const int epb = 256 >> p.ql_log;
                fm_bwd_entry_kernel<false><<<(unsigned)((N + epb - 1) / epb), 256, 0, stream>>>(p);
            }
        }
    }
    FMB_CHECK_LAUNCH("fm_bwd_entry_kernel");
    if (rl) { p.run_list = reinterpret_cast<const int4*>(rl->entries); p.run_segc = rl->seg_count; p.run_nseg = rl->nseg; p.run_cap = rl->seg_cap; }
    return launch_runs(p, two, stream);
}

FMB_API int fmb_fm_backward_update_rl(const int32_t* sorted_keys, const int32_t* perm, int64_t N, int64_t n_entries,
                                      const float* xv, float* table, int F, int k, const float* S, int s_pitch,
                                      const float* gs, int gs_stride, int use_fm2, const float* gvec,
                                      int32_t key_limit, float lr, int mode, const fmb_runlist_t* rl, void* ws, size_t ws_bytes,
                                      cudaStream_t stream) {
    return fmb_fm_backward_update_rl_ex(sorted_keys, perm, N, n_entries, xv, table, F, k, S, s_pitch, gs, gs_stride, use_fm2,
                                        gvec, key_limit, lr, mode, nullptr, rl, ws, ws_bytes, stream);
}

FMB_API int fmb_fm_backward_update_ex(const int32_t* sorted_keys, const int32_t* perm, int64_t N, int64_t n_entries,
                                      const float* xv, float* table, int F, int k, const float* S, int s_pitch,
                                      const float* gs, int gs_stride, int use_fm2, const float* gvec,
                                      int32_t key_limit, float lr, int mode, void* ws, size_t ws_bytes,
                                      cudaStream_t stream) {
    return fmb_fm_backward_update_rl(sorted_keys, perm, N, n_entries, xv, table, F, k, S, s_pitch, gs, gs_stride, use_fm2, gvec,
                                     key_limit, lr, mode, nullptr, ws, ws_bytes, stream);
}

// Run kernel alone: sums the contributions staged in ws (by fmb_fm_step_fused, at sorted positions) over every run
// of >= 2 equal keys, in sample order, and updates those rows.  Same arguments as fmb_fm_backward_update.
struct fmb_ftrl_t { float* zn; float* bias_zn; float beta, l1, l2; };   // include/fmb200.h

// rl (nullable): the runs of >= 2 entries found by the sort one step ahead (fmb_sort_fields_ex / fmb_pos_flags_ex); with it
// one warp is started per RUN instead of per 32 sorted positions.

static thread_local int g_runs_pdl = 0;   // per calling thread: set and consumed by consecutive calls of one host thread
// internal (session.cu): the NEXT fmb_fm_backward_runs_list call is launched as a programmatic dependent of the kernel
// in front of it on its stream (the fused kernel, which executes griddepcontrol.launch_dependents)
FMB_API void fmb_runs_list_next_is_dependent(int on) { g_runs_pdl = on; }

FMB_API int fmb_fm_backward_runs_list(const int32_t* sorted_keys, int64_t N, float* table, int F, int k, float lr,
                                      int mode, const fmb_ftrl_t* ftrl, const fmb_runlist_t* rl,
                                      void* ws, size_t ws_bytes, cudaStream_t stream) {
    FMB_CHECK_ARG(sorted_keys && table && ws, "fmb_fm_backward_runs: null pointer");
    FMB_CHECK_ARG(!rl || (rl->entries && rl->seg_count && rl->nseg >= 1 && rl->nseg <= 2048 && rl->seg_cap >= 1),
                  "fmb_fm_backward_runs: bad run list");
    FMB_CHECK_ARG(N > 0 && F > 0 && F < 512 && k > 0 && k <= 124, "fmb_fm_backward_runs: bad shape N=%lld F=%d k=%d (need F < 512, k <= 124)",
                  (long long)N, F, k);
    FMB_CHECK_ARG(mode == 0 || mode == 1 || (mode == 2 && ftrl && ftrl->zn) ||
                  (mode == 3 && ftrl && reinterpret_cast<const fmb_adagrad_t*>(ftrl)->sums),
                  "fmb_fm_backward_runs: unknown update mode %d", mode);
    if (ws_bytes < fmb_bwd_workspace_bytes(N, k)) { fmb_set_error("fmb_fm_backward_runs: workspace too small"); return FMB_ERR_WS; }
    BwdParams p;
    memset(&p, 0, sizeof(p));
    p.skeys = sorted_keys; p.N = N; p.table = table;
    p.F = F; p.k = k; p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4);
    p.use_fm2 = 1; p.gvec = nullptr; p.lr = lr; p.mode = mode; p.key_limit = 0x7fffffff;
    p.astep = -(lr / 0.1f);
    p.dbg = nullptr;
    p.Npad = bwd_npad(N);
    p.G = (float*)ws;
    if (mode == 2) { p.ftrl.zn = ftrl->zn; p.ftrl.bias_zn = ftrl->bias_zn; p.ftrl.beta = ftrl->beta; p.ftrl.l1 = ftrl->l1; p.ftrl.l2 = ftrl->l2; }
    if (mode == 3) {   // the state slot carries an fmb_adagrad_t in mode 3 (include/fmb200.h)
        const fmb_adagrad_t* a = reinterpret_cast<const fmb_adagrad_t*>(ftrl);
        p.ada.sums = a->sums; p.ada.bias_sum = a->bias_sum; p.ada.eps = a->eps;
    }
    if (rl) { p.run_list = reinterpret_cast<const int4*>(rl->entries); p.run_segc = rl->seg_count; p.run_nseg = rl->nseg; p.run_cap = rl->seg_cap; }
    p.pdl = rl ? g_runs_pdl : 0;
    g_runs_pdl = 0;
    p.dbg = g_runs_dbg;
    return launch_runs(p, false, stream);
}

FMB_API int fmb_fm_backward_runs_ex(const int32_t* sorted_keys, int64_t N, float* table, int F, int k, float lr,
                                    int mode, const fmb_ftrl_t* ftrl, void* ws, size_t ws_bytes, cudaStream_t stream) {
    return fmb_fm_backward_runs_list(sorted_keys, N, table, F, k, lr, mode, ftrl, nullptr, ws, ws_bytes, stream);
}

FMB_API int fmb_fm_backward_runs(const int32_t* sorted_keys, int64_t N, float* table, int F, int k, float lr,
                                 int mode, void* ws, size_t ws_bytes, cudaStream_t stream) {
    return fmb_fm_backward_runs_ex(sorted_keys, N, table, F, k, lr, mode, nullptr, ws, ws_bytes, stream);
}

// every run, rows hit once included (the AFM step stages ALL its per-entry gradients: csrc/afm.cu)
FMB_API int fmb_fm_backward_runs_all(const int32_t* sorted_keys, int64_t N, float* table, int F, int k, float lr,
                                     int mode, void* ws, size_t ws_bytes, cudaStream_t stream) {
    FMB_CHECK_ARG(sorted_keys && table && ws, "fmb_fm_backward_runs_all: null pointer");
    FMB_CHECK_ARG(N > 0 && F > 0 && F < 512 && k > 0 && k <= 124, "fmb_fm_backward_runs_all: bad arguments");
    FMB_CHECK_ARG(mode == 0 || mode == 1, "fmb_fm_backward_runs_all: unknown update mode %d", mode);
    if (ws_bytes < fmb_bwd_workspace_bytes(N, k)) { fmb_set_error("fmb_fm_backward_runs_all: workspace too small"); return FMB_ERR_WS; }
    BwdParams p;
    memset(&p, 0, sizeof(p));
    p.skeys = sorted_keys; p.N = N; p.table = table;
    p.F = F; p.k = k; p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4);
    p.use_fm2 = 1; p.lr = lr; p.mode = mode; p.key_limit = 0x7fffffff; p.astep = -(lr / 0.1f);
    p.Npad = bwd_npad(N); p.G = (float*)ws; p.min_run1 = 1;
    return launch_runs(p, false, stream);
}

// multi-GPU variant of fmb_fm_backward_runs (csrc/shard2.cu): the partial gradient of every run of >= 2 equal keys goes
// to the inbox of the row's owner instead of being applied.  inbox: G peer-mapped pointers to [G][N][16] floats.
FMB_API int fmb_shard2_runs(const int32_t* sorted_keys, int64_t N, int F, int k, void* ws, size_t ws_bytes,
                            void* const* inbox, int G, int me, cudaStream_t stream) {
    FMB_CHECK_ARG(sorted_keys && ws && inbox, "fmb_shard2_runs: null pointer");
    FMB_CHECK_ARG(N > 0 && F > 0 && F < 512 && k > 0 && k <= 15 && G >= 1 && G <= 8 && me >= 0 && me < G, "fmb_shard2_runs: bad arguments");
    if (ws_bytes < fmb_bwd_workspace_bytes(N, k)) { fmb_set_error("fmb_shard2_runs: workspace too small"); return FMB_ERR_WS; }
    BwdParams p;
    memset(&p, 0, sizeof(p));
    p.skeys = sorted_keys; p.N = N; p.table = nullptr;
    p.F = F; p.k = k; p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4);
    p.use_fm2 = 1; p.key_limit = 0x7fffffff;
    p.Npad = bwd_npad(N);
    p.G = (float*)ws;
    for (int o = 0; o < G; ++o) p.inbox[o] = (float*)inbox[o];
    p.shard_G = G; p.shard_me = me; p.shard_N = N;
    return launch_runs(p, false, stream);
}

FMB_API int fmb_fm_backward_update(const int32_t* sorted_keys, const int32_t* perm, int64_t N, const float* xv,
                                   float* table, int F, int k, const float* S, const float* gs, int use_fm2,
                                   const float* gvec, float lr, int mode, void* ws, size_t ws_bytes,
                                   cudaStream_t stream) {
    return fmb_fm_backward_update_ex(sorted_keys, perm, N, N, xv, table, F, k, S, fmb_round_up(k, 4), gs, 1, use_fm2,
                                     gvec, 0x7fffffff, lr, mode, ws, ws_bytes, stream);
}
