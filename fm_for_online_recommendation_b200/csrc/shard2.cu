// shard2.cu -- row-sharded multi-GPU FM step with O(B*F) work per rank (BASELINE.json configs[4]; SURVEY.md 8e).
//
// Row r of the packed table lives on rank r % G at local row r / G.  Every rank steps on ITS OWN batch of B samples;
// one call on every rank performs the step over the global batch of G*B samples (loss = mean over G*B, torch.sigmoid
// positions and the bias gradient over the concatenated batch).  The reference has no distributed code; this is the
// B200-native design for its Criteo-scale configuration, built on NVLink peer memory instead of collectives:
//
//   forward   the fused step kernel gathers rows straight from the owners' table shards (cp.async on peer-mapped
//             pointers: 64-byte reads over NVLink / NVSwitch), so logits are computed in the REFERENCE's field order --
//             bit-identical to the single-GPU step on the concatenated batch (the round-1 path folded owner partials)
//   backward  a rank reduces the duplicates of its own batch in sample order (the single-GPU run kernel) and stores one
//             partial gradient per distinct row into the owner's inbox, at the row's position in the rank's stable sort;
//             entries that are the only hit of their row in the rank's batch are stored by the fused kernel itself
//   exchange  epoch flags in peer memory (fmb_shard_signal): no NCCL call in the step
//   owner     scans the G sorted key lists (pushed one step ahead, with the sort), counts the ranks that hit each owned
//             row, adds their partials IN RANK ORDER and applies the row update
// The only change in arithmetic versus one GPU is that order ("rank-partial": oracle/fm_oracle.c rank_B); rows hit by a
// single rank -- all but the hot rows of the small fields and a few per cent of the others -- see no change at all.
// Work per rank per step: B*F entries forward and backward, G*B*F sorted KEYS scanned (10 MB at G = 8), <= B*F inbox
// slots applied -- nothing grows with the global batch except that key scan.
#include "fmb_common.cuh"
#include <cstring>

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

// Consumer-side wait of an exchange: returns once all G peers have published (fmb_shard_signal, mode 1) the epoch this
// rank itself has reached on `channel`.  flags: uint32 [8 channels][8 ranks] written by the peers; epoch: my own counters.
// Called by every thread of a block; bounded spin, *error = 1 + channel on a time-out (the step's results are then void:
// ShardedFM2 polls the word).
struct WaitSpec { const uint32_t* flags; const uint32_t* epoch; int* error; int channel, G; };
__device__ __forceinline__ void wait_epoch(const WaitSpec& w) {
    if (w.channel < 0) return;
    if ((int)threadIdx.x < w.G) {
        const uint32_t e = w.epoch[w.channel];
        const uint32_t* f = w.flags + w.channel * 8 + threadIdx.x;
        bool ok = false;
        for (long long spin = 0; spin < (1ll << 26) && !ok; ++spin) {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];\n" : "=r"(v) : "l"(f) : "memory");
            ok = (int32_t)(v - e) >= 0;
        }
        if (!ok && w.error) *w.error = 1 + w.channel;
    }
    __syncthreads();
}

constexpr int SLOTW = 16;   // floats per inbox slot (64 bytes: k + 1 <= 16 on this path)

struct S2Params {
    float* tables[8];      // peer-mapped table shards (only tables[me] is read: remote rows arrive in rowbox)
    const float* rowbox;   // [N][SLOTW] rows the owners pushed for MY entries, at my sorted positions
    const float* hot;      // [R_hot][SLOTW] replica of the rows of the small ("hot") fields, kept current by the owners
    const int32_t* hot_base;   // [F] first hot-table row of field f, or -1 (device array)
    const int32_t* field_off;  // [F+1]
    float* inbox[8];       // peer-mapped inboxes [G sources][N slots][SLOTW]
    float* dl[8];          // peer-mapped [2][G*B]: delta | per-sample loss of the global batch
    const float* bias;
    int B, F, k, rowp, kp4, SB, cu, ql_log, jl_log, loss_kind;
    int G, me, gshift;     // gshift = log2(G) when G is a power of two, else -1
    float* Gst;            // local component-major staging of multi-hit entries (run kernel input)
    int64_t Npad, N;
    WaitSpec wait;         // the rowbox must be complete (ROWS channel) before the gather
};

//   ids [B,F] global row ids of MY batch;  xv [B,F] or NULL;  y [B];  posflag [B*F]: sorted position | multi-hit flag
__global__ void __launch_bounds__(256) shard2_fused_kernel(const int32_t* __restrict__ ids, const float* __restrict__ xv,
                                                           const float* __restrict__ y, const uint32_t* __restrict__ posflag,
                                                           S2Params p) {
    extern __shared__ __align__(16) float smem[];
    const int F = p.F, k = p.k, SB = p.SB, G = p.G;
    const int rp = p.cu * 4;
    float* rows_s = smem;                          // [SB][F][rp]
    float* x_s = rows_s + (size_t)SB * F * rp;     // [SB][F]
    float* bi_s = x_s + SB * F;                    // [SB][k]
    float* S_s = bi_s + SB * k;                    // [SB][kp4]
    float* d_s = S_s + SB * p.kp4;                 // [SB]
    int32_t* ids_s = reinterpret_cast<int32_t*>(d_s + SB);            // [SB][F]
    uint32_t* pos_s = reinterpret_cast<uint32_t*>(ids_s + SB * F);    // [SB][F]
    const int b0 = blockIdx.x * SB;
    const int nv = min(SB, p.B - b0);

    wait_epoch(p.wait);
    for (int e = threadIdx.x; e < nv * F; e += blockDim.x) {
        ids_s[e] = __ldg(ids + (size_t)b0 * F + e);
        x_s[e] = xv ? __ldg(xv + (size_t)b0 * F + e) : 1.0f;
        pos_s[e] = __ldg(posflag + (size_t)b0 * F + e);
    }
    __syncthreads();
    // gather: every row read is LOCAL -- hot-field replica, my own shard, or the slot its owner pushed it to (64-byte
    // reads over NVLink are round trips with few requests in flight: 90 us for 10 MB measured; posted writes stream)
    {
        const int q = threadIdx.x & ((1 << p.ql_log) - 1);
        const int estep = blockDim.x >> p.ql_log;
        if (q < p.cu)
            for (int ef = threadIdx.x >> p.ql_log; ef < nv * F; ef += estep) {
                const int r = ids_s[ef];
                const int f = ef % F;
                const int hb = __ldg(p.hot_base + f);
                const float* src;
                if (hb >= 0) src = p.hot + (size_t)(hb + r - __ldg(p.field_off + f)) * SLOTW;            // replicated hot row
                else if ((p.gshift >= 0 ? (r & (G - 1)) : r % G) == p.me)
                    src = p.tables[p.me] + (size_t)(p.gshift >= 0 ? (r >> p.gshift) : r / G) * p.rowp;  // my own shard
                else src = p.rowbox + (size_t)(pos_s[ef] & 0x7fffffffu) * SLOTW;                         // pushed by its owner
                cp_async16(rows_s + (size_t)ef * rp + q * 4, src + q * 4);
            }
    }
    cp_async_wait_all();
    __syncthreads();
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
                S_s[s * p.kp4 + j] = Sj;
            }
    }
    __syncthreads();
    {
        const int s = threadIdx.x >> 3, l8 = threadIdx.x & 7;
        const int nv8 = (nv + 3) & ~3;
        if (s < nv8) {
            const int sc = min(s, nv - 1);
            const float* r = rows_s + (size_t)sc * F * rp + k;
            const float* xs = x_s + sc * F;
            const float sf = fmb::aten_row_sum_lanes8([&](int f) { return __fmul_rn(r[(size_t)f * rp], xs[f]); }, F, l8, 0xffffffffu);
            const float* bs = bi_s + sc * k;
            const float sb = fmb::aten_row_sum_lanes8([&](int j) { return bs[j]; }, k, l8, 0xffffffffu);
            if (l8 == 0 && s < nv) {
                const int b = b0 + s;
                const float z = __fadd_rn(__fadd_rn(sf, sb), __ldg(p.bias));
                float lv, d;
                // sample b of rank `me` is element me*B + b of the concatenated batch of G*B samples
                fmb::bce_logits_value_grad(p.loss_kind, z, y[b], p.me * p.B + b, G * p.B, lv, d);
                d_s[s] = d;
                const size_t gb = (size_t)p.me * p.B + b;
                for (int o = 0; o < G; ++o) {          // every rank needs every delta (bias gradient) and loss value
                    p.dl[o][gb] = d;
                    p.dl[o][(size_t)G * p.B + gb] = lv;
                }
            }
        }
    }
    __syncthreads();
    // contributions: a row hit once in MY batch goes straight to its owner's inbox (slot = my rank, sorted position),
    // the others are staged locally for the run kernel
    const int items = nv * F * p.cu;
    for (int it = threadIdx.x; it < items; it += blockDim.x) {
        const int ef = it / p.cu, q = it - ef * p.cu;
        const int s = ef / F;
        const float x = x_s[ef], d = d_s[s];
        const uint32_t pf = pos_s[ef];
        const size_t pos = pf & 0x7fffffffu;
        const float* Ss = S_s + s * p.kp4;
        const float4 v4 = *reinterpret_cast<const float4*>(rows_s + (size_t)ef * rp + q * 4);
        const float v[4] = {v4.x, v4.y, v4.z, v4.w};
        float a[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int j = q * 4 + t;
            a[t] = 0.f;
            if (j < k) {
                const float ej = __fmul_rn(v[t], x);
                a[t] = __fmul_rn(__fsub_rn(__fmul_rn(d, Ss[j]), __fmul_rn(d, ej)), x);
            } else if (j == k) {
                a[t] = __fmul_rn(d, x);
            }
        }
        if (!(pf >> 31)) {
            const int o = p.gshift >= 0 ? (ids_s[ef] & (G - 1)) : ids_s[ef] % G;   // partial of a single entry = 0 + contribution
            *reinterpret_cast<float4*>(p.inbox[o] + ((size_t)p.me * p.N + pos) * SLOTW + q * 4) =
                make_float4(__fadd_rn(0.f, a[0]), __fadd_rn(0.f, a[1]), __fadd_rn(0.f, a[2]), __fadd_rn(0.f, a[3]));
        } else {
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (q * 4 + t <= k) p.Gst[(size_t)(q * 4 + t) * p.Npad + pos] = a[t];
        }
    }
}

// my sorted keys -> slab `me` of every rank's keys_all [G][N]
struct PeerI32 { int32_t* p[8]; };
__global__ void __launch_bounds__(256) push_keys_kernel(const int32_t* __restrict__ skeys, int64_t N, int G, int me,
                                                        PeerI32 dst) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= N) return;
    const int32_t v = skeys[i];
    for (int o = 0; o < G; ++o) dst.p[o][(size_t)me * N + i] = v;
}

struct OwnerParams {
    const int32_t* keys_all;   // [G][N] every rank's sorted keys (per field: B keys, sorted by row id, ties in sample order)
    const float* inbox;        // [G][N][SLOTW] partial gradients at run-start positions
    float* table;              // my shard
    uint32_t* cnt;             // [R_local] ranks that hit each owned row this step (zero between steps)
    float* rowbox[8];          // peer-mapped rowboxes (push_rows)
    float* hot[8];             // peer-mapped hot-row replicas
    const int32_t* hot_base;   // [F]
    const int32_t* field_off;  // [F+1]
    int N, B, F, k, rowp, G, me, mode, gshift;   // gshift: log2(G) when G is a power of two, else -1
    float lr, astep;
    uint32_t* list;            // [G*N] compact list of the owned run starts (s*N + i), any order
    uint32_t* nlist;           // [2] list length of this step (index `par`) / of the next one (zeroed here)
    int par;
    WaitSpec wait;             // the partials must have landed (PUSH channel) before they are counted
};

__device__ __forceinline__ int own_mod(const OwnerParams& p, int key) { return p.gshift >= 0 ? (key & (p.G - 1)) : key % p.G; }
__device__ __forceinline__ int own_div(const OwnerParams& p, int key) { return p.gshift >= 0 ? (key >> p.gshift) : key / p.G; }

// grid: x over sorted positions (a block never straddles a field when B % 256 == 0, else the test below is per thread),
// y = source rank.  Is position i of source s the first entry of a run of a row I own?
__device__ __forceinline__ bool owned_run_start(const OwnerParams& p, int s, int i, int* key, int* field) {
    const int32_t kk = __ldg(p.keys_all + (size_t)s * p.N + i);
    if (own_mod(p, kk) != p.me) return false;
    const int f = i / p.B;
    if (i > f * p.B && __ldg(p.keys_all + (size_t)s * p.N + i - 1) == kk) return false;
    *key = kk; *field = f;
    return true;
}

// pass 1: count the ranks hitting every owned row and build the compact list of owned run starts, so that the apply
// pass runs full warps (ownership r % G interleaves: 1 lane in G would be active otherwise)
__global__ void __launch_bounds__(256) owner_count_kernel(OwnerParams p) {
    wait_epoch(p.wait);
    const int i = blockIdx.x * 256 + threadIdx.x, s = blockIdx.y;
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) p.nlist[1 - p.par] = 0;   // next step's counter
    int key = 0, f = 0;
    const bool mine = i < p.N && owned_run_start(p, s, i, &key, &f);
    if (mine) atomicAdd(p.cnt + own_div(p, key), 1u);   // integer: order-independent
    // block-aggregated append: one atomic on the list length per block
    __shared__ uint32_t wcount[8], bbase;
    const unsigned m = __ballot_sync(0xffffffffu, mine);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) wcount[warp] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int w = 0; w < 8; ++w) { const uint32_t c = wcount[w]; wcount[w] = tot; tot += c; }
        bbase = tot ? atomicAdd(p.nlist + p.par, tot) : 0u;
    }
    __syncthreads();
    if (mine) p.list[bbase + wcount[warp] + __popc(m & ((1u << lane) - 1u))] = (uint32_t)s * (uint32_t)p.N + (uint32_t)i;
}

// first position of `key` in source s's sorted field segment [lo, lo+B), or -1
__device__ __forceinline__ int find_key(const OwnerParams& p, int s, int lo, int32_t key) {
    const int32_t* a = p.keys_all + (size_t)s * p.N + lo;
    int l = 0, h = p.B;
    while (l < h) { const int m = (l + h) >> 1; if (__ldg(a + m) < key) l = m + 1; else h = m; }
    return (l < p.B && __ldg(a + l) == key) ? lo + l : -1;
}

// pass 2: four lanes per listed run start: lane q applies 16-byte chunk q of the row (for the rare rows several ranks
// hit, the searches are done by all four lanes -- same addresses, one transaction).  Grid-stride over the list.
__global__ void __launch_bounds__(256) owner_apply_kernel(OwnerParams p) {
    const uint32_t n = p.nlist[p.par];
    const int cu = (p.k + 1 + 3) / 4;
    for (uint32_t t = blockIdx.x * 256 + threadIdx.x; t < n * 4; t += gridDim.x * 256) {   // one item per thread (grid covers G*N*4)
        const uint32_t li = t >> 2;
        const int q = (int)(t & 3);
        const uint32_t sp = p.list[li];
        const int s = (int)(sp / (uint32_t)p.N), i = (int)(sp - (uint32_t)s * (uint32_t)p.N);
        const int32_t key = __ldg(p.keys_all + sp);
        const int f = i / p.B;
        const int lrow = own_div(p, key);
        const uint32_t c = p.cnt[lrow];
        const int lo = f * p.B;
        size_t src_pos[8];
        int nsrc = 1;
        src_pos[0] = sp;
        bool leader = true;
        if (c > 1) {
            // several ranks hit this row: the lowest rank among them adds the partials in rank order
            for (int r = 0; r < s && leader; ++r)
                if (find_key(p, r, lo, key) >= 0) leader = false;
            for (int r = s + 1; r < p.G && leader; ++r) {
                const int pos = find_key(p, r, lo, key);
                if (pos >= 0) src_pos[nsrc++] = (size_t)r * p.N + pos;
            }
        }
        if (!leader || q >= cu) continue;
        float* row = p.table + (size_t)lrow * p.rowp;
        float4 g = __ldg(reinterpret_cast<const float4*>(p.inbox + src_pos[0] * SLOTW + q * 4));
        for (int r = 1; r < nsrc; ++r) {
            const float4 h = __ldg(reinterpret_cast<const float4*>(p.inbox + src_pos[r] * SLOTW + q * 4));
            g.x = __fadd_rn(g.x, h.x); g.y = __fadd_rn(g.y, h.y); g.z = __fadd_rn(g.z, h.z); g.w = __fadd_rn(g.w, h.w);
        }
        const float4 v = *reinterpret_cast<const float4*>(row + q * 4);
        float4 o = v;
        if (q * 4 + 0 <= p.k) o.x = fmb::apply_update_a(v.x, g.x, p.lr, p.astep, p.mode);
        if (q * 4 + 1 <= p.k) o.y = fmb::apply_update_a(v.y, g.y, p.lr, p.astep, p.mode);
        if (q * 4 + 2 <= p.k) o.z = fmb::apply_update_a(v.z, g.z, p.lr, p.astep, p.mode);
        if (q * 4 + 3 <= p.k) o.w = fmb::apply_update_a(v.w, g.w, p.lr, p.astep, p.mode);
        const bool moved = __float_as_int(o.x) != __float_as_int(v.x) || __float_as_int(o.y) != __float_as_int(v.y) ||
                           __float_as_int(o.z) != __float_as_int(v.z) || __float_as_int(o.w) != __float_as_int(v.w);
        if (moved) {
            *reinterpret_cast<float4*>(row + q * 4) = o;
            const int hb = __ldg(p.hot_base + f);
            if (hb >= 0) {   // a hot-field row: keep every rank's replica current
                const size_t h = (size_t)(hb + key - __ldg(p.field_off + f)) * SLOTW + q * 4;
                for (int r = 0; r < p.G; ++r) *reinterpret_cast<float4*>(p.hot[r] + h) = o;
            }
        }
    }
}

// pass 3: the counters go back to zero for the next step (after every apply thread has read them)
__global__ void __launch_bounds__(256) owner_reset_kernel(OwnerParams p) {
    const uint32_t n = p.nlist[p.par];
    for (uint32_t t = blockIdx.x * 256 + threadIdx.x; t < n; t += gridDim.x * 256)
        p.cnt[own_div(p, __ldg(p.keys_all + p.list[t]))] = 0;
}

// Row service for the NEXT forward pass: every entry of every other rank's sorted list that names a row I own (outside
// the replicated hot fields) gets that row stored into the requester's rowbox at the entry's sorted position.  Posted
// 16-byte stores over NVLink; four lanes per entry.
__global__ void __launch_bounds__(256) push_rows_kernel(OwnerParams p) {
    // four lanes per key (one per 16-byte chunk): a thread per key copying 48 bytes was slower (44 vs 32 us at G = 2)
    const int t = blockIdx.x * 256 + threadIdx.x, s = blockIdx.y;
    const int i = t >> 2, q = t & 3;
    if (i >= p.N || s == p.me || q >= (p.k + 1 + 3) / 4) return;
    const int32_t key = __ldg(p.keys_all + (size_t)s * p.N + i);
    if (own_mod(p, key) != p.me) return;
    if (__ldg(p.hot_base + i / p.B) >= 0) return;
    const float4 v = *reinterpret_cast<const float4*>(p.table + (size_t)own_div(p, key) * p.rowp + q * 4);
    *reinterpret_cast<float4*>(p.rowbox[s] + (size_t)i * SLOTW + q * 4) = v;
}

// my owned rows of the hot fields -> every rank's replica (initialisation / after loading parameters)
__global__ void __launch_bounds__(256) push_hot_kernel(OwnerParams p, int R_hot) {
    const int t = blockIdx.x * 256 + threadIdx.x;
    const int h = t >> 2, q = t & 3;
    if (h >= R_hot || q >= (p.k + 1 + 3) / 4) return;
    // field of hot row h
    int f = 0;
    for (int g = 0; g < p.F; ++g) { const int hb = __ldg(p.hot_base + g); if (hb >= 0 && hb <= h) f = g; }
    const int key = __ldg(p.field_off + f) + (h - __ldg(p.hot_base + f));
    if (own_mod(p, key) != p.me) return;
    const float4 v = *reinterpret_cast<const float4*>(p.table + (size_t)own_div(p, key) * p.rowp + q * 4);
    for (int r = 0; r < p.G; ++r) *reinterpret_cast<float4*>(p.hot[r] + (size_t)h * SLOTW + q * 4) = v;
}

static int ilog2_ceil(int x) { int l = 0; while ((1 << l) < x) ++l; return l; }

}  // namespace

FMB_API int fmb_shard2_slot_floats(void) { return SLOTW; }

// Forward + loss + contributions of MY batch (see file header).  tables/inbox/dl: arrays of G peer-mapped pointers
// (entry `me` = my own buffers).  posflag: fmb_pos_flags of MY ids.  ws: fmb_bwd_workspace_bytes(B*F, k) bytes, handed
// to fmb_shard2_runs afterwards.  dl[o]: [2][G*B] floats (delta | loss) of the step's parity.
FMB_API int fmb_shard2_fused(const int32_t* ids, const float* xv, const float* y, const uint32_t* posflag,
                             void* const* tables, void* const* inbox, void* const* dl, const float* rowbox,
                             const float* hot, const int32_t* hot_base, const int32_t* field_off, const float* bias,
                             int G, int me, int B, int F, int k, int loss_kind, void* ws, size_t ws_bytes,
                             const uint32_t* wait_flags, const uint32_t* wait_epoch_words, int wait_channel, int* error,
                             cudaStream_t stream) {
    FMB_CHECK_ARG(ids && y && posflag && tables && inbox && dl && rowbox && hot && hot_base && field_off && bias && ws,
                  "fmb_shard2_fused: null pointer");
    FMB_CHECK_ARG(G >= 1 && G <= 8 && me >= 0 && me < G, "fmb_shard2_fused: bad rank %d of %d", me, G);
    FMB_CHECK_ARG(B > 0 && F > 0 && F < 512 && k > 0 && k + 1 <= SLOTW, "fmb_shard2_fused: bad shape B=%d F=%d k=%d (k <= 15)", B, F, k);
    const int64_t N = (int64_t)B * F;
    if (ws_bytes < fmb_bwd_workspace_bytes(N, k)) { fmb_set_error("fmb_shard2_fused: workspace too small"); return FMB_ERR_WS; }
    S2Params p;
    for (int o = 0; o < 8; ++o) {
        p.tables[o] = o < G ? (float*)tables[o] : nullptr;
        p.inbox[o] = o < G ? (float*)inbox[o] : nullptr;
        p.dl[o] = o < G ? (float*)dl[o] : nullptr;
    }
    p.rowbox = rowbox; p.hot = hot; p.hot_base = hot_base; p.field_off = field_off;
    p.bias = bias; p.B = B; p.F = F; p.k = k; p.rowp = fmb_round_up(k + 1, 16); p.kp4 = fmb_round_up(k, 4);
    p.cu = (k + 1 + 3) / 4; p.ql_log = ilog2_ceil(p.cu); p.jl_log = ilog2_ceil(p.kp4);
    p.loss_kind = loss_kind; p.G = G; p.me = me;
    p.gshift = -1;
    for (int l = 0; l < 4; ++l) if ((1 << l) == G) p.gshift = l;
    p.Gst = (float*)ws; p.Npad = (N + 3) / 4 * 4 + 64; p.N = N;
    p.wait.flags = wait_flags; p.wait.epoch = wait_epoch_words; p.wait.error = error; p.wait.G = G;
    p.wait.channel = (wait_flags && wait_epoch_words) ? wait_channel : -1;
    int SB = 256 >> p.jl_log;
    if (SB < 4) SB = 4;
    if (SB > 32) SB = 32;
    auto bytes = [&](int sb) {
        return sizeof(float) * ((size_t)sb * F * p.cu * 4 + (size_t)3 * sb * F + (size_t)sb * k + (size_t)sb * p.kp4 + sb);
    };
    while (SB > 1 && bytes(SB) > 48 * 1024) SB >>= 1;
    p.SB = SB;
    static bool attr_set = false;
    if (!attr_set) {
        cudaFuncSetAttribute(shard2_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        attr_set = true;
    }
    shard2_fused_kernel<<<(B + SB - 1) / SB, 256, bytes(SB), stream>>>(ids, xv, y, posflag, p);
    FMB_CHECK_LAUNCH("shard2_fused_kernel");
    return FMB_OK;
}

// my sorted keys [N] -> slab `me` of every rank's keys_all (dst: G peer-mapped pointers to [G][N] int32)
FMB_API int fmb_shard2_push_keys(const int32_t* sorted_keys, int64_t N, int G, int me, void* const* dst,
                                 cudaStream_t stream) {
    FMB_CHECK_ARG(sorted_keys && dst && N > 0 && G >= 1 && G <= 8 && me >= 0 && me < G, "fmb_shard2_push_keys: bad arguments");
    PeerI32 d;
    for (int o = 0; o < 8; ++o) d.p[o] = o < G ? (int32_t*)dst[o] : nullptr;
    push_keys_kernel<<<(unsigned)((N + 255) / 256), 256, 0, stream>>>(sorted_keys, N, G, me, d);
    FMB_CHECK_LAUNCH("push_keys_kernel");
    return FMB_OK;
}

static int fill_owner(OwnerParams& p, const int32_t* keys_all, const float* inbox, float* table, uint32_t* cnt,
                      void* const* rowbox, void* const* hot, const int32_t* hot_base, const int32_t* field_off, int G, int me,
                      int B, int F, int k, float lr, int mode) {
    FMB_CHECK_ARG(keys_all && table && hot && hot_base && field_off, "fmb_shard2 owner: null pointer");
    FMB_CHECK_ARG(G >= 1 && G <= 8 && me >= 0 && me < G && B > 0 && F > 0 && k > 0 && k + 1 <= SLOTW, "fmb_shard2 owner: bad arguments");
    FMB_CHECK_ARG((int64_t)B * F < ((int64_t)1 << 29), "fmb_shard2 owner: B*F too large");
    memset(&p, 0, sizeof(p));
    p.keys_all = keys_all; p.inbox = inbox; p.table = table; p.cnt = cnt; p.N = B * F;
    for (int o = 0; o < G; ++o) { p.rowbox[o] = rowbox ? (float*)rowbox[o] : nullptr; p.hot[o] = (float*)hot[o]; }
    p.hot_base = hot_base; p.field_off = field_off;
    p.B = B; p.F = F; p.k = k; p.rowp = fmb_round_up(k + 1, 16); p.G = G; p.me = me; p.mode = mode;
    p.gshift = -1;
    for (int l = 0; l < 4; ++l) if ((1 << l) == G) p.gshift = l;
    p.lr = lr; p.astep = -(lr / 0.1f);
    return FMB_OK;
}

// Owner side: count the ranks that hit each owned row, add their partials in rank order, update the row (and every
// rank's replica of it when the row belongs to a hot field).  keys_all [G][N], inbox [G][N][16], cnt [R_local] (zero on
// entry, zero on return) are MY buffers; hot: G peer-mapped replicas.
FMB_API int fmb_shard2_owner_apply(const int32_t* keys_all, const float* inbox, float* table, uint32_t* cnt,
                                   uint32_t* list, uint32_t* nlist, int parity, void* const* hot, const int32_t* hot_base,
                                   const int32_t* field_off, int G, int me, int B, int F, int k, float lr, int mode,
                                   const uint32_t* wait_flags, const uint32_t* wait_epoch_words, int wait_channel,
                                   int* error, cudaStream_t stream) {
    FMB_CHECK_ARG(inbox && cnt && list && nlist && (parity == 0 || parity == 1), "fmb_shard2_owner_apply: null pointer");
    FMB_CHECK_ARG(mode != 4, "fmb_shard2_owner_apply: update mode 4 (SparseAdam) is not supported by the sharded step");
    FMB_CHECK_ARG(mode == 0 || mode == 1, "fmb_shard2_owner_apply: unknown update mode %d", mode);
    OwnerParams p;
    if (int rc = fill_owner(p, keys_all, inbox, table, cnt, nullptr, hot, hot_base, field_off, G, me, B, F, k, lr, mode)) return rc;
    p.list = list; p.nlist = nlist; p.par = parity;
    p.wait.flags = wait_flags; p.wait.epoch = wait_epoch_words; p.wait.error = error; p.wait.G = G;
    p.wait.channel = (wait_flags && wait_epoch_words) ? wait_channel : -1;
    const dim3 g1((p.N + 255) / 256, G);
    owner_count_kernel<<<g1, 256, 0, stream>>>(p);
    owner_apply_kernel<<<(unsigned)(((int64_t)p.N * 4 * (G > 1 ? 2 : 1) + 255) / 256), 256, 0, stream>>>(p);   // the list holds ~N entries
    owner_reset_kernel<<<(unsigned)(((int64_t)p.N * (G > 1 ? 2 : 1) + 255) / 256), 256, 0, stream>>>(p);
    FMB_CHECK_LAUNCH("owner kernels");
    return FMB_OK;
}

// Row service: store the rows I own that the other ranks' batches (keys_all of the NEXT step) name into their rowboxes.
FMB_API int fmb_shard2_push_rows(const int32_t* keys_all, float* table, void* const* rowbox, void* const* hot,
                                 const int32_t* hot_base, const int32_t* field_off, int G, int me, int B, int F, int k,
                                 cudaStream_t stream) {
    FMB_CHECK_ARG(rowbox, "fmb_shard2_push_rows: null pointer");
    OwnerParams p;
    if (int rc = fill_owner(p, keys_all, nullptr, table, nullptr, rowbox, hot, hot_base, field_off, G, me, B, F, k, 0.f, 0)) return rc;
    if (G == 1) return FMB_OK;
    push_rows_kernel<<<dim3((p.N * 4 + 255) / 256, G), 256, 0, stream>>>(p);
    FMB_CHECK_LAUNCH("push_rows_kernel");
    return FMB_OK;
}

// my owned rows of the hot fields -> every rank's replica [R_hot][16] (after initialising / loading parameters)
FMB_API int fmb_shard2_push_hot(float* table, void* const* hot, const int32_t* hot_base, const int32_t* field_off, int R_hot,
                                int G, int me, int F, int k, cudaStream_t stream) {
    OwnerParams p;
    static const int32_t dummy = 0;
    if (int rc = fill_owner(p, &dummy, nullptr, table, nullptr, nullptr, hot, hot_base, field_off, G, me, 1, F, k, 0.f, 0)) return rc;
    if (R_hot <= 0) return FMB_OK;
    push_hot_kernel<<<(R_hot * 4 + 255) / 256, 256, 0, stream>>>(p, R_hot);
    FMB_CHECK_LAUNCH("push_hot_kernel");
    return FMB_OK;
}
