// gemm_tc.cu -- tcgen05 (5th-generation tensor core) GEMM for the DeepFM / NFM tower where it is a real
// dense contraction (BASELINE configs[3]: B = 8192, H = 400: 15.9 GFLOP per fit step; SURVEY.md 8a A4).
//
// C[M,N] = epilogue( A(M x K) * B(K x N) ), operands addressed through (row, col) strides like the SIMT
// kernel of mlp.cu, so the forward (NT), dX (NN) and dW (TN) products all map onto it.  fp32 in, fp32 out:
// every operand is split x = hi + lo with hi = x truncated to TF32, and three tcgen05.mma.kind::tf32
// products (lo*hi, hi*lo, hi*hi) accumulate in fp32 in tensor memory ("3xTF32": ~1e-6 relative, inside the
// 1e-5 tolerance of BASELINE.json; plain TF32 would be ~1e-3).
//
// One CTA computes a 128 x TBN tile (TBN = 128 or 208: 400 = 2 x 208 - 16 wastes 4 % instead of 28 %) with nine
// warps in three roles:
//   * warps 0-7 and 8-15 are two PRODUCER groups; group g stages the K-slices (32 wide) t = g, g+2, ... into its own
//     shared-memory stage.  A producer prefetches its NEXT slice from global memory into registers (two slices ahead
//     of the tensor core), waits on the stage's `empty` mbarrier, splits and stores the current one, then arrives on
//     the stage's `full` mbarrier.  The canonical K-major no-swizzle core-matrix layout is chosen for the staging:
//     8-row groups are contiguous (SBO = 128 B) and the K-direction stride is rows*16 + 16 B (LBO), so the 16-byte
//     chunk (row r, k-chunk c) sits at c*LBO + r*16 and both a K-contiguous source (lanes = 8 k-chunks x 4 rows)
//     and a row-contiguous source (lanes = 32 rows) store conflict-free.  Sixteen warps because the staging code
//     is a dependent chain per warp (~6 cycles per instruction): the slice period is set by warp count, not by
//     bandwidth (ncu: 4 warps per scheduler needed to get under the 1080 cycles the 12 MMAs of a slice take);
//   * one thread of warp 16 is the MMA ISSUER: wait `full`, 12 tcgen05.mma (4 k-steps x {lo*hi, hi*lo, hi*hi}),
//     tcgen05.commit on `empty`; the tensor core runs slice t while the producers stage t+1 and fetch t+2;
//   * the sixteen producer warps then drain TMEM (tcgen05.ld, lane = row) through shared memory so that the bias /
//     relu-mask loads and the C stores are row-contiguous 16-byte accesses.
// K is also split across CTAs (blockIdx.z) when the tile grid alone cannot fill 148 SMs (the dW product:
// M = N = 400, K = batch) and whenever one pass would accumulate more than 1024 terms in TMEM (the tensor
// core's fp32 accumulator truncates; error grows with the K of one pass).  Split partials go to a workspace
// and a second kernel adds them in split order and applies the epilogue, so results are run-to-run identical.
//
// This path is NOT bit-comparable with the oracle (the tensor core's summation order is not the oracle's
// left-to-right FMA chain); mlp.cu picks it only for large shapes and tests compare it within tolerance.
#include "fmb_common.cuh"

namespace {

constexpr int TBM = 128, TBK = 32;
constexpr int PRODUCERS = 512, GROUP = 256;         // two producer groups of eight warps
constexpr int TC_THREADS = PRODUCERS + 32;          // + the MMA-issuing warp
constexpr int KCH = TBK / 4;                        // 16-byte k-chunks per slice
constexpr int MAX_K_PER_PASS = 1024;

struct TcParams {
    const float* A; int64_t sam, sak;
    const float* B; int64_t sbk, sbn;
    float* C; int64_t scm;
    int M, N, K;
    int kchunk;              // K range of one split (multiple of TBK); gridDim.z splits
    int epi;                 // 0 none, 1 bias+relu, 2 mask
    const float* bias;
    const float* mask; int64_t smm;
    float* colsum;           // colsum[m] = sum_k A(m,k)
    float* ws;               // split partials [splits][M][N] (gridDim.z > 1)
    float* wsc;              // split partial column sums [splits][M]
    int* error;              // set to 1 if an mbarrier wait times out (never expected)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;   // K-direction stride between core matrices
    d |= (uint64_t)((128u >> 4) & 0x3FFF) << 32;        // SBO: 8-row groups are contiguous
    d |= (uint64_t)1 << 46;                             // descriptor version of sm_100
    return d;                                           // base offset 0, swizzle mode 0 (none)
}

__device__ __forceinline__ void mma_tf32(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}

__device__ __forceinline__ void mbar_init(uint64_t* b, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(b)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) {
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}\n" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* b) {   // arrives when every MMA issued so far has completed
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(b)) : "memory");
}
__device__ __forceinline__ bool mbar_wait(uint64_t* b, uint32_t parity) {
    const uint32_t addr = smem_u32(b);
    for (int spin = 0; spin < (1 << 22); ++spin) {
        uint32_t r;
        asm volatile("{\n\t.reg .pred q;\n\tmbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\tselp.u32 %0, 1, 0, q;\n\t}\n"
                     : "=r"(r) : "r"(addr), "r"(parity) : "memory");
        if (r) return true;
    }
    return false;
}

// One operand's K-slice held in the registers of one producer group (256 threads, warps w8 = 0..7):
//   K-contiguous source   : slot j = (row (lane>>3) + 4*w8 + 32*j, k-chunk lane&7)
//   row-contiguous source : slot j = (row lane + 32*j,             k-chunk w8)
// Row validity and the per-thread base pointer do not depend on the slice, so they are set up once (init);
// slices that lie entirely inside [kbeg, kend) take the check-free path.
template <int ROWS>
struct Slice {
    static constexpr int NV = (ROWS + 31) / 32;
    static constexpr int LBO = ROWS * 16 + 16;
    float4 v[NV];
    const float* base;   // element (first row of this thread, k = first k of this thread's chunk at k0 = 0)
    int64_t jstep, sk;   // pointer step between slots; k stride
    int nvalid;          // slots j < nvalid are inside the matrix (and the tile)
    int soff;            // byte offset of slot 0 in the stage
    bool kcontig, vec;

    __device__ __forceinline__ void init(const float* src, int64_t srow, int64_t sk_, int row0, int rows_valid, int w8, int lane) {
        kcontig = (sk_ == 1);
        sk = sk_;
        vec = kcontig && (srow % 4 == 0) && ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
        const int r0 = kcontig ? (lane >> 3) + 4 * w8 : lane;
        const int lim = min(ROWS, rows_valid - row0) - r0;          // rows r0 + 32 j < limit
        nvalid = lim <= 0 ? 0 : (lim + 31) / 32;
        if (kcontig) { base = src + (int64_t)(row0 + r0) * srow + 4 * (lane & 7); jstep = 32 * srow; soff = (lane & 7) * LBO + r0 * 16; }
        else { base = src + (int64_t)(4 * w8) * sk_ + (row0 + r0) * srow; jstep = 32 * srow; soff = w8 * LBO + r0 * 16; }
    }

    __device__ __forceinline__ void load(int k0, int kend, int w8, int lane) {
        if (k0 + TBK <= kend) {   // whole slice in range (block-uniform)
            if (kcontig && vec) {
                const float* q = base + k0;
#pragma unroll
                for (int j = 0; j < NV; ++j)
                    v[j] = j < nvalid ? *reinterpret_cast<const float4*>(q + j * jstep) : make_float4(0.f, 0.f, 0.f, 0.f);
            } else {
                const int64_t ks = kcontig ? 1 : sk;
                const float* q = base + (int64_t)k0 * ks;
#pragma unroll
                for (int j = 0; j < NV; ++j) {
                    float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (j < nvalid) { const float* r = q + j * jstep; x.x = r[0]; x.y = r[ks]; x.z = r[2 * ks]; x.w = r[3 * ks]; }
                    v[j] = x;
                }
            }
        } else {                  // last, partial slice: per-element K checks
            const int64_t ks = kcontig ? 1 : sk;
            const int gk = k0 + 4 * (kcontig ? (lane & 7) : w8);
            const float* q = base + (int64_t)k0 * ks;
#pragma unroll
            for (int j = 0; j < NV; ++j) {
                float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                if (j < nvalid) {
                    const float* r = q + j * jstep;
                    if (gk < kend) x.x = r[0];
                    if (gk + 1 < kend) x.y = r[ks];
                    if (gk + 2 < kend) x.z = r[2 * ks];
                    if (gk + 3 < kend) x.w = r[3 * ks];
                }
                v[j] = x;
            }
        }
    }

    // split into TF32 hi + remainder lo and store into the stage (rows beyond the matrix hold zeros)
    __device__ __forceinline__ void store(unsigned char* hi, unsigned char* lo, int w8, int lane) const {
        const int r0 = kcontig ? (lane >> 3) + 4 * w8 : lane;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            if (ROWS % 32 != 0 && j == NV - 1 && r0 + 32 * j >= ROWS) continue;
            const float4 x = v[j];
            float4 h, l;
            h.x = __uint_as_float(__float_as_uint(x.x) & 0xFFFFE000u); l.x = x.x - h.x;
            h.y = __uint_as_float(__float_as_uint(x.y) & 0xFFFFE000u); l.y = x.y - h.y;
            h.z = __uint_as_float(__float_as_uint(x.z) & 0xFFFFE000u); l.z = x.z - h.z;
            h.w = __uint_as_float(__float_as_uint(x.w) & 0xFFFFE000u); l.w = x.w - h.w;
            *reinterpret_cast<float4*>(hi + soff + j * 512) = h;
            *reinterpret_cast<float4*>(lo + soff + j * 512) = l;
        }
    }
};

template <int TBN>
__global__ void __launch_bounds__(TC_THREADS, 1) gemm_tc_kernel(TcParams p) {
    constexpr int LBO_A = Slice<TBM>::LBO, LBO_B = Slice<TBN>::LBO;
    constexpr int A_BYTES = KCH * LBO_A, B_BYTES = KCH * LBO_B;
    constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    constexpr int TMEM_COLS = TBN <= 128 ? 128 : 256;
    constexpr int PITCH = TBN + 4;                       // epilogue tile row pitch (floats): conflict-free 16-B stores
    constexpr int TILE_BYTES = TBM * PITCH * 4;
    constexpr int NPART = 16;                            // partial column sums per row (8 per group)
    static_assert(TILE_BYTES + NPART * TBM * 4 <= 2 * STAGE_BYTES, "epilogue tile must fit in the idle ring");
    static_assert(TBN % 16 == 0, "four column quarters of whole 4-column TMEM loads");
    extern __shared__ __align__(1024) unsigned char tc_smem[];
    __shared__ __align__(8) uint64_t full_bar[2], empty_bar[2], done_bar;
    __shared__ uint32_t tmem_base_s;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.y * TBM, n0 = blockIdx.x * TBN;
    const int kbeg = blockIdx.z * p.kchunk, kend = min(p.K, kbeg + p.kchunk);
    const int T = (kend - kbeg + TBK - 1) / TBK;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(&tmem_base_s)), "n"(TMEM_COLS));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n");
    }
    if (tid == 32) {
        mbar_init(&full_bar[0], GROUP); mbar_init(&full_bar[1], GROUP);
        mbar_init(&empty_bar[0], 1); mbar_init(&empty_bar[1], 1);
        mbar_init(&done_bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem = tmem_base_s;
    const bool do_colsum = p.colsum && blockIdx.x == 0;
    bool ok = true;

    if (warp == PRODUCERS / 32) {
        // ------------------------------------------------------------------ MMA issuer
        if (lane == 0) {
            // instruction descriptor: D = F32, A = B = TF32, both K-major, N = TBN, M = 128
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(TBN >> 3) << 17) | ((uint32_t)(TBM >> 4) << 24);
            for (int t = 0; t < T; ++t) {
                const int g = t & 1;
                ok &= mbar_wait(&full_bar[g], (t >> 1) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
                const uint32_t ah = smem_u32(tc_smem + g * STAGE_BYTES), al = ah + A_BYTES, bh = ah + 2 * A_BYTES, bl = bh + B_BYTES;
#pragma unroll
                for (int q = 0; q < TBK / 8; ++q) {   // one MMA consumes K = 8 (two core matrices along K)
                    const uint32_t ao = q * 2 * LBO_A, bo = q * 2 * LBO_B;
                    mma_tf32(tmem, make_desc(al + ao, LBO_A), make_desc(bh + bo, LBO_B), idesc, (t | q) ? 1u : 0u);
                    mma_tf32(tmem, make_desc(ah + ao, LBO_A), make_desc(bl + bo, LBO_B), idesc, 1u);
                    mma_tf32(tmem, make_desc(ah + ao, LBO_A), make_desc(bh + bo, LBO_B), idesc, 1u);
                }
                mma_commit(&empty_bar[g]);   // the stage may be refilled once these MMAs have read it
            }
            mma_commit(&done_bar);
            if (!ok && p.error) *p.error = 1;
        }
    } else {
        // ------------------------------------------------------------------ producers, then epilogue
        const int g = warp >> 3, w8 = warp & 7;
        Slice<TBM> sa;
        Slice<TBN> sb;
        sa.init(p.A, p.sam, p.sak, m0, p.M, w8, lane);
        sb.init(p.B, p.sbn, p.sbk, n0, p.N, w8, lane);
        float ps[Slice<TBM>::NV];   // partial row sums of A (4 rows per thread)
#pragma unroll
        for (int j = 0; j < Slice<TBM>::NV; ++j) ps[j] = 0.f;
        unsigned char* st = tc_smem + g * STAGE_BYTES;
        if (g < T) {
            sa.load(kbeg + g * TBK, kend, w8, lane);
            sb.load(kbeg + g * TBK, kend, w8, lane);
        }
        for (int t = g; t < T; t += 2) {
            const int n = t >> 1;
            if (n >= 1) ok &= mbar_wait(&empty_bar[g], (n - 1) & 1);   // the MMAs of slice t-2 have read this stage
            sa.store(st, st + A_BYTES, w8, lane);
            sb.store(st + 2 * A_BYTES, st + 2 * A_BYTES + B_BYTES, w8, lane);
            if (do_colsum) {
#pragma unroll
                for (int j = 0; j < Slice<TBM>::NV; ++j) ps[j] += (sa.v[j].x + sa.v[j].y) + (sa.v[j].z + sa.v[j].w);
            }
            if (t + 2 < T) {
                sa.load(kbeg + (t + 2) * TBK, kend, w8, lane);
                sb.load(kbeg + (t + 2) * TBK, kend, w8, lane);
            }
            asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");   // generic smem writes -> tensor-core proxy
            mbar_arrive(&full_bar[g]);
        }
        ok &= mbar_wait(&done_bar, 0);   // every MMA has completed: accumulator final, ring idle
        if (!ok && p.error) *p.error = 1;
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");

        float* tile = reinterpret_cast<float*>(tc_smem);                 // [128][PITCH]
        float* red = reinterpret_cast<float*>(tc_smem + TILE_BYTES);     // [NPART][128]
        // ---- TMEM -> shared: warp w reads lanes [32(w&3), +32) = rows 32(w&3) + lane, column quarter w>>2
        {
            const int row = (warp & 3) * 32 + lane;
            const int cbeg = (warp >> 2) * (TBN / 4);
#pragma unroll 1
            for (int c0 = cbeg; c0 < cbeg + TBN / 4; c0 += 4) {
                if (n0 + c0 >= p.N) break;   // warp-uniform
                uint32_t v[4];
                const uint32_t taddr = tmem + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)c0;
                asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n"
                             : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr));
                asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
                *reinterpret_cast<float4*>(tile + row * PITCH + c0) =
                    make_float4(__uint_as_float(v[0]), __uint_as_float(v[1]), __uint_as_float(v[2]), __uint_as_float(v[3]));
            }
        }
        if (do_colsum) {
            const int part = 8 * g + (sa.kcontig ? (lane & 7) : w8);
            const int r0 = sa.kcontig ? (lane >> 3) + 4 * w8 : lane;
#pragma unroll
            for (int j = 0; j < Slice<TBM>::NV; ++j) red[part * TBM + r0 + 32 * j] = ps[j];
        }
        asm volatile("bar.sync 1, %0;\n" ::"n"(PRODUCERS) : "memory");
        if (do_colsum && tid < TBM && m0 + tid < p.M) {
            float c = 0.f;
#pragma unroll
            for (int q = 0; q < NPART; ++q) c += red[q * TBM + tid];
            if (gridDim.z > 1) p.wsc[(size_t)blockIdx.z * p.M + m0 + tid] = c;
            else p.colsum[m0 + tid] = c;
        }
        // ---- shared -> global: a warp owns rows warp, warp+16, ...; lanes along n, 16 bytes each
        {
            const bool split = gridDim.z > 1;
            const int ncols = min(TBN, p.N - n0);
            const int64_t ldc = split ? p.N : p.scm;
            float* cbase = split ? p.ws + (size_t)blockIdx.z * p.M * p.N : p.C;
            const int epi = split ? 0 : p.epi;
            const bool vec = (ldc % 4 == 0) && ((reinterpret_cast<uintptr_t>(cbase) & 15) == 0) && (ncols % 4 == 0) &&
                             (epi != 2 || ((p.smm % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.mask) & 15) == 0))) &&
                             (epi != 1 || ((reinterpret_cast<uintptr_t>(p.bias) & 15) == 0));
            constexpr int RPW = TBM / 16;   // 8 rows per warp
            if (vec) {
                const int nc4 = ncols >> 2;
#pragma unroll 1
                for (int c4 = lane; c4 < nc4; c4 += 32) {
                    const int gn = n0 + 4 * c4;
                    float4 bv = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (epi == 1) bv = *reinterpret_cast<const float4*>(p.bias + gn);
#pragma unroll
                    for (int rb = 0; rb < RPW; rb += 4) {   // four rows in flight: mask loads first, stores last
                        float4 mk[4], x[4];
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int r = warp + 16 * (rb + i), gm = m0 + r;
                            mk[i] = make_float4(1.f, 1.f, 1.f, 1.f);
                            if (epi == 2 && gm < p.M) mk[i] = *reinterpret_cast<const float4*>(p.mask + gm * p.smm + gn);
                            x[i] = *reinterpret_cast<const float4*>(tile + r * PITCH + 4 * c4);
                        }
#pragma unroll
                        for (int i = 0; i < 4; ++i) {
                            const int gm = m0 + warp + 16 * (rb + i);
                            if (gm >= p.M) continue;
                            float4 y = x[i];
                            if (epi == 1) {
                                y.x = fmaxf(__fadd_rn(y.x, bv.x), 0.f); y.y = fmaxf(__fadd_rn(y.y, bv.y), 0.f);
                                y.z = fmaxf(__fadd_rn(y.z, bv.z), 0.f); y.w = fmaxf(__fadd_rn(y.w, bv.w), 0.f);
                            } else if (epi == 2) {
                                y.x = mk[i].x > 0.f ? y.x : 0.f; y.y = mk[i].y > 0.f ? y.y : 0.f;
                                y.z = mk[i].z > 0.f ? y.z : 0.f; y.w = mk[i].w > 0.f ? y.w : 0.f;
                            }
                            *reinterpret_cast<float4*>(cbase + gm * ldc + gn) = y;
                        }
                    }
                }
            } else {
                for (int r = warp; r < TBM; r += 16) {
                    const int gm = m0 + r;
                    if (gm >= p.M) break;
                    for (int c = lane; c < ncols; c += 32) {
                        const int gn = n0 + c;
                        float x = tile[r * PITCH + c];
                        if (epi == 1) { x = __fadd_rn(x, p.bias[gn]); x = x > 0.f ? x : 0.f; }
                        else if (epi == 2) { x = p.mask[gm * p.smm + gn] > 0.f ? x : 0.f; }
                        cbase[gm * ldc + gn] = x;
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "n"(TMEM_COLS));
}

// C = epilogue( sum over splits, in split order ); colsum likewise
__global__ void splitk_reduce_kernel(TcParams p, int splits) {
    const int64_t total = (int64_t)p.M * p.N;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < total) {
        float x = 0.f;
        for (int s = 0; s < splits; ++s) x = __fadd_rn(x, p.ws[(size_t)s * total + i]);
        const int gm = (int)(i / p.N), gn = (int)(i % p.N);
        if (p.epi == 1) { x = __fadd_rn(x, p.bias[gn]); x = x > 0.f ? x : 0.f; }
        else if (p.epi == 2) { x = p.mask[gm * p.smm + gn] > 0.f ? x : 0.f; }
        p.C[gm * p.scm + gn] = x;
    }
    if (p.colsum && i < p.M) {
        float c = 0.f;
        for (int s = 0; s < splits; ++s) c = __fadd_rn(c, p.wsc[(size_t)s * p.M + i]);
        p.colsum[i] = c;
    }
}

template <int TBN>
constexpr size_t tc_smem_bytes() { return (size_t)2 * (2 * KCH * (TBM * 16 + 16) + 2 * KCH * (TBN * 16 + 16)) + 1024; }

}  // namespace

static int* g_tc_error = nullptr;
static float* g_tc_ws = nullptr;   // split-K workspace; a grown one replaces it but none is freed (fmb_gemm_tc_launch)
static size_t g_tc_ws_bytes = 0;
static int g_tc_sms = 0;

// C = epilogue(A * B) on the tensor cores (see file header). Same operand convention as mlp.cu's gemm.
int fmb_gemm_tc_launch(const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbk, int64_t sbn, float* C,
                       int64_t scm, int M, int N, int K, int epi, const float* bias, const float* mask, int64_t smm,
                       float* colsum, cudaStream_t stream) {
    if (!g_tc_error) {
        if (cudaMalloc(&g_tc_error, sizeof(int)) != cudaSuccess) return FMB_ERR_CUDA;
        cudaMemset(g_tc_error, 0, sizeof(int));
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_tc_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_tc_sms <= 0) g_tc_sms = 148;
        cudaFuncSetAttribute(gemm_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes<128>());
        cudaFuncSetAttribute(gemm_tc_kernel<208>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc_smem_bytes<208>());
    }
    // tile width: the one that wastes less of N (ties -> 128)
    const int n128 = (N + 127) / 128, n208 = (N + 207) / 208;
    const int tbn = (n208 * 208 < n128 * 128) ? 208 : 128;
    const int tiles = ((M + TBM - 1) / TBM) * (tbn == 208 ? n208 : n128);
    // K splits: enough CTAs for one wave, and never more than MAX_K_PER_PASS terms in one TMEM pass
    int splits = 1;
    if (tiles * 2 <= g_tc_sms) splits = g_tc_sms / tiles;
    splits = max(splits, (K + MAX_K_PER_PASS - 1) / MAX_K_PER_PASS);
    splits = min(splits, (K + 4 * TBK - 1) / (4 * TBK));   // at least 4 slices per split
    splits = max(splits, 1);
    int kchunk = ((K + splits - 1) / splits + TBK - 1) / TBK * TBK;
    splits = (K + kchunk - 1) / kchunk;
    TcParams p;
    p.A = A; p.sam = sam; p.sak = sak; p.B = B; p.sbk = sbk; p.sbn = sbn; p.C = C; p.scm = scm;
    p.M = M; p.N = N; p.K = K; p.kchunk = kchunk; p.epi = epi; p.bias = bias; p.mask = mask; p.smm = smm; p.colsum = colsum;
    p.error = g_tc_error; p.ws = nullptr; p.wsc = nullptr;
    if (splits > 1) {
        const size_t need = ((size_t)splits * M * N + (size_t)splits * M) * sizeof(float);
        if (need > g_tc_ws_bytes) {
            // the superseded buffer stays allocated for the life of the process: launches still in flight and CUDA
            // graphs captured earlier (deep.py's fit graphs) hold its address.  Each new buffer is at least twice the
            // last, so the kept ones total less than the current one.
            const size_t bytes = need > 2 * g_tc_ws_bytes ? need : 2 * g_tc_ws_bytes;
            float* grown = nullptr;
            if (cudaMalloc(&grown, bytes) != cudaSuccess) { fmb_set_error("gemm_tc: cannot allocate %zu workspace bytes", bytes); return FMB_ERR_CUDA; }
            g_tc_ws = grown;
            g_tc_ws_bytes = bytes;
        }
        p.ws = g_tc_ws;
        p.wsc = g_tc_ws + (size_t)splits * M * N;
    }
    dim3 grid(tbn == 208 ? n208 : n128, (M + TBM - 1) / TBM, splits);
    if (tbn == 208) gemm_tc_kernel<208><<<grid, TC_THREADS, tc_smem_bytes<208>(), stream>>>(p);
    else gemm_tc_kernel<128><<<grid, TC_THREADS, tc_smem_bytes<128>(), stream>>>(p);
    if (splits > 1) {
        const int64_t total = (int64_t)M * N;
        splitk_reduce_kernel<<<(unsigned)((total + 255) / 256), 256, 0, stream>>>(p, splits);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { fmb_set_error("gemm_tc_kernel: %s", cudaGetErrorString(e)); return FMB_ERR_CUDA; }
    return FMB_OK;
}

// 1 if a tensor-core GEMM ever timed out on its mbarrier (diagnostic)
FMB_API int fmb_gemm_tc_error(void) {
    int v = 0;
    if (g_tc_error) cudaMemcpy(&v, g_tc_error, sizeof(int), cudaMemcpyDeviceToHost);
    return v;
}

// Standalone tensor-core GEMM for tests: C[M,N] = A[M,K] * B[N,K]^T (both row-major, K contiguous).
FMB_API int fmb_gemm_tc_nt(const float* A, const float* B, float* C, int M, int N, int K, cudaStream_t stream) {
    FMB_CHECK_ARG(A && B && C && M > 0 && N > 0 && K > 0, "fmb_gemm_tc_nt: bad arguments");
    return fmb_gemm_tc_launch(A, K, 1, B, 1, K, C, N, M, N, K, 0, nullptr, nullptr, 0, nullptr, stream);
}

// Same through arbitrary strides and the fused epilogues (tests of the TN / NN forms):
//   C[m*scm + n] = epi( sum_k A[m*sam + k*sak] * B[k*sbk + n*sbn] ), colsum[m] = sum_k A(m,k) (nullable)
FMB_API int fmb_gemm_tc_strided(const float* A, int64_t sam, int64_t sak, const float* B, int64_t sbk, int64_t sbn,
                                float* C, int64_t scm, int M, int N, int K, int epi, const float* bias,
                                const float* mask, int64_t smm, float* colsum, cudaStream_t stream) {
    FMB_CHECK_ARG(A && B && C && M > 0 && N > 0 && K > 0, "fmb_gemm_tc_strided: bad arguments");
    FMB_CHECK_ARG(epi >= 0 && epi <= 2 && (epi != 1 || bias) && (epi != 2 || mask), "fmb_gemm_tc_strided: bad epilogue");
    return fmb_gemm_tc_launch(A, sam, sak, B, sbk, sbn, C, scm, M, N, K, epi, bias, mask, smm, colsum, stream);
}
