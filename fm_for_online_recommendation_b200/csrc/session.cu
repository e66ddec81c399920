// session.cu -- a training session: owns every temporary of the hot path (device workspaces and
// pinned host staging) so that one C call performs a whole `update_embedding` / `fit` step.
//
// This is the drop-in boundary for the FM training step: the entry points take plain pointers and
// sizes; `*_host` variants take HOST buffers and do the H2D/D2H copies themselves (what a maintainer
// of the reference would bind in place of fm_adam.py:56-82 / deepfm_adam.py:91-117).
#include "fmb_common.cuh"
#include <cstdlib>
#include <cstring>
#include <cstddef>
#include <new>

extern "C" {
int fmb_fm_forward(const int32_t*, const float*, const float*, const float*, int, int, int, float*, float*, float*,
                   float*, float*, const float*, int, float*, float*, cudaStream_t);
size_t fmb_sort_workspace_bytes(int64_t);
int fmb_sort_segment(const int32_t*, int64_t, int, void*, size_t, int32_t*, int32_t*, int32_t*, int32_t*,
                     cudaStream_t);
size_t fmb_bwd_workspace_bytes(int64_t, int);
int fmb_sort_fields_max_batch(void);
struct fmb_runlist_t { int32_t* entries; uint32_t* seg_count; int nseg, seg_cap; };
void fmb_runlist_shape(int, int, int*, int*);
int fmb_sort_fields_ex(const int32_t*, int, int, const int32_t*, int32_t*, int32_t*, uint32_t*, const fmb_runlist_t*, int, cudaStream_t);
int fmb_pos_flags_ex(const int32_t*, const int32_t*, int64_t, uint32_t*, const fmb_runlist_t*, cudaStream_t);
int fmb_fm_backward_update(const int32_t*, const int32_t*, int64_t, const float*, float*, int, int, const float*,
                           const float*, int, const float*, float, int, void*, size_t, cudaStream_t);
int fmb_finish_step(const float*, const float*, int, float*, float, int, float*, cudaStream_t);
struct fmb_ftrl_t { float* zn; float* bias_zn; float beta, l1, l2; };
struct fmb_adagrad_t { float* sums; float* bias_sum; float* mlp_sums; float eps; };
int fmb_fm_backward_runs_list(const int32_t*, int64_t, float*, int, int, float, int, const fmb_ftrl_t*, const fmb_runlist_t*,
                              void*, size_t, cudaStream_t);
int fmb_finish_step_ex(const float*, const float*, int, float*, float, int, const fmb_ftrl_t*, float*, cudaStream_t);
int fmb_fm_step_fused_ex(const int32_t*, const float*, const float*, float*, const float*, const uint32_t*, int, int, int,
                         int, float, int, const fmb_ftrl_t*, float*, float*, void*, size_t, cudaStream_t);
int fmb_fm_backward_runs_ex(const int32_t*, int64_t, float*, int, int, float, int, const fmb_ftrl_t*, void*, size_t,
                            cudaStream_t);
int fmb_pos_flags(const int32_t*, const int32_t*, int64_t, uint32_t*, cudaStream_t);
int fmb_fm_step_fused(const int32_t*, const float*, const float*, float*, const float*, const uint32_t*, int, int, int,
                      int, float, int, float*, float*, void*, size_t, cudaStream_t);
int fmb_fm_backward_runs(const int32_t*, int64_t, float*, int, int, float, int, void*, size_t, cudaStream_t);
int fmb_is_fused_kernel_fn(const void*);
void fmb_runs_list_next_is_dependent(int);
const void* fmb_finish_kernel_fn(void);
int fmb_sort_fields_kernel_fns(const void**, int*, int*);
}

// One captured step graph per CONFIGURATION (batch size, loss, update mode, with/without xv, sorted in the step or
// before it, with/without the sort of the next batch riding along) -- never per batch: the per-batch pointers
// (ids, xv, y of the fused kernel; ids of the sort kernels) are re-pointed before every launch with
// cudaGraphExecKernelNodeSetParams, so a training loop over a device-resident dataset replays ONE graph.
#define FMB_GRAPH_CACHE 32
struct StepVariant {
    int B, key_bits, loss_kind, mode, has_xv, pre, has_next, cur;
    const void *table, *bias;
    float lr;
    cudaGraph_t graph;        // kept alive: its nodes own the argument storage the patches start from
    cudaGraphExec_t exec;
    cudaGraphNode_t n_fused, n_finish, n_sort_cur[2], n_sort_next[2];   // a per-field sort is up to two kernels (radix + sparse fields)
    int np_sort_cur[2], np_sort_next[2];
    int nlaunch;
    // per-batch pointers the nodes currently hold: a node is only re-pointed when its pointers change (a host loop over
    // two input slots, or one resident batch, replays the graph as it is)
    const void *cur_ids, *cur_xv, *cur_y, *cur_sort_ids, *cur_next_ids, *cur_loss;
};

struct fmb_session {
    int F, k, rowp, kp4;
    int64_t maxB;
    // device
    int32_t* d_ids;
    float* d_xv;
    float* d_y;
    float* d_S;
    float* d_z;
    float* d_delta;
    float* d_lossv;
    float* d_loss;
    int32_t* d_skeys;   // sorted keys / permutation of the step being run (points into the two buffers below)
    int32_t* d_perm;
    int32_t* d_skeys_buf[2];
    int32_t* d_perm_buf[2];
    uint32_t* d_posflag_buf[2];   // per entry: sorted position | multi-hit flag (fmb_pos_flags), one per sorted buffer
    int32_t* d_runlist_buf[2];    // runs of >= 2 entries {position, key, n0, 0} found by the sort: [rl_nseg][rl_cap][4]
    uint32_t* d_runcount_buf[2];  // entries per segment [rl_nseg]
    int rl_nseg, rl_cap;          // shape for the largest batch (fmb_runlist_shape)
    void* d_sort_ws2;             // radix workspace of the pre-sort (the in-step sort may be using d_sort_ws)
    // pre-sort: the sort depends on the ids only, so the sort of batch t+1 may run (on st1) while step t is
    // still in its backward kernels.  presort_ids names the batch whose sorted form sits in presort_buf.
    const int32_t* presort_ids;
    int presort_B, presort_buf, last_buf;
    int presort_ext;     // the pending pre-sort ran outside a step graph: steps must wait for ev_presort
    int presort_stale;   // set by fmb_session_presort_invalidate
    cudaEvent_t ev_presort, ev_buf_free[2];
    int buf_used[2];
    void* d_sort_ws;
    size_t sort_ws_bytes;
    void* d_bwd_ws;
    size_t bwd_ws_bytes;
    int32_t* d_field_off;  // [F+1] global row offset of every field (enables the per-field sort)
    // pinned host staging
    int32_t* h_ids;
    float* h_xv;
    float* h_y;
    float* h_loss;
    // second input slot + copy stream for the pipelined host entry point (slot 0 = the buffers above)
    int32_t* d_ids2; float* d_xv2; float* d_y2; float* d_loss2;
    int32_t* h_ids2; float* h_xv2; float* h_y2;
    // slots 2 and 3 (allocated on first use): with four slots the host runs up to three steps ahead of the GPU
    int32_t* d_idsx[2]; float* d_xvx[2]; float* d_yx[2];
    int32_t* h_idsx[2]; float* h_xvx[2]; float* h_yx[2];
    cudaStream_t st_copy;
    cudaEvent_t ev_h2d[4], ev_done[4];
    int slot_used[4];
    int64_t launches;  // kernels launched through this session (bench.py's gpu_launches)
    // CUDA-graph cache of whole steps, keyed by every argument that is baked into the kernels
    cudaStream_t st0, st1, st2, st3, st4;   // st0/st1: graph capture (main / side branch); st2: pre-sorts; st3: sparse-field
                                            // part of a sort; st4: long runs of the run kernel
    cudaEvent_t ev_sp_fork, ev_sp_join, ev_join4;
    int64_t steps_done;
    cudaEvent_t ev_fork, ev_fwd, ev_sort, ev_join;
    int use_graph, use_prio;
    int host_path;         // set while fmb_session_fm_step_host_async runs its step (one graph per input slot)
    int use_pdl;           // FMB_PDL=0 switches the programmatic dependent launch of the run kernel off
    int sort_after;        // FMB_SORT_AFTER=1 (experiment; default 0): the next batch's sort waits for the fused kernel
    int sparse_ok;         // FMB_SORT_SPARSE_OK unless FMB_SPARSE=0: fields with >= 16*B rows skip the sort (radix_sort.cu)
    int ngraphs, next_evict;
    StepVariant gvar[FMB_GRAPH_CACHE];
    cudaEvent_t ev_join2;
    // graphs of stand-alone pre-sorts (host entry point: one per input slot and sorted buffer), keyed by ids pointer
    struct { const int32_t* ids; int B, key_bits, buf, nl; cudaGraphExec_t exec; cudaGraph_t graph; } psg[8];
    int npsg, presort_warm;
    fmb_ftrl_t ftrl;       // update mode 2 (fmb_session_set_ftrl)
    int ftrl_set;
    fmb_adagrad_t ada;     // update mode 3 (fmb_session_set_adagrad)
    int ada_set;
};

#define CU(call)                                                                              \
    do {                                                                                      \
        cudaError_t e__ = (call);                                                             \
        if (e__ != cudaSuccess) { fmb_set_error("%s: %s", #call, cudaGetErrorString(e__)); return FMB_ERR_CUDA; } \
    } while (0)

FMB_API void fmb_session_destroy(fmb_session* s) {
    if (!s) return;
    cudaFree(s->d_ids); cudaFree(s->d_xv); cudaFree(s->d_y); cudaFree(s->d_S); cudaFree(s->d_z);
    cudaFree(s->d_delta); cudaFree(s->d_lossv); cudaFree(s->d_loss);
    for (int i = 0; i < 2; ++i) { cudaFree(s->d_skeys_buf[i]); cudaFree(s->d_perm_buf[i]); cudaFree(s->d_posflag_buf[i]); cudaFree(s->d_runlist_buf[i]); cudaFree(s->d_runcount_buf[i]); if (s->ev_buf_free[i]) cudaEventDestroy(s->ev_buf_free[i]); }
    cudaFree(s->d_sort_ws2);
    if (s->ev_join2) cudaEventDestroy(s->ev_join2);
    for (int i = 0; i < s->npsg; ++i) if (s->psg[i].exec) { cudaGraphExecDestroy(s->psg[i].exec); cudaGraphDestroy(s->psg[i].graph); }
    if (s->ev_sp_fork) cudaEventDestroy(s->ev_sp_fork);
    if (s->ev_sp_join) cudaEventDestroy(s->ev_sp_join);
    if (s->st3) cudaStreamDestroy(s->st3);
    if (s->st4) cudaStreamDestroy(s->st4);
    if (s->ev_join4) cudaEventDestroy(s->ev_join4);
    if (s->ev_presort) cudaEventDestroy(s->ev_presort);
    cudaFree(s->d_sort_ws); cudaFree(s->d_bwd_ws); cudaFree(s->d_field_off);
    cudaFreeHost(s->h_ids); cudaFreeHost(s->h_xv); cudaFreeHost(s->h_y); cudaFreeHost(s->h_loss);
    cudaFree(s->d_ids2); cudaFree(s->d_xv2); cudaFree(s->d_y2); cudaFree(s->d_loss2);
    cudaFreeHost(s->h_ids2); cudaFreeHost(s->h_xv2); cudaFreeHost(s->h_y2);
    if (s->st_copy) cudaStreamDestroy(s->st_copy);
    for (int i = 0; i < 4; ++i) { if (s->ev_h2d[i]) cudaEventDestroy(s->ev_h2d[i]); if (s->ev_done[i]) cudaEventDestroy(s->ev_done[i]); }
    for (int i = 0; i < 2; ++i) {
        cudaFree(s->d_idsx[i]); cudaFree(s->d_xvx[i]); cudaFree(s->d_yx[i]);
        cudaFreeHost(s->h_idsx[i]); cudaFreeHost(s->h_xvx[i]); cudaFreeHost(s->h_yx[i]);
    }
    for (int i = 0; i < s->ngraphs; ++i) { cudaGraphExecDestroy(s->gvar[i].exec); cudaGraphDestroy(s->gvar[i].graph); }
    if (s->st0) cudaStreamDestroy(s->st0);
    if (s->st1) cudaStreamDestroy(s->st1);
    if (s->st2) cudaStreamDestroy(s->st2);
    if (s->ev_fork) cudaEventDestroy(s->ev_fork);
    if (s->ev_fwd) cudaEventDestroy(s->ev_fwd);
    if (s->ev_sort) cudaEventDestroy(s->ev_sort);
    if (s->ev_join) cudaEventDestroy(s->ev_join);
    delete s;
}

// F fields, embedding size k, up to max_batch samples per step.  field_off_host [F+1] (nullable):
// global row offset of each field; when given and B <= fmb_sort_fields_max_batch() the step uses
// the one-kernel per-field sort instead of the generic radix sort (same result).
FMB_API int fmb_session_create(fmb_session** out, int F, int k, int64_t max_batch, const int32_t* field_off_host) {
    FMB_CHECK_ARG(out && F > 0 && k > 0 && max_batch > 0, "fmb_session_create: bad arguments");
    FMB_CHECK_ARG(max_batch * F < ((int64_t)1 << 31), "fmb_session_create: max_batch*F must fit int32");
    fmb_session* s = new (std::nothrow) fmb_session();
    FMB_CHECK_ARG(s, "fmb_session_create: out of host memory");
    memset(s, 0, sizeof(*s));
    s->F = F; s->k = k; s->rowp = fmb_round_up(k + 1, 16); s->kp4 = fmb_round_up(k, 4); s->maxB = max_batch;
    const int64_t N = max_batch * F;
    fmb_runlist_shape((int)(max_batch < 65536 ? max_batch : 65536), F, &s->rl_nseg, &s->rl_cap);
    if ((int64_t)s->rl_nseg * s->rl_cap < N / 2 + 64) s->rl_cap = (int)((N / 2 + 64 + s->rl_nseg - 1) / s->rl_nseg);   // generic path: one segment of N/2
    s->sort_ws_bytes = fmb_sort_workspace_bytes(N);
    s->bwd_ws_bytes = fmb_bwd_workspace_bytes(N, k);
    cudaError_t e = cudaSuccess;
    auto dm = [&](void** p, size_t n) { if (e == cudaSuccess) e = cudaMalloc(p, n); };
    auto hm = [&](void** p, size_t n) { if (e == cudaSuccess) e = cudaMallocHost(p, n); };
    dm((void**)&s->d_ids, N * 4); dm((void**)&s->d_xv, N * 4); dm((void**)&s->d_y, max_batch * 4);
    dm((void**)&s->d_S, max_batch * s->kp4 * 4); dm((void**)&s->d_z, max_batch * 4);
    dm((void**)&s->d_delta, max_batch * 4); dm((void**)&s->d_lossv, max_batch * 4); dm((void**)&s->d_loss, 256);
    for (int i = 0; i < 2; ++i) { dm((void**)&s->d_skeys_buf[i], N * 4); dm((void**)&s->d_perm_buf[i], N * 4); dm((void**)&s->d_posflag_buf[i], N * 4); dm((void**)&s->d_runlist_buf[i], (size_t)s->rl_nseg * s->rl_cap * 16); dm((void**)&s->d_runcount_buf[i], (size_t)s->rl_nseg * 8 + 256); }
    if (!(field_off_host && max_batch <= fmb_sort_fields_max_batch())) dm(&s->d_sort_ws2, s->sort_ws_bytes);
    s->d_skeys = s->d_skeys_buf[0]; s->d_perm = s->d_perm_buf[0];
    dm(&s->d_sort_ws, s->sort_ws_bytes); dm(&s->d_bwd_ws, s->bwd_ws_bytes);
    hm((void**)&s->h_ids, N * 4); hm((void**)&s->h_xv, N * 4); hm((void**)&s->h_y, max_batch * 4);
    hm((void**)&s->h_loss, 256);
    dm((void**)&s->d_ids2, N * 4); dm((void**)&s->d_xv2, N * 4); dm((void**)&s->d_y2, max_batch * 4);
    dm((void**)&s->d_loss2, 256);
    hm((void**)&s->h_ids2, N * 4); hm((void**)&s->h_xv2, N * 4); hm((void**)&s->h_y2, max_batch * 4);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->st_copy, cudaStreamNonBlocking);
    for (int i = 0; i < 4; ++i) {
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_h2d[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_done[i], cudaEventDisableTiming);
    }
    if (field_off_host) {
        dm((void**)&s->d_field_off, (size_t)(F + 1) * 4);
        if (e == cudaSuccess) e = cudaMemcpy(s->d_field_off, field_off_host, (size_t)(F + 1) * 4, cudaMemcpyHostToDevice);
    }
    {
        // The sort of the NEXT batch is captured on the HIGH-priority stream, the step's own kernels on the low-priority
        // one (graphs are instantiated with cudaGraphInstantiateFlagUseNodePriority).  The fused kernel's 1 024 CTAs fill
        // every thread slot of the GPU; launched first they kept the sort's 156 clustered CTAs waiting until the first
        // tiles retired (~20 us: the step took sort + 20 us whatever the fused kernel cost).  With priority the sort's
        // CTAs are placed first (one per SM), the tiles take the remaining seven slots, and both chains start together.
        // FMB_PRIO=0: no priorities; FMB_PRIO=2: the other way round (for comparison).
        int least = 0, greatest = 0;
        const char* pe = getenv("FMB_PRIO");
        s->use_prio = pe ? atoi(pe) : 1;
        if (s->use_prio && cudaDeviceGetStreamPriorityRange(&least, &greatest) != cudaSuccess) s->use_prio = 0;
        if (!s->use_prio) least = greatest = 0;
        if (s->use_prio == 1) { const int t = least; least = greatest; greatest = t; }   // st0/st1 low, st2 high
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&s->st0, cudaStreamNonBlocking, greatest);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&s->st1, cudaStreamNonBlocking, greatest);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&s->st2, cudaStreamNonBlocking, least);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&s->st3, cudaStreamNonBlocking, least);
        if (e == cudaSuccess) e = cudaStreamCreateWithPriority(&s->st4, cudaStreamNonBlocking, greatest);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_join4, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_sp_fork, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_sp_join, cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_fork, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_fwd, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_sort, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_join, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_presort, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_join2, cudaEventDisableTiming);
    for (int i = 0; i < 2; ++i) if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_buf_free[i], cudaEventDisableTiming);
    {
        const char* ng = getenv("FMB_NO_GRAPH");
        s->use_graph = !(ng && ng[0] == '1');
        const char* sp = getenv("FMB_SPARSE");
        s->sparse_ok = !(sp && sp[0] == '0');
        const char* pd = getenv("FMB_PDL");
        s->use_pdl = !(pd && pd[0] == '0');
        const char* sa = getenv("FMB_SORT_AFTER");
        s->sort_after = sa && sa[0] == '1';
    }
    if (e != cudaSuccess) {
        fmb_set_error("fmb_session_create: %s", cudaGetErrorString(e));
        fmb_session_destroy(s);
        return FMB_ERR_CUDA;
    }
    *out = s;
    return FMB_OK;
}

// update mode 2 (FTRL-Proximal): the per-coordinate state the session's steps read and write.  zn_dev [R][2][rowp]
// (z and n sub-rows of every packed row), bias_zn_dev [2]; zero-initialised by the caller.  Step graphs captured
// before this call are dropped.
FMB_API int fmb_session_set_ftrl(fmb_session* s, float* zn_dev, float* bias_zn_dev, float beta, float l1, float l2) {
    FMB_CHECK_ARG(s && zn_dev && bias_zn_dev && l1 >= 0.f && l2 >= 0.f, "fmb_session_set_ftrl: bad arguments");
    s->ftrl.zn = zn_dev; s->ftrl.bias_zn = bias_zn_dev; s->ftrl.beta = beta; s->ftrl.l1 = l1; s->ftrl.l2 = l2;
    s->ftrl_set = 1;
    for (int i = 0; i < s->ngraphs; ++i) { cudaGraphExecDestroy(s->gvar[i].exec); cudaGraphDestroy(s->gvar[i].graph); }
    s->ngraphs = 0; s->next_evict = 0;
    return FMB_OK;
}

// update mode 3 (Adagrad): the sums the session's steps read and write.  sums_dev [R][rowp] (row r's sums at row r's
// offsets of the packed table), bias_sum_dev [1]; initialised by the caller (initial_accumulator_value).  Step graphs
// captured before this call are dropped.
FMB_API int fmb_session_set_adagrad(fmb_session* s, float* sums_dev, float* bias_sum_dev, float eps) {
    FMB_CHECK_ARG(s && sums_dev && bias_sum_dev && eps >= 0.f, "fmb_session_set_adagrad: bad arguments");
    s->ada.sums = sums_dev; s->ada.bias_sum = bias_sum_dev; s->ada.mlp_sums = nullptr; s->ada.eps = eps;
    s->ada_set = 1;
    for (int i = 0; i < s->ngraphs; ++i) { cudaGraphExecDestroy(s->gvar[i].exec); cudaGraphDestroy(s->gvar[i].graph); }
    s->ngraphs = 0; s->next_evict = 0;
    return FMB_OK;
}

FMB_API int64_t fmb_session_launches(const fmb_session* s) { return s ? s->launches : 0; }
FMB_API int fmb_session_graph_count(const fmb_session* s) { return s ? s->ngraphs : 0; }

static bool by_field_sort(const fmb_session* s, int B) { return s->d_field_off && B <= fmb_sort_fields_max_batch(); }

// stable sort of a batch's row ids + per-entry (sorted position | multi-hit flag) words into sorted buffer `buf`
static int sort_launch(fmb_session* s, const int32_t* ids, int B, int key_bits, int buf, void* radix_ws,
                       cudaStream_t st, int* nlaunch) {
    const int64_t N = (int64_t)B * s->F;
    int rc;
    fmb_runlist_t rl;
    rl.entries = s->d_runlist_buf[buf]; rl.seg_count = s->d_runcount_buf[buf];
    if (by_field_sort(s, B)) {   // posflag and the run list come out of the sort kernels themselves; sparse fields skip the sort
        fmb_runlist_shape(B, s->F, &rl.nseg, &rl.seg_cap);
        if (!s->sparse_ok) {
            *nlaunch += 1;
            return fmb_sort_fields_ex(ids, B, s->F, s->d_field_off, s->d_skeys_buf[buf], s->d_perm_buf[buf],
                                      s->d_posflag_buf[buf], &rl, 0, st);
        }
        // dense fields: radix kernel on `st`; sparse fields: hash kernel beside it on st3 (independent outputs).  The
        // sparse kernel only writes the position words of multi-hit entries: the others must read 0.
        cudaMemsetAsync(s->d_posflag_buf[buf], 0, (size_t)N * 4, st);
        cudaEventRecord(s->ev_sp_fork, st);
        cudaStreamWaitEvent(s->st3, s->ev_sp_fork, 0);
        rc = fmb_sort_fields_ex(ids, B, s->F, s->d_field_off, s->d_skeys_buf[buf], s->d_perm_buf[buf], s->d_posflag_buf[buf],
                                &rl, 1 | 2, st);
        if (rc) return rc;
        rc = fmb_sort_fields_ex(ids, B, s->F, s->d_field_off, s->d_skeys_buf[buf], s->d_perm_buf[buf], s->d_posflag_buf[buf],
                                &rl, 1 | 4, s->st3);
        cudaEventRecord(s->ev_sp_join, s->st3);
        cudaStreamWaitEvent(st, s->ev_sp_join, 0);
        *nlaunch += 2;
        return rc;
    } else {
        rc = fmb_sort_segment(ids, N, key_bits, radix_ws, s->sort_ws_bytes, s->d_skeys_buf[buf], s->d_perm_buf[buf],
                              nullptr, nullptr, st);
        *nlaunch += 3 * ((key_bits + 7) / 8);
    }
    if (rc) return rc;
    rl.nseg = 1; rl.seg_cap = (int)(N / 2 + 1);
    cudaMemsetAsync(s->d_runcount_buf[buf], 0, 8, st);
    rc = fmb_pos_flags_ex(s->d_skeys_buf[buf], s->d_perm_buf[buf], N, s->d_posflag_buf[buf], &rl, st);
    *nlaunch += 1;
    return rc;
}

// The kernels of one FM-only step (rows read once, see fm_step.cu):
//   main : [sort + position words of this batch, unless pre-sorted] -> fused forward/loss/single-hit updates
//          -> run kernel (multi-hit rows, sample order)
//   side : bias step + mean loss (needs delta/lossv only)            side2: sort of the NEXT batch (ids only)
static int fm_step_launch(fmb_session* s, const int32_t* ids, const float* xv, const float* y, int B, float* table,
                          float* bias, int key_bits, int loss_kind, float lr, int mode, float* loss_dev,
                          const int32_t* next_ids, cudaStream_t main, cudaStream_t side, cudaStream_t side2, int cur,
                          bool pre, int* nlaunch) {
    const int64_t N = (int64_t)B * s->F;
    int rc;
    *nlaunch = 0;
    cudaEventRecord(s->ev_fork, main);
    cudaStreamWaitEvent(side, s->ev_fork, 0);
    if (next_ids && !s->sort_after) {
        cudaStreamWaitEvent(side2, s->ev_fork, 0);
        rc = sort_launch(s, next_ids, B, key_bits, 1 - cur, s->d_sort_ws2, side2, nlaunch);
        if (rc) return rc;
        cudaEventRecord(s->ev_join2, side2);
    }
    if (!pre) {
        rc = sort_launch(s, ids, B, key_bits, cur, s->d_sort_ws, main, nlaunch);
        if (rc) return rc;
    }
    // the state slot of the step's kernels: the FTRL state, or in mode 3 the Adagrad state (include/fmb200.h)
    const fmb_ftrl_t* ft = mode == 3 ? (s->ada_set ? reinterpret_cast<const fmb_ftrl_t*>(&s->ada) : nullptr)
                                     : (s->ftrl_set ? &s->ftrl : nullptr);
    rc = fmb_fm_step_fused_ex(ids, xv, y, table, bias, s->d_posflag_buf[cur], B, s->F, s->k, loss_kind, lr, mode, ft,
                              s->d_delta, s->d_lossv, s->d_bwd_ws, s->bwd_ws_bytes, main);
    if (rc) return rc;
    cudaEventRecord(s->ev_fwd, main);
    cudaStreamWaitEvent(side, s->ev_fwd, 0);
    if (next_ids && s->sort_after) {
        // Experiment (FMB_SORT_AFTER=1): the sort of the NEXT batch starts when the fused kernel is done and runs beside
        // the run kernel and the bias step.  The fused kernel then takes 19 us instead of 26-33 (the sort's CTAs no longer
        // keep its 1 024 tiles from being resident at once), but the sort chain (~20 us) ends after the run kernel:
        // 51.8 us per step against 42.7 with the sort started at the top of the graph.
        cudaStreamWaitEvent(side2, s->ev_fwd, 0);
        rc = sort_launch(s, next_ids, B, key_bits, 1 - cur, s->d_sort_ws2, side2, nlaunch);
        if (rc) return rc;
        cudaEventRecord(s->ev_join2, side2);
    }
    rc = fmb_finish_step_ex(s->d_delta, s->d_lossv, B, bias, lr, mode, ft, loss_dev ? loss_dev : s->d_loss, side);
    if (rc) return rc;
    cudaEventRecord(s->ev_join, side);
    fmb_runlist_t rl;
    rl.entries = s->d_runlist_buf[cur]; rl.seg_count = s->d_runcount_buf[cur];
    if (by_field_sort(s, B)) fmb_runlist_shape(B, s->F, &rl.nseg, &rl.seg_cap);
    else { rl.nseg = 1; rl.seg_cap = (int)(N / 2 + 1); }
    fmb_runs_list_next_is_dependent(s->use_pdl);
    rc = fmb_fm_backward_runs_list(s->d_skeys_buf[cur], N, table, s->F, s->k, lr, mode, ft, &rl, s->d_bwd_ws, s->bwd_ws_bytes, main);
    if (rc) return rc;
    cudaStreamWaitEvent(main, s->ev_join, 0);
    if (next_ids) cudaStreamWaitEvent(main, s->ev_join2, 0);
    *nlaunch += 3;
    return FMB_OK;
}

// re-point one kernel node of an instantiated step graph at new per-batch pointers: argument i of the node is
// replaced by *repl[i] wherever repl[i] != NULL; the other arguments keep the values captured in `graph`.
static int patch_node(cudaGraphExec_t exec, cudaGraphNode_t node, int nparams, const void* const* repl) {
    cudaKernelNodeParams kp;
    CU(cudaGraphKernelNodeGetParams(node, &kp));
    void* args[16];
    for (int i = 0; i < nparams; ++i) args[i] = repl[i] ? const_cast<void*>(repl[i]) : kp.kernelParams[i];
    kp.kernelParams = args;
    kp.extra = nullptr;
    CU(cudaGraphExecKernelNodeSetParams(exec, node, &kp));
    return FMB_OK;
}

static int capture_variant(fmb_session* s, StepVariant* v, const int32_t* ids, const float* xv, const float* y,
                           float* table, float* bias, const int32_t* next_ids) {
    cudaGraph_t graph = nullptr;
    int nl = 0;
    CU(cudaStreamBeginCapture(s->st0, cudaStreamCaptureModeThreadLocal));
    const int rc = fm_step_launch(s, ids, xv, y, v->B, table, bias, v->key_bits, v->loss_kind, v->lr, v->mode, s->d_loss,
                                  next_ids, s->st0, s->st1, s->st2, v->cur, v->pre != 0, &nl);
    cudaError_t e = cudaStreamEndCapture(s->st0, &graph);
    if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) { fmb_set_error("graph capture: %s", cudaGetErrorString(e)); return FMB_ERR_CUDA; }
    // find the nodes that carry per-batch pointers
    cudaGraphNode_t nodes[64];
    size_t nn = 64;
    CU(cudaGraphGetNodes(graph, nodes, &nn));
    const void* sort_fns[8];
    int sort_np[8], sort_ska[8];
    const int nsort = fmb_sort_fields_kernel_fns(sort_fns, sort_np, sort_ska);
    v->n_fused = v->n_finish = nullptr;
    for (int j = 0; j < 2; ++j) v->n_sort_cur[j] = v->n_sort_next[j] = nullptr;
    for (size_t i = 0; i < nn; ++i) {
        cudaGraphNodeType ty;
        CU(cudaGraphNodeGetType(nodes[i], &ty));
        if (ty != cudaGraphNodeTypeKernel) continue;
        cudaKernelNodeParams kp;
        CU(cudaGraphKernelNodeGetParams(nodes[i], &kp));
        if (fmb_is_fused_kernel_fn(kp.func)) { v->n_fused = nodes[i]; continue; }
        if (kp.func == fmb_finish_kernel_fn()) { v->n_finish = nodes[i]; continue; }
        for (int t = 0; t < nsort; ++t)
            if (kp.func == sort_fns[t]) {
                const int32_t* out = *static_cast<int32_t**>(kp.kernelParams[sort_ska[t]]);   // sorted_keys argument
                const bool is_cur = out == s->d_skeys_buf[v->cur];
                cudaGraphNode_t* dst = is_cur ? v->n_sort_cur : v->n_sort_next;
                int* dnp = is_cur ? v->np_sort_cur : v->np_sort_next;
                const int j = dst[0] ? 1 : 0;
                dst[j] = nodes[i]; dnp[j] = sort_np[t];
            }
    }
    if (!v->n_fused || !v->n_finish || (!v->pre && !v->n_sort_cur[0]) || (v->has_next && !v->n_sort_next[0])) {
        cudaGraphDestroy(graph);
        fmb_set_error("step graph: kernel nodes not found");
        return FMB_ERR_CUDA;
    }
    cudaGraphExec_t exec = nullptr;
    e = cudaGraphInstantiate(&exec, graph, s->use_prio ? cudaGraphInstantiateFlagUseNodePriority : 0);
    if (e != cudaSuccess) { cudaGraphDestroy(graph); fmb_set_error("graph instantiate: %s", cudaGetErrorString(e)); return FMB_ERR_CUDA; }
    v->graph = graph; v->exec = exec; v->nlaunch = nl;
    return FMB_OK;
}

// One FM-only training step with DEVICE inputs (FMAdam.update_embedding/fit, and the update_embedding of the
// DeepFM/NFM/ONN classes whose loss is on forward_fm only).
//   loss_kind 0: BCEWithLogits(z_fm)   (fm_adam.py:66, deepfm_adam.py:101, deepfm_onn.py:166)
//   loss_kind 1: BCEWithLogits(sigmoid(z_fm))   (fm_adam.py:80, nfm_adam.py:100, nfm_onn.py:168)
//   loss_dev (nullable): receives the mean loss (device scalar).
//   next_ids (nullable): ids [B,F] of the batch the NEXT call will step on; their sort (it depends on the ids only)
//   rides along on a side branch of this step, and the next call -- recognised by its ids pointer -- skips its own.
// The step replays a CUDA graph captured once per configuration and re-pointed at this call's batch;
// FMB_NO_GRAPH=1 (and batches too large for the per-field sort) launch the kernels directly.
FMB_API int fmb_session_fm_step_next(fmb_session* s, const int32_t* ids, const float* xv, const float* y, int B,
                                     float* table, float* bias, int key_bits, int loss_kind, float lr, int mode,
                                     const int32_t* next_ids, float* loss_dev, cudaStream_t stream) {
    FMB_CHECK_ARG(s && ids && y && table && bias, "fmb_session_fm_step: null pointer");
    FMB_CHECK_ARG(B > 0 && B <= s->maxB, "fmb_session_fm_step: B=%d exceeds session max_batch", B);
    int nl = 0;
    // sorted form of this batch: already produced by a previous call (next_ids / fmb_session_presort), or sorted here
    const bool pre = s->presort_ids == ids && s->presort_B == B && !s->presort_stale;
    s->presort_stale = 0;
    const int cur = pre ? s->presort_buf : 1 - s->last_buf;
    if (pre) {
        if (s->presort_ext) CU(cudaStreamWaitEvent(stream, s->ev_presort, 0));
    } else {
        if (s->buf_used[cur]) CU(cudaStreamWaitEvent(stream, s->ev_buf_free[cur], 0));
        if (s->presort_ids && s->presort_ext) CU(cudaStreamWaitEvent(stream, s->ev_presort, 0));   // a pre-sort nobody used
    }
    s->presort_ids = nullptr;
    // the next batch is sorted into the other buffer, last read by the step before this one (already ordered: same stream)
    if (next_ids && s->buf_used[1 - cur]) CU(cudaStreamWaitEvent(stream, s->ev_buf_free[1 - cur], 0));
    s->last_buf = cur;
    int rc = FMB_OK;
    // the very first step runs eagerly: it sets the kernels' function attributes outside any capture
    if (!s->use_graph || s->steps_done == 0 || !by_field_sort(s, B)) {
        rc = fm_step_launch(s, ids, xv, y, B, table, bias, key_bits, loss_kind, lr, mode, loss_dev, next_ids, stream,
                            s->st1, s->st2, cur, pre, &nl);
        if (rc) return rc;
        s->launches += nl;
    } else {
        StepVariant key;
        memset(&key, 0, sizeof(key));
        key.B = B; key.key_bits = key_bits; key.loss_kind = loss_kind; key.mode = mode; key.has_xv = xv != nullptr;
        key.pre = pre; key.has_next = next_ids != nullptr; key.cur = cur; key.table = table; key.bias = bias; key.lr = lr;
        StepVariant* v = nullptr;
        const size_t keylen = offsetof(StepVariant, graph);
        // Several graphs may share a key: one per set of per-batch pointers, up to four (the host entry point's four
        // input slots replay their graphs without re-pointing a node); beyond that the first one is re-pointed.
        float* want_loss = loss_dev ? loss_dev : s->d_loss;
        int same_key = 0;
        for (int i = 0; i < s->ngraphs; ++i)
            if (memcmp(&s->gvar[i], &key, keylen) == 0) {
                ++same_key;
                if (!v) v = &s->gvar[i];
                if (s->gvar[i].cur_ids == ids && s->gvar[i].cur_y == y && s->gvar[i].cur_loss == want_loss) { v = &s->gvar[i]; same_key = 99; break; }
            }
        if (v && same_key < 4 && s->host_path) v = nullptr;     // host path: capture one more instead of re-pointing
        if (!v) {
            rc = capture_variant(s, &key, ids, xv, y, table, bias, next_ids);
            if (rc) return rc;
            int slot;
            if (s->ngraphs < FMB_GRAPH_CACHE) slot = s->ngraphs++;
            else {
                slot = s->next_evict; s->next_evict = (s->next_evict + 1) % FMB_GRAPH_CACHE;
                cudaGraphExecDestroy(s->gvar[slot].exec); cudaGraphDestroy(s->gvar[slot].graph);
            }
            s->gvar[slot] = key;
            v = &s->gvar[slot];
        }
        if (v->cur_ids != ids || v->cur_xv != xv || v->cur_y != y) {
            const void* repl[16] = {nullptr};
            repl[0] = &ids; repl[1] = &xv; repl[2] = &y;
            rc = patch_node(v->exec, v->n_fused, 5, repl);
            if (rc) return rc;
            v->cur_ids = ids; v->cur_xv = xv; v->cur_y = y;
        }
        if (!pre && v->cur_sort_ids != ids) {
            const void* repl[16] = {nullptr};
            repl[0] = &ids;
            for (int j = 0; j < 2 && v->n_sort_cur[j]; ++j) {
                rc = patch_node(v->exec, v->n_sort_cur[j], v->np_sort_cur[j], repl);
                if (rc) return rc;
            }
            v->cur_sort_ids = ids;
        }
        if (next_ids && v->cur_next_ids != next_ids) {
            const void* repl[16] = {nullptr};
            repl[0] = &next_ids;
            for (int j = 0; j < 2 && v->n_sort_next[j]; ++j) {
                rc = patch_node(v->exec, v->n_sort_next[j], v->np_sort_next[j], repl);
                if (rc) return rc;
            }
            v->cur_next_ids = next_ids;
        }
        {   // the bias-step kernel writes the mean loss straight to the caller's scalar (a 4-byte copy behind every graph
            // launch was a stream operation of its own: ~4 us of bubble per step)
            float* lo = loss_dev ? loss_dev : s->d_loss;
            if (v->cur_loss != lo) {
                const void* repl[16] = {nullptr};
                repl[6] = &lo;
                rc = patch_node(v->exec, v->n_finish, 9, repl);
                if (rc) return rc;
                v->cur_loss = lo;
            }
        }
        CU(cudaGraphLaunch(v->exec, stream));
        s->launches += v->nlaunch;
    }
    CU(cudaEventRecord(s->ev_buf_free[cur], stream));
    s->buf_used[cur] = 1;
    if (next_ids) {
        s->presort_ids = next_ids; s->presort_B = B; s->presort_buf = 1 - cur; s->presort_ext = 0;
        CU(cudaEventRecord(s->ev_buf_free[1 - cur], stream));
        s->buf_used[1 - cur] = 1;
    }
    s->steps_done += 1;
    return FMB_OK;
}

FMB_API int fmb_session_fm_step(fmb_session* s, const int32_t* ids, const float* xv, const float* y, int B,
                                float* table, float* bias, int key_bits, int loss_kind, float lr, int mode,
                                float* loss_dev, cudaStream_t stream) {
    return fmb_session_fm_step_next(s, ids, xv, y, B, table, bias, key_bits, loss_kind, lr, mode, nullptr, loss_dev, stream);
}

// Sort batch `ids` now, on the session's side stream, into the sorted buffer the running step is NOT using; the
// next fmb_session_fm_step called with the same `ids` pointer and B skips its own sort.  The sort depends on the
// ids only, so this overlaps the kernels of the step in flight.  `ready` (nullable) is an event the ids depend on
// (e.g. their H2D copy).  The ids must not change until that step has run.
static int presort_impl(fmb_session* s, const int32_t* ids, int B, int key_bits, cudaEvent_t ready) {
    const int buf = 1 - s->last_buf;
    if (s->buf_used[buf]) CU(cudaStreamWaitEvent(s->st2, s->ev_buf_free[buf], 0));
    if (ready) CU(cudaStreamWaitEvent(s->st2, ready, 0));
    int nl = 0;
    if (s->use_graph && s->presort_warm && by_field_sort(s, B)) {
        // memset + radix kernel + sparse-field kernel on two streams with their events: one graph launch instead of
        // nine stream operations (the host entry point is bound by the host's submission time)
        int g = -1;
        for (int i = 0; i < s->npsg; ++i)
            if (s->psg[i].ids == ids && s->psg[i].B == B && s->psg[i].key_bits == key_bits && s->psg[i].buf == buf) g = i;
        if (g < 0) {
            cudaGraph_t graph = nullptr;
            CU(cudaStreamBeginCapture(s->st2, cudaStreamCaptureModeThreadLocal));
            const int rc = sort_launch(s, ids, B, key_bits, buf, s->d_sort_ws2 ? s->d_sort_ws2 : s->d_sort_ws, s->st2, &nl);
            const cudaError_t e = cudaStreamEndCapture(s->st2, &graph);
            if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
            if (e != cudaSuccess) { fmb_set_error("pre-sort graph capture: %s", cudaGetErrorString(e)); return FMB_ERR_CUDA; }
            cudaGraphExec_t exec = nullptr;
            if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) { cudaGraphDestroy(graph); fmb_set_error("pre-sort graph instantiate failed"); return FMB_ERR_CUDA; }
            g = s->npsg < 8 ? s->npsg++ : 0;
            if (s->psg[g].exec) { cudaGraphExecDestroy(s->psg[g].exec); cudaGraphDestroy(s->psg[g].graph); }
            s->psg[g].ids = ids; s->psg[g].B = B; s->psg[g].key_bits = key_bits; s->psg[g].buf = buf; s->psg[g].nl = nl;
            s->psg[g].exec = exec; s->psg[g].graph = graph;
        }
        nl = s->psg[g].nl;
        CU(cudaGraphLaunch(s->psg[g].exec, s->st2));
    } else {
        const int rc = sort_launch(s, ids, B, key_bits, buf, s->d_sort_ws2 ? s->d_sort_ws2 : s->d_sort_ws, s->st2, &nl);
        if (rc) return rc;
        s->presort_warm = 1;
    }
    CU(cudaEventRecord(s->ev_presort, s->st2));
    s->launches += nl;
    s->presort_ids = ids; s->presort_B = B; s->presort_buf = buf; s->presort_ext = 1;
    return FMB_OK;
}

FMB_API int fmb_session_presort(fmb_session* s, const int32_t* ids, int B, int key_bits) {
    FMB_CHECK_ARG(s && ids && B > 0 && B <= s->maxB, "fmb_session_presort: bad arguments");
    return presort_impl(s, ids, B, key_bits, nullptr);
}

// Forget any pre-sorted batch: the next step sorts its own ids.  Callers that cannot guarantee that the buffer
// behind a pre-sorted ids pointer still holds the same batch (freed and re-allocated tensors) call this.
FMB_API void fmb_session_presort_invalidate(fmb_session* s) {
    if (!s || !s->presort_ids) return;
    s->presort_stale = 1;
}

// true when `p` is page-locked host memory the copy engine can read directly (no staging copy needed)
static bool host_ptr_is_pinned(const void* p) {
    // the answer for the last few pointers is remembered (a training loop passes the same pinned buffers again and again;
    // cudaPointerGetAttributes is a driver call)
    static thread_local const void* seen[16];
    static thread_local bool pinned[16];
    static thread_local int nseen = 0, nextw = 0;
    for (int i = 0; i < nseen; ++i) if (seen[i] == p) return pinned[i];
    cudaPointerAttributes a;
    bool r = false;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) cudaGetLastError();
    else r = a.type == cudaMemoryTypeHost;
    seen[nextw] = p; pinned[nextw] = r; nextw = (nextw + 1) % 16; if (nseen < 16) ++nseen;
    return r;
}
// Pipelined step with HOST inputs.  `slot` (0..3) selects one of four device input buffers: the copies of
// step t+1 (on the session's copy stream) overlap the kernels of step t (on `stream`); a caller that cycles through all four
// slots and collects a step's loss three steps later never waits for the GPU while it submits (fmb_session_host_slots()).  Pinned / registered
// host buffers are read in place, pageable ones go through the session's pinned staging area.  The loss
// arrives in pinned memory; fmb_session_wait_loss(slot) waits for it.  Every step still moves its own
// 4*B*F (+4*B*F) + 4*B bytes in and 4 bytes out.
FMB_API int fmb_session_fm_step_host_async(fmb_session* s, int slot, const int32_t* ids_host, const float* xv_host,
                                           const float* y_host, int B, float* table, float* bias, int key_bits,
                                           int loss_kind, float lr, int mode, cudaStream_t stream) {
    FMB_CHECK_ARG(s && ids_host && y_host && table && bias, "fmb_session_fm_step_host_async: null pointer");
    FMB_CHECK_ARG(slot >= 0 && slot < 4, "fmb_session_fm_step_host_async: slot must be 0..3");
    FMB_CHECK_ARG(B > 0 && B <= s->maxB, "fmb_session_fm_step_host_async: B=%d exceeds session max_batch", B);
    const size_t N = (size_t)B * s->F;
    if (slot >= 2 && !s->d_idsx[slot - 2]) {     // slots 2 and 3: buffers on first use
        const size_t NN = (size_t)s->maxB * s->F;
        const int j = slot - 2;
        cudaError_t e = cudaMalloc((void**)&s->d_idsx[j], NN * 4);
        if (e == cudaSuccess) e = cudaMalloc((void**)&s->d_xvx[j], NN * 4);
        if (e == cudaSuccess) e = cudaMalloc((void**)&s->d_yx[j], (size_t)s->maxB * 4);
        if (e == cudaSuccess) e = cudaMallocHost((void**)&s->h_idsx[j], NN * 4);
        if (e == cudaSuccess) e = cudaMallocHost((void**)&s->h_xvx[j], NN * 4);
        if (e == cudaSuccess) e = cudaMallocHost((void**)&s->h_yx[j], (size_t)s->maxB * 4);
        if (e != cudaSuccess) { fmb_set_error("fmb_session_fm_step_host_async: %s", cudaGetErrorString(e)); return FMB_ERR_CUDA; }
    }
    int32_t* d_ids = slot >= 2 ? s->d_idsx[slot - 2] : (slot ? s->d_ids2 : s->d_ids);
    float* d_xv = slot >= 2 ? s->d_xvx[slot - 2] : (slot ? s->d_xv2 : s->d_xv);
    float* d_y = slot >= 2 ? s->d_yx[slot - 2] : (slot ? s->d_y2 : s->d_y);
    float* d_loss = slot ? s->d_loss2 : s->d_loss;
    int32_t* h_ids = slot >= 2 ? s->h_idsx[slot - 2] : (slot ? s->h_ids2 : s->h_ids);
    float* h_xv = slot >= 2 ? s->h_xvx[slot - 2] : (slot ? s->h_xv2 : s->h_xv);
    float* h_y = slot >= 2 ? s->h_yx[slot - 2] : (slot ? s->h_y2 : s->h_y);
    // the previous user of this slot (two steps ago) must be done with the device buffers and the staging area
    if (s->slot_used[slot]) CU(cudaEventSynchronize(s->ev_done[slot]));
    const void* src_ids = ids_host;
    const void* src_y = y_host;
    const void* src_xv = xv_host;
    if (!host_ptr_is_pinned(ids_host)) { memcpy(h_ids, ids_host, N * 4); src_ids = h_ids; }
    if (!host_ptr_is_pinned(y_host)) { memcpy(h_y, y_host, (size_t)B * 4); src_y = h_y; }
    if (xv_host && !host_ptr_is_pinned(xv_host)) { memcpy(h_xv, xv_host, N * 4); src_xv = h_xv; }
    CU(cudaMemcpyAsync(d_ids, src_ids, N * 4, cudaMemcpyHostToDevice, s->st_copy));
    CU(cudaMemcpyAsync(d_y, src_y, (size_t)B * 4, cudaMemcpyHostToDevice, s->st_copy));
    if (xv_host) CU(cudaMemcpyAsync(d_xv, src_xv, N * 4, cudaMemcpyHostToDevice, s->st_copy));
    CU(cudaEventRecord(s->ev_h2d[slot], s->st_copy));
    CU(cudaStreamWaitEvent(stream, s->ev_h2d[slot], 0));
    // the sort of this batch starts as soon as its ids have landed: it overlaps the step still in flight
    int rc = presort_impl(s, d_ids, B, key_bits, s->ev_h2d[slot]);
    if (rc) return rc;
    // the bias-step kernel writes the mean loss straight into the pinned result word (4 bytes over PCIe: the D2H of the
    // step, without a copy operation of its own)
    (void)d_loss;
    s->host_path = 1;
    rc = fmb_session_fm_step(s, d_ids, xv_host ? d_xv : nullptr, d_y, B, table, bias, key_bits, loss_kind, lr,
                                 mode, s->h_loss + 8 * slot, stream);
    s->host_path = 0;
    if (rc) return rc;
    CU(cudaEventRecord(s->ev_done[slot], stream));
    s->slot_used[slot] = 1;
    return FMB_OK;
}

// number of input slots of fmb_session_fm_step_host_async
FMB_API int fmb_session_host_slots(void) { return 4; }

// waits for the step last submitted on `slot` and returns its mean loss
FMB_API int fmb_session_wait_loss(fmb_session* s, int slot, float* loss_host) {
    FMB_CHECK_ARG(s && slot >= 0 && slot < 4 && s->slot_used[slot], "fmb_session_wait_loss: nothing submitted on slot %d", slot);
    CU(cudaEventSynchronize(s->ev_done[slot]));
    if (loss_host) *loss_host = s->h_loss[8 * slot];
    return FMB_OK;
}

// Same step with HOST inputs: copies ids/xv/y in (xv_host NULL = all ones, nothing copied), runs
// the step, copies the loss back and waits for it.  Bytes moved per step: H2D 4*B*F (+4*B*F) + 4*B,
// D2H 4.
FMB_API int fmb_session_fm_step_host(fmb_session* s, const int32_t* ids_host, const float* xv_host,
                                     const float* y_host, int B, float* table, float* bias, int key_bits,
                                     int loss_kind, float lr, int mode, float* loss_host, cudaStream_t stream) {
    FMB_CHECK_ARG(s && ids_host && y_host && table && bias, "fmb_session_fm_step_host: null pointer");
    FMB_CHECK_ARG(B > 0 && B <= s->maxB, "fmb_session_fm_step_host: B=%d exceeds session max_batch", B);
    const size_t N = (size_t)B * s->F;
    memcpy(s->h_ids, ids_host, N * 4);
    memcpy(s->h_y, y_host, (size_t)B * 4);
    CU(cudaMemcpyAsync(s->d_ids, s->h_ids, N * 4, cudaMemcpyHostToDevice, stream));
    CU(cudaMemcpyAsync(s->d_y, s->h_y, (size_t)B * 4, cudaMemcpyHostToDevice, stream));
    if (xv_host) {
        memcpy(s->h_xv, xv_host, N * 4);
        CU(cudaMemcpyAsync(s->d_xv, s->h_xv, N * 4, cudaMemcpyHostToDevice, stream));
    }
    int rc = fmb_session_fm_step(s, s->d_ids, xv_host ? s->d_xv : nullptr, s->d_y, B, table, bias, key_bits,
                                 loss_kind, lr, mode, s->d_loss, stream);
    if (rc) return rc;
    CU(cudaMemcpyAsync(s->h_loss, s->d_loss, 4, cudaMemcpyDeviceToHost, stream));
    CU(cudaStreamSynchronize(stream));
    if (loss_host) *loss_host = s->h_loss[0];
    return FMB_OK;
}
