// common.cu -- error plumbing and library identity for libfmb200.so
#include "fmb_common.cuh"
#include <cmath>
#include <cstdarg>
#include <cstdio>

static thread_local char g_err[512] = "";

void fmb_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

FMB_API const char* fmb_last_error(void) { return g_err; }
FMB_API int fmb_version(void) { return 100; }
// row pitch of the packed table in floats: rows are 64-byte aligned (HBM bursts are 64 B; a 48-byte row
// at a 48-byte pitch straddles two bursts 3 times out of 4 -- measured 35 MB of DRAM reads for 15 MB of rows)
FMB_API int fmb_rowp(int k) { return fmb_round_up(k + 1, 16); }
FMB_API int fmb_kp4(int k) { return fmb_round_up(k, 4); }

// number of visible CUDA devices (0 when there is no GPU / no driver): lets the Python side fail
// loudly instead of falling back to anything.
FMB_API int fmb_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// Update mode 4's float scalars of step t, in C double exactly as CPython evaluates torch's expressions (glibc pow and
// sqrt, the same operation order), then rounded to float as ATen rounds a Python scalar before it multiplies:
//   out[0] = SparseAdam's -step_size = -(lr * math.sqrt(1 - b2**t) / (1 - b1**t))
//   out[1] = Adam's -step_size = -(lr / (1 - b1**t));  out[2] = Adam's bias_correction2 ** 0.5
// CUDA's double pow is not correctly rounded, so the device never computes these.
FMB_API void fmb_adam_scalars(float lr, double beta1, double beta2, int64_t t, float* out) {
    const double bc1 = 1.0 - pow(beta1, (double)t);
    const double bc2 = 1.0 - pow(beta2, (double)t);
    out[0] = (float)(-((double)lr * sqrt(bc2) / bc1));
    out[1] = (float)(-((double)lr / bc1));
    out[2] = (float)pow(bc2, 0.5);
}

// One more step of update mode 4: the tables and the bias count every step, the tower (tower != 0) only the steps that
// give it a gradient (torch skips a parameter whose .grad is None).  Fills a->cur with the scalars of that step.
FMB_API int fmb_sparse_adam_advance(fmb_sparse_adam_t* a, float lr, int tower) {
    FMB_CHECK_ARG(a, "fmb_sparse_adam_advance: null state");
    float s[3];
    fmb_adam_scalars(lr, a->beta1, a->beta2, ++a->step, s);
    a->cur.emb_step = s[0]; a->cur.bias_step = s[1]; a->cur.bias_bc2s = s[2];
    if (tower) {
        fmb_adam_scalars(lr, a->beta1, a->beta2, ++a->mlp_step, s);
        a->cur.mlp_step = s[1]; a->cur.mlp_bc2s = s[2];
    }
    return FMB_OK;
}

// The scalars of N single-example fit steps of fmb_online_deep_run_ex (kinds 0-2), advancing the counters by N:
// out [4 + 5N] = (1-b1, b2, 1-b2, eps) as floats, then one fmb_adam_step_t per example.  tower: the model has one.
FMB_API int fmb_sparse_adam_online_steps(fmb_sparse_adam_t* a, float lr, int tower, int N, float* out) {
    FMB_CHECK_ARG(a && out && N > 0, "fmb_sparse_adam_online_steps: bad arguments");
    out[0] = (float)(1.0 - a->beta1); out[1] = (float)a->beta2; out[2] = (float)(1.0 - a->beta2); out[3] = a->eps;
    for (int n = 0; n < N; ++n) {
        fmb_sparse_adam_advance(a, lr, tower);
        float* r = out + 4 + (size_t)5 * n;
        r[0] = a->cur.emb_step; r[1] = a->cur.bias_step; r[2] = a->cur.bias_bc2s; r[3] = a->cur.mlp_step; r[4] = a->cur.mlp_bc2s;
    }
    return FMB_OK;
}
