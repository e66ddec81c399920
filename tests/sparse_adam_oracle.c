/*
 * sparse_adam_oracle.c -- CPU oracle of update mode 4 (torch.optim.SparseAdam on the embedding tables, torch.optim.Adam
 * on the bias and the tower, both kept across calls), TEST INFRASTRUCTURE ONLY.
 *
 * The deep-family oracle (oracle/fm_oracle.c) is compiled into this translation unit unchanged, so the forward pass, the
 * loss, the tower's backward and the per-row gradient sums (bwd_entry: sample order) are the very code the other modes are
 * checked with; this file adds only what mode 4 changes: the update of every parameter, with two moments per coordinate.
 * tests/sparse_adam_ref.py builds it and drives it next to oracle.deep.OracleDeep.
 *
 * Per-step scalars, in C double as CPython computes them, then rounded to float as ATen rounds a Python scalar:
 *   SparseAdam  step_size = lr * sqrt(1 - b2^t) / (1 - b1^t)       -> (float)(-step_size)
 *   Adam        step_size = lr / (1 - b1^t);  bc2s = (1 - b2^t)^0.5 -> (float)(-step_size), (float)bc2s
 * Update rules, as torch 2.11's CPU kernels round them (pinned on torch in tests/test_sparse_adam.py; the CUDA side is
 * fmb::sparse_adam_update / fmb::adam_update in csrc/fmb_common.cuh):
 *   SparseAdam (optim/_functional.py sparse_adam)     Adam (optim/adam.py _single_tensor_adam)
 *   u1 = (g - m) * (1-b1);  m' = m + u1                m' = fma(1-b1, g - m, m)               (lerp_)
 *   u2 = (g*g - v) * (1-b2);  v' = v + u2              v' = fma((1-b2) * g, g, v * b2)        (mul_, addcmul_)
 *   p' = p + s * ((u1 + m) / (sqrt(u2 + v) + eps))     p' = p + (s * m') / (sqrt(v') / bc2s + eps)   (addcdiv_)
 * with sqrt = MKL's vsSqrt (orc_sqrt_mkl).
 *
 * Build: gcc -O2 -fPIC -shared -std=c11 -ffp-contract=off -fno-fast-math -I oracle (tests/sparse_adam_ref.py).
 */
#include "fm_oracle.c"

/* the float scalars of step t: [0] SparseAdam's -step_size, [1] Adam's -step_size, [2] Adam's sqrt(bias_correction2) */
API void orc_adam_scalars(double lr, double beta1, double beta2, int64_t t, float* out) {
    const double bc1 = 1.0 - pow(beta1, (double)t);
    const double bc2 = 1.0 - pow(beta2, (double)t);
    out[0] = (float)(-(lr * sqrt(bc2) / bc1));
    out[1] = (float)(-(lr / bc1));
    out[2] = (float)pow(bc2, 0.5);
}

API float orc_sparse_adam_update(float p, float g, float* m, float* v, float b1c, float b2c, float eps, float step) {
    const float mo = *m, vo = *v;
    const float u1 = (g - mo) * b1c;
    const float u2 = (g * g - vo) * b2c;
    *m = mo + u1;
    *v = vo + u2;
    const float denom = orc_sqrt_mkl(u2 + vo) + eps;
    return p + step * ((u1 + mo) / denom);
}

API float orc_adam_update(float p, float g, float* m, float* v, float b1c, float b2f, float b2c, float eps, float step,
                          float bc2s) {
    const float m1 = fmaf(b1c, g - *m, *m);
    const float v1 = fmaf(b2c * g, g, *v * b2f);
    *m = m1;
    *v = v1;
    const float denom = orc_sqrt_mkl(v1) / bc2s + eps;
    return p + (step * m1) / denom;
}

/* both moments of every parameter (caller-owned, zero at the start) and both step counters */
typedef struct {
    float *mV, *vV;       /* [R*k] */
    float *mw1, *vw1;     /* [R]   */
    float *mbias, *vbias; /* [1]   */
    float *mmlp, *vmlp;   /* [orc_mlp_numel] or NULL */
    double beta1, beta2;
    float eps;
    int64_t step;         /* steps of the tables and the bias */
    int64_t mlp_step;     /* steps of the tower (fit only) */
} orc_sa;

typedef struct { float b1c, b2f, b2c, eps, emb, step, bc2s; } sa_scal;

static sa_scal sa_scalars(const orc_model* m, const orc_sa* a, int64_t t) {
    float s[3];
    orc_adam_scalars((double)m->lr, a->beta1, a->beta2, t, s);
    sa_scal r = {(float)(1.0 - a->beta1), (float)a->beta2, (float)(1.0 - a->beta2), a->eps, s[0], s[1], s[2]};
    return r;
}

API void orc_vec_adam(float* p, const float* g, float* mm, float* vv, int64_t n, float b1c, float b2f, float b2c, float eps,
                      float step, float bc2s) {
    for (int64_t i = 0; i < n; ++i) p[i] = orc_adam_update(p[i], g[i], mm + i, vv + i, b1c, b2f, b2c, eps, step, bc2s);
}

/* embedding_dense_backward (rows summed in sample order: bwd_entry), then one SparseAdam step per row hit -- a zero
 * gradient too: the moments decay and the weight moves by m' */
static void sa_backward_update(orc_model* m, const orc_sa* a, const sa_scal* sc, const int32_t* ids, const float* xv, int B,
                               const float* S, const float* gs, int use_fm2, const float* gvec) {
    const int F = m->F, k = m->k, kp = k + 1;
    int32_t* tl = (int32_t*)malloc(sizeof(int32_t) * (size_t)B * F);
    bwd_ctx c = {m, ids, xv, B, S, gs, use_fm2, gvec, tl, NULL, 0, NULL, NULL};
    size_t nt = 0;
    for (int b = 0; b < B; ++b)
        for (int f = 0; f < F; ++f) bwd_entry(&c, b, f, tl, &nt);
    for (size_t t = 0; t < nt; ++t) {
        const int32_t r = tl[t];
        float* v = m->V + (size_t)r * k;
        float* ga = m->gA + (size_t)r * kp;
        float* gb = m->gB + (size_t)r * kp;
        for (int j = 0; j < k; ++j) {
            const float g = (use_fm2 && gvec) ? ga[j] + gb[j] : (gvec ? gb[j] : ga[j]);
            const size_t o = (size_t)r * k + j;
            v[j] = orc_sparse_adam_update(v[j], g, a->mV + o, a->vV + o, sc->b1c, sc->b2c, sc->eps, sc->emb);
            ga[j] = 0.f; gb[j] = 0.f;
        }
        m->w1[r] = orc_sparse_adam_update(m->w1[r], ga[k], a->mw1 + r, a->vw1 + r, sc->b1c, sc->b2c, sc->eps, sc->emb);
        ga[k] = 0.f;
        m->touched[r] = 0;
    }
    free(tl);
}

static void sa_bias(orc_model* m, const orc_sa* a, const sa_scal* sc, float gbias) {
    m->bias[0] = orc_adam_update(m->bias[0], gbias, a->mbias, a->vbias, sc->b1c, sc->b2f, sc->b2c, sc->eps, sc->step, sc->bc2s);
}

/* update_embedding (orc_update_embedding with mode 4): the tower has no gradient, so neither it nor its counter moves */
API float orc_sa_update_embedding(orc_model* m, orc_sa* a, const int32_t* ids, const float* xv, const float* y, int B) {
    const sa_scal sc = sa_scalars(m, a, ++a->step);
    fwd_buf w; fb_alloc(m, B, &w);
    orc_fm_forward(m, ids, xv, B, NULL, w.S, w.bi, w.sf, w.sb, w.zfm);
    float* delta = (float*)malloc(sizeof(float) * B);
    const int kind = is_nfm(m) ? 1 : 0;
    const float loss = orc_loss_delta(kind, w.zfm, y, B, delta);
    const float gbias = orc_sum_aten(delta, B);
    sa_backward_update(m, a, &sc, ids, xv, B, w.S, delta, 1, NULL);
    sa_bias(m, a, &sc, gbias);
    free(delta); fb_free(&w);
    return loss;
}

/* fit (orc_fit with mode 4) of FMAdam / DeepFMAdam / NFMAdam; the ONN classes' hedge fit uses no optimizer */
API void orc_sa_fit(orc_model* m, orc_sa* a, const int32_t* ids, const float* xv, const float* y, int B) {
    if (is_onn(m)) { orc_fit(m, ids, xv, y, B); return; }
    const sa_scal sc = sa_scalars(m, a, ++a->step);
    fwd_buf w; fb_alloc(m, B, &w);
    float* z = (float*)malloc(sizeof(float) * B);
    float* delta = (float*)malloc(sizeof(float) * B);
    full_forward(m, ids, xv, B, &w, z, NULL);
    const int kind = (m->kind == K_NFM) ? 0 : 1;
    (void)orc_loss_delta(kind, z, y, B, delta);
    const float gbias = orc_sum_aten(delta, B);
    if (m->kind == K_FM) {
        sa_backward_update(m, a, &sc, ids, xv, B, w.S, delta, 1, NULL);
    } else {
        const sa_scal sm = sa_scalars(m, a, ++a->mlp_step);
        const int64_t n = orc_mlp_numel(m);
        float* gmlp = (float*)malloc(sizeof(float) * n);
        float* gbi = (float*)malloc(sizeof(float) * (size_t)B * m->k);
        orc_mlp_backward(m, w.bi, w.act, delta, m->L - 1, B, gmlp, gbi);
        sa_backward_update(m, a, &sc, ids, xv, B, w.S, delta, m->kind == K_DEEPFM, gbi);
        orc_vec_adam(m->mlp, gmlp, a->mmlp, a->vmlp, n, sm.b1c, sm.b2f, sm.b2c, sm.eps, sm.step, sm.bc2s);
        free(gmlp); free(gbi);
    }
    sa_bias(m, a, &sc, gbias);
    free(z); free(delta); fb_free(&w);
}

/* run_experiment (orc_run_experiment with mode 4): predict, then fit with batch size 1, example by example */
API void orc_sa_run_experiment(orc_model* m, orc_sa* a, const int32_t* ids, const float* xv, const float* y, int N,
                               int64_t* conf, uint8_t* preds) {
    conf[0] = conf[1] = conf[2] = conf[3] = 0;
    for (int i = 0; i < N; ++i) {
        uint8_t p;
        orc_predict(m, ids + (size_t)i * m->F, xv + (size_t)i * m->F, 1, &p);
        orc_sa_fit(m, a, ids + (size_t)i * m->F, xv + (size_t)i * m->F, y + i, 1);
        const int yi = y[i] == 1.0f;
        if ((int)p == yi) { if (yi) conf[0]++; else conf[2]++; }
        else { if (yi) conf[3]++; else conf[1]++; }
        if (preds) preds[i] = p;
    }
}
