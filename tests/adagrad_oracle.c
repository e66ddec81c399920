/*
 * adagrad_oracle.c -- CPU oracle of update mode 3 (torch.optim.Adagrad), TEST INFRASTRUCTURE ONLY.
 *
 * The deep-family oracle (oracle/fm_oracle.c) is compiled into this translation unit unchanged, so the forward pass, the
 * loss, the tower's backward and the per-row gradient sums (bwd_entry: sample order) are the very code the other modes are
 * checked with; this file adds only what Adagrad changes: the update of every parameter that has a gradient, with a
 * persistent sum per coordinate.  tests/adagrad_ref.py builds it and drives it next to oracle.deep.OracleDeep.
 *
 * Update rule, as torch 2.11's CPU _single_tensor_adagrad rounds it (lr_decay = 0, weight_decay = 0; pinned on
 * torch.optim.Adagrad in tests/test_adagrad.py; the CUDA side is fmb::adagrad_update in csrc/fmb_common.cuh):
 *   state_sum.addcmul_(grad, grad, value=1)      s' = fma(g, g, s)
 *   std = state_sum.sqrt().add_(eps)             std = sqrt_mkl(s') + eps      (Tensor.sqrt is MKL's vsSqrt)
 *   param.addcdiv_(grad, std, value=-lr)         p' = p + ((-lr * g) / std)
 *
 * Build: gcc -O2 -fPIC -shared -std=c11 -ffp-contract=off -fno-fast-math -I oracle (tests/adagrad_ref.py).
 */
#include "fm_oracle.c"

API float orc_adagrad_update(float p, float g, float* s, float lr, float eps) {
    const float ss = fmaf(g, g, *s);
    *s = ss;
    const float sd = orc_sqrt_mkl(ss) + eps;
    return p + ((-lr * g) / sd);
}
API void orc_vec_adagrad(float* p, const float* g, float* s, int64_t n, float lr, float eps) {
    for (int64_t i = 0; i < n; ++i) p[i] = orc_adagrad_update(p[i], g[i], s + i, lr, eps);
}

/* the sums of every parameter, caller-owned (initial_accumulator_value) */
typedef struct {
    float* sV;    /* [R*k] */
    float* sw1;   /* [R]   */
    float* sbias; /* [1]   */
    float* smlp;  /* [orc_mlp_numel] or NULL */
    float eps;
} orc_ada;

/* embedding_dense_backward (rows summed in sample order: bwd_entry), then one Adagrad step per row hit */
static void ada_backward_update(orc_model* m, const orc_ada* a, const int32_t* ids, const float* xv, int B, const float* S,
                                const float* gs, int use_fm2, const float* gvec) {
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
            v[j] = orc_adagrad_update(v[j], g, a->sV + (size_t)r * k + j, m->lr, a->eps);
            ga[j] = 0.f; gb[j] = 0.f;
        }
        m->w1[r] = orc_adagrad_update(m->w1[r], ga[k], a->sw1 + r, m->lr, a->eps);
        ga[k] = 0.f;
        m->touched[r] = 0;
    }
    free(tl);
}

/* update_embedding (orc_update_embedding with mode 3): loss on forward_fm, the tower has no gradient and is skipped */
API float orc_ada_update_embedding(orc_model* m, const orc_ada* a, const int32_t* ids, const float* xv, const float* y, int B) {
    fwd_buf w; fb_alloc(m, B, &w);
    orc_fm_forward(m, ids, xv, B, NULL, w.S, w.bi, w.sf, w.sb, w.zfm);
    float* delta = (float*)malloc(sizeof(float) * B);
    const int kind = is_nfm(m) ? 1 : 0;
    const float loss = orc_loss_delta(kind, w.zfm, y, B, delta);
    const float gbias = orc_sum_aten(delta, B);
    ada_backward_update(m, a, ids, xv, B, w.S, delta, 1, NULL);
    m->bias[0] = orc_adagrad_update(m->bias[0], gbias, a->sbias, m->lr, a->eps);
    free(delta); fb_free(&w);
    return loss;
}

/* fit (orc_fit with mode 3) of FMAdam / DeepFMAdam / NFMAdam; the ONN classes' hedge fit uses no optimizer */
API void orc_ada_fit(orc_model* m, const orc_ada* a, const int32_t* ids, const float* xv, const float* y, int B) {
    if (is_onn(m)) { orc_fit(m, ids, xv, y, B); return; }
    fwd_buf w; fb_alloc(m, B, &w);
    float* z = (float*)malloc(sizeof(float) * B);
    float* delta = (float*)malloc(sizeof(float) * B);
    full_forward(m, ids, xv, B, &w, z, NULL);
    const int kind = (m->kind == K_NFM) ? 0 : 1;
    (void)orc_loss_delta(kind, z, y, B, delta);
    const float gbias = orc_sum_aten(delta, B);
    if (m->kind == K_FM) {
        ada_backward_update(m, a, ids, xv, B, w.S, delta, 1, NULL);
    } else {
        const int64_t n = orc_mlp_numel(m);
        float* gmlp = (float*)malloc(sizeof(float) * n);
        float* gbi = (float*)malloc(sizeof(float) * (size_t)B * m->k);
        orc_mlp_backward(m, w.bi, w.act, delta, m->L - 1, B, gmlp, gbi);
        ada_backward_update(m, a, ids, xv, B, w.S, delta, m->kind == K_DEEPFM, gbi);
        orc_vec_adagrad(m->mlp, gmlp, a->smlp, n, m->lr, a->eps);
        free(gmlp); free(gbi);
    }
    m->bias[0] = orc_adagrad_update(m->bias[0], gbias, a->sbias, m->lr, a->eps);
    free(z); free(delta); fb_free(&w);
}

/* run_experiment (orc_run_experiment with mode 3): predict, then fit with batch size 1, example by example */
API void orc_ada_run_experiment(orc_model* m, const orc_ada* a, const int32_t* ids, const float* xv, const float* y, int N,
                                int64_t* conf, uint8_t* preds) {
    conf[0] = conf[1] = conf[2] = conf[3] = 0;
    for (int i = 0; i < N; ++i) {
        uint8_t p;
        orc_predict(m, ids + (size_t)i * m->F, xv + (size_t)i * m->F, 1, &p);
        orc_ada_fit(m, a, ids + (size_t)i * m->F, xv + (size_t)i * m->F, y + i, 1);
        const int yi = y[i] == 1.0f;
        if ((int)p == yi) { if (yi) conf[0]++; else conf[2]++; }
        else { if (yi) conf[3]++; else conf[1]++; }
        if (preds) preds[i] = p;
    }
}
