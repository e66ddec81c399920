"""The DeepFM / NFM towers at every shape and batch-size sequence their kernels take.

1. The SIMT tower (mlp.cu's 64 x 64 x 16 gemm_kernel, head_sum_kernel, heads.cu) and the per-example kernel (online.cu)
   bit for bit against the C oracle after every step, across the tile edges in B, H and k, H >= 512 (ATen's summation
   cascade in the head sums), the largest tower online.cu's 200 KB shared-memory rule accepts, and one tower above the
   2^24 tensor-core threshold with the tensor cores switched off.  Every tower is scaled so that its top layer is neither
   dead nor all-positive, and every shape is asserted to sit on the intended side of the threshold.
2. The tcgen05 path (gemm_tc.cu) against float64, element by element: |C - C64| <= tau * (|A| |B|)_ij + FLOOR, with tau
   calibrated on the B200 and shown (CPU test) to be tight enough to see one dropped K-slice, an omitted bias, a flipped
   relu-mask entry and a column sum missing one split.
3. The fit graphs deep.py captures, replayed after a larger batch has grown the model's workspaces or the process-wide
   split-K workspace.

CPU tests (no mark): every case's premises, the 200 KB rule and the tensor-core launch plan restated, the bound's
sensitivity."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _util import ROOT, synth
from test_gpu_fm_shapes import _model, _push_padded, _refused, _same, _still_trains

SIZES = [7, 5, 11, 3, 13, 4, 40]
TC_LOG2 = 24                                 # mlp.cu TC_THRESHOLD_LOG2: products of >= 2^24 multiply-adds
EPS32 = float(np.finfo(np.float32).eps)
FLOOR = 1e-30                                # absolute floor of the element-wise bound
# Calibrated on a B200 at its 1 000 W power limit: the largest |C - C64| / (|A| |B|)_ij over GEMM_CASES was 2.42e-6
# (M = N = 2048; each case's own figure is noted beside it), so TAU = 7.63e-6 leaves a margin of 3x.  TAU_SUM bounds
# the column sums (plain fp32 adds) relative to sum_k |A(m,k)|: largest measured 8.3e-8, TAU_SUM = 9.5e-7.
TAU = 2.0 ** -17
TAU_SUM = 2.0 ** -20
SENTINEL = 1234.5


@pytest.fixture(autouse=True)
def _restore_switches():
    yield
    os.environ.pop("FMB_HEDGE_SINGLE", None)
    if torch.cuda.is_available():
        _lib().fmb_set_tensor_cores(1)


def _lib():
    import fm_for_online_recommendation_b200 as pkg
    return pkg.require_cuda()


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


# ---------------------------------------------------------------------------------------------------------------------
# towers: covering set, scaling, premises
# ---------------------------------------------------------------------------------------------------------------------
def _largest_product(B, k, L, H):
    """the largest M * N * K among the tower's forward, dX and dW products (mlp.cu sends each to the tensor cores from
    2^24 on): B x H x k for the first layer, B x H x H for the others"""
    return B * H * max(k, H if L > 1 else 0)


# (kind, update mode, H, k, L, B): every H edge of the 64-wide tile and of online.cu's two-outputs-per-thread split for
# both classes, each k edge of the 16-deep tile, L in {1, 2, 7}, B in {1, 63, 64, 65} and larger, B * H * H < 2^24
SIMT_CASES = [
    ("DeepFMAdam", 0, 1, 1, 1, 65), ("NFMAdam", 1, 1, 17, 7, 1000),
    ("DeepFMAdam", 1, 3, 4, 2, 64), ("NFMAdam", 0, 3, 124, 1, 63),
    ("DeepFMAdam", 0, 4, 15, 7, 63), ("NFMAdam", 1, 4, 16, 2, 250),
    ("DeepFMAdam", 1, 31, 16, 1, 1), ("NFMAdam", 0, 31, 33, 7, 65),
    ("DeepFMAdam", 0, 32, 17, 2, 64), ("NFMAdam", 1, 32, 1, 7, 1),
    ("DeepFMAdam", 1, 33, 33, 7, 65), ("NFMAdam", 0, 33, 4, 1, 1000),
    ("DeepFMAdam", 0, 63, 124, 1, 1), ("NFMAdam", 1, 63, 15, 2, 63),
    ("DeepFMAdam", 1, 64, 1, 7, 63), ("NFMAdam", 0, 64, 16, 2, 64),
    ("DeepFMAdam", 0, 65, 4, 2, 1000), ("NFMAdam", 1, 65, 17, 7, 65),
    ("DeepFMAdam", 1, 127, 15, 1, 64), ("NFMAdam", 0, 127, 33, 2, 1),
    ("DeepFMAdam", 0, 128, 16, 7, 65), ("NFMAdam", 1, 128, 124, 1, 1000),
    ("DeepFMAdam", 1, 129, 17, 2, 1), ("NFMAdam", 0, 129, 1, 7, 63),
    ("DeepFMAdam", 0, 255, 33, 7, 64), ("NFMAdam", 1, 255, 4, 2, 255),
    ("DeepFMAdam", 1, 256, 124, 2, 255), ("NFMAdam", 0, 256, 15, 1, 65),
    ("DeepFMAdam", 0, 257, 1, 1, 63), ("NFMAdam", 1, 257, 16, 7, 1),
    ("DeepFMAdam", 1, 400, 4, 7, 65), ("NFMAdam", 0, 400, 17, 2, 104),
    ("DeepFMAdam", 0, 511, 15, 2, 64), ("NFMAdam", 1, 511, 124, 7, 63),
]
# hedge fit on the L-pass route (SIMT): (kind, H, k, L, batch_size)
HEDGE_CASES = [
    ("DeepFMOnn", 1, 4, 3, 64), ("NFMOnn", 31, 16, 2, 65), ("DeepFMOnn", 32, 17, 3, 1), ("NFMOnn", 33, 1, 1, 63),
    ("DeepFMOnn", 63, 33, 2, 64), ("NFMOnn", 64, 15, 3, 65), ("DeepFMOnn", 65, 124, 1, 1), ("NFMOnn", 127, 4, 2, 63),
    ("DeepFMOnn", 128, 16, 3, 64), ("NFMOnn", 129, 17, 2, 65), ("DeepFMOnn", 255, 1, 3, 63), ("NFMOnn", 256, 33, 2, 64),
    ("DeepFMOnn", 257, 15, 3, 65), ("NFMOnn", 400, 124, 2, 1), ("DeepFMOnn", 511, 4, 3, 63),
]
# head sums through ATen's cascade (H >= 512), SIMT: (kind, update mode, H, k, L, B)
CASCADE_CASES = [("DeepFMAdam", 1, 512, 4, 2, 3), ("NFMAdam", 0, 1000, 17, 2, 2), ("DeepFMAdam", 1, 2047, 1, 2, 1),
                 ("DeepFMOnn", 0, 1000, 16, 3, 3)]
RUN_KINDS = ["DeepFMAdam", "NFMAdam", "DeepFMOnn", "NFMOnn"]
RUN_HS = [1, 31, 32, 33, 255, 256, 257, 511]
RUN_N = 48
ONLINE_F, ONLINE_K, ONLINE_H = len(SIZES), 4, 511


def _run_k(H, L):
    return [1, 4, 15, 16, 17, 33, 124][(RUN_HS.index(H) + L) % 7]


def _shape_tower(orc, Xi, Xv):
    """Rescale the oracle's tower in place (float32) so that on the calibration batch every layer's pre-activations
    spread by rho = min(1, 2 / H) and every neuron's threshold sits between two consecutive distinct values of its
    pre-activations, where it leaves the active fraction closest to one half (ties count: a relu'd single neuron feeds
    many exact zeros to the next layer).  So about half of each layer is active, whatever the depth, and each head (a
    sum of H activations) stays O(1): no sigmoid saturates and no gradient is vacuously zero."""
    x = orc.fm_parts(Xi, Xv)["bi"].astype(np.float64)
    rho = min(1.0, 2.0 / orc.H)
    for W, c in orc.layer_views():
        pre = x @ W.astype(np.float64).T
        s = pre.std()
        if s > 0:
            W *= np.float32(rho / s)
            pre = x @ W.astype(np.float64).T
        for j in range(orc.H):
            u, cnt = np.unique(pre[:, j], return_counts=True)
            if len(u) == 1:
                c[j] = np.float32(-u[0] + rho / 2)
                continue
            above = (cnt.sum() - np.cumsum(cnt))[:-1] / cnt.sum()      # active fraction above u[i], u[i + 1]'s midpoint
            i = int(np.argmin(np.abs(above - 0.5)))
            c[j] = np.float32(-(u[i] + u[i + 1]) / 2)
        x = np.maximum(pre + c.astype(np.float64), 0.0)


def _top_active(orc, Xi, Xv):
    """fraction of the top layer's activations above zero, in float64 from the oracle's parameters"""
    x = orc.fm_parts(Xi, Xv)["bi"].astype(np.float64)
    for W, c in orc.layer_views():
        x = np.maximum(x @ W.astype(np.float64).T + c.astype(np.float64), 0.0)
    return float((x > 0).mean())


def _calib(orc, seed, first=None):
    """_shape_tower on 64 calibration samples and the first batch the case steps on (Xi, Xv)"""
    Xi, Xv, _ = synth(orc.feature_sizes, 64, seed + 999, real_xv=True)
    if first is not None:
        Xi, Xv = np.concatenate([Xi, first[0]]), np.concatenate([Xv, first[1]])
    _shape_tower(orc, Xi, Xv)


def _bare_oracle(kind, k, L, H, mode, **kw):
    """the oracle test_gpu_fm_shapes._model builds, without the CUDA model"""
    from oracle.deep import OracleDeep
    lr = 0.05 if mode else 1e-3
    orc = OracleDeep(kind, SIZES, k, L, H, lr=lr, seed=0, update_mode=min(mode, 1), **kw)
    orc.w1 *= np.float32(0.1)
    orc.V *= np.float32(0.1)
    orc.bias[:] = np.float32(0.1)
    return orc


def _premise(orc, Xi, Xv, B, tc_side=False):
    frac = _top_active(orc, Xi, Xv)
    assert 0.1 <= frac <= 0.9, ("top layer's active fraction", frac)
    big = _largest_product(B, orc.k, orc.L, orc.H) >= 1 << TC_LOG2
    assert big == tc_side, ("side of the 2^24 rule", B, orc.k, orc.L, orc.H)


def _batches(B, seed, n=3):
    """real-valued, then Zipf all-ones, then real-valued: the fit's eager call, capture and replay"""
    return [synth(SIZES, B, seed + i, real_xv=(i != 1), zipf=(i == 1)) for i in range(n)]


def _tower_pair(kind, mode, H, k, L, seed, first=None, **kw):
    m, orc = _model(kind, SIZES, k, mode, L, H, **kw)
    _calib(orc, seed, first)
    _push_padded(m, orc)
    return m, orc


def _forward_same(m, orc, Xi, Xv, step):
    got, want = m.forward(Xi, Xv), orc.forward(Xi, Xv)
    if isinstance(got, tuple):
        assert np.array_equal(got[0].cpu().numpy(), want[0]) and np.array_equal(got[1].cpu().numpy(), want[1]), step
    else:
        assert np.array_equal(got.cpu().numpy(), want), (step, "forward")
    assert np.array_equal(m.predict(Xi, Xv), orc.predict(Xi, Xv)), (step, "predict")


def _tower_steps(m, orc, batches):
    for i, (Xi, Xv, Y) in enumerate(batches):
        _forward_same(m, orc, Xi, Xv, i)
        m.fit(Xi, Xv, Y)
        orc.fit(Xi, Xv, Y)
        _same(m, orc, ("fit", i))
        got = m.update_embedding(Xi, Xv, Y).item()
        want = orc.update_embedding(Xi, Xv, Y)
        assert np.float32(got) == np.float32(want), (i, got, want)
        _same(m, orc, ("update_embedding", i))


def _online_smem_bytes(F, k, L, H):
    """online.cu's shared-memory need of one CTA (host code of fmb_online_deep_run_ex restated); refused above 200 KB"""
    cu = (k + 1 + 3) // 4
    mx = max(H, k)
    return 4 * (F * cu * 4 + 2 * F + 2 * k + L * H + 2 * mx + k + 2 * max(L, 1) + 16)


def _online_largest_L(F, k, H):
    L = 1
    while _online_smem_bytes(F, k, L + 1, H) <= 200 * 1024:
        L += 1
    return L


# ---------------------------------------------------------------------------------------------------------------------
# tensor cores: launch plan, element-wise float64 bound
# ---------------------------------------------------------------------------------------------------------------------
TBM, TBK, MAX_K_PER_PASS, SMS = 128, 32, 1024, 148


def _cdiv(a, b):
    return -(-a // b)


def _tc_plan(M, N, K, sms=SMS):
    """gemm_tc.cu's launch plan restated (tile width, tiles, splits, kchunk) with the split count after each rule"""
    n128, n208 = _cdiv(N, 128), _cdiv(N, 208)
    tbn = 208 if n208 * 208 < n128 * 128 else 128
    tiles = _cdiv(M, TBM) * (n208 if tbn == 208 else n128)
    wave = sms // tiles if tiles * 2 <= sms else 1
    passes = max(wave, _cdiv(K, MAX_K_PER_PASS))
    capped = max(min(passes, _cdiv(K, 4 * TBK)), 1)
    kchunk = _cdiv(_cdiv(K, capped), TBK) * TBK
    splits = _cdiv(K, kchunk)
    return dict(tbn=tbn, tiles=tiles, wave=wave, passes=passes, capped=capped, kchunk=kchunk, splits=splits)


# (M, N, K, layout of A, layout of B, epilogue, column sums): every M, N and K edge, both tile widths, each operand
# layout the loads tell apart (kc: K-contiguous, 16-byte aligned; kc_odd: row stride % 4 != 0; off1: base one float
# past an aligned address; rc: row-contiguous, the dW / dX forms), the three epilogues
GEMM_CASES = [   # measured on the B200: largest err / (|A| |B|)_ij, and of the column sums
    (1, 1, 1, "kc", "kc", 0, True),                  # 1.9e-07, 0.0e+00
    (127, 4, 31, "kc_odd", "kc", 1, False),          # 5.1e-07
    (128, 128, 32, "kc", "kc", 2, True),             # 6.7e-07, 3.9e-08
    (129, 129, 33, "off1", "kc_odd", 0, True),       # 8.0e-07, 5.2e-08
    (8192, 208, 1024, "kc", "kc", 1, False),         # 1.1e-06
    (129, 209, 1025, "rc", "kc", 2, True),           # 2.8e-07, 1.4e-08
    (128, 400, 4097, "kc", "rc", 0, True),           # 1.4e-07, 1.4e-08
    (8192, 417, 33, "rc", "rc", 2, False),           # 1.0e-06
    (127, 624, 1024, "off1", "off1", 1, True),       # 2.8e-07, 1.4e-08
    (129, 624, 4097, "kc_odd", "kc_odd", 2, True),   # 1.8e-07, 8.4e-09
    (8192, 624, 4097, "rc", "rc", 0, True),          # 8.7e-07, 1.0e-08
    (129, 1, 1025, "rc", "off1", 1, False),          # 1.5e-07
    (128, 4, 4097, "kc", "off1", 0, True),           # 1.3e-07, 1.4e-08
    (8192, 128, 31, "off1", "rc", 0, True),          # 8.9e-07, 8.3e-08
    (127, 129, 1, "rc", "kc", 2, True),              # 1.3e-06, 0.0e+00
    (1, 209, 32, "off1", "rc", 1, True),             # 5.5e-07, 7.7e-09
    (2048, 2048, 1024, "kc", "kc", 0, True),         # 2.4e-06, 2.2e-08
    (2048, 2048, 1000, "rc", "rc", 2, True),         # 2.2e-06, 2.4e-08
    (8192, 400, 1025, "kc", "kc", 1, True),          # 1.3e-06, 2.3e-08
    (128, 417, 1024, "kc_odd", "rc", 2, False),      # 2.7e-07
    (8192, 209, 4097, "kc", "kc", 0, False),         # 7.7e-07
]
# fmb_mlp_forward / backward / backward_hedge with the tensor cores on: (B, H, k, L)
TOWER_TC_SHAPES = [(256, 256, 10, 3), (1024, 400, 10, 3), (8192, 130, 17, 2), (300, 1500, 8, 2)]


def _operand(rows, K, layout, gen):
    """rows x K operand X(r, k) laid out as `layout` over padded storage (the padding holds values a load past the edge
    would pick up).  Returns (storage, address, stride of r, stride of k, X as a strided view)."""
    dev = "cuda" if gen.device.type == "cuda" else "cpu"
    if layout == "rc":
        ld = rows + 3
        s = torch.randn(K, ld, generator=gen, device=dev)
        return s, s.data_ptr(), 1, ld, s[:, :rows].t()
    ld = _cdiv(K, 4) * 4 + (1 if layout == "kc_odd" else 0)
    off = 1 if layout == "off1" else 0
    flat = torch.randn(rows * ld + off, generator=gen, device=dev)
    s = flat[off:].view(rows, ld)
    return flat, s.data_ptr(), ld, 1, s[:, :K]


def _worst(err, mag):
    return float((err / (mag + FLOOR)).max()) if err.numel() else 0.0


def _within(got, ref, mag, tau, what):
    """|got - ref| <= tau * mag + FLOOR element by element; returns the largest err / mag"""
    err = (got.double() - ref).abs()
    bad = err > tau * mag + FLOOR
    assert not bool(bad.any()), (what, int(bad.sum()), _worst(err, mag))
    return _worst(err, mag)


def _gemm_case(lib, case, seed, tau=TAU, tau_sum=TAU_SUM):
    """one fmb_gemm_tc_strided launch against float64; C and the column sums sit in sentinel-filled buffers larger than
    the result (scm > N, extra rows); a repeat launch is bit-identical.  Returns the worst ratios (product, column sums)."""
    M, N, K, la, lb, epi, cs = case
    g = torch.Generator(device="cuda").manual_seed(seed)
    sa_, pa, sam, sak, A = _operand(M, K, la, g)
    sb_, pb, sbn, sbk, Bt = _operand(N, K, lb, g)        # Bt[n, k] = B(k, n)
    scm = N + (3 if seed % 2 else 4)
    Cbuf = torch.full((M + 5, scm), SENTINEL, device="cuda")
    colsum = torch.full((M + 8,), SENTINEL, device="cuda") if cs else None
    bias = mask = None
    smm = 0
    if epi == 1:
        bflat = torch.randn(N + 1, generator=g, device="cuda")
        bias = bflat[seed % 2:seed % 2 + N]
    if epi == 2:
        smm = N + (1 if seed % 3 == 0 else 4)
        mflat = torch.randn(M, smm, generator=g, device="cuda")
        mask = mflat[:, :N]
    A64, B64 = A.double(), Bt.double()
    ref = A64 @ B64.t()
    mag = A64.abs() @ B64.abs().t()
    if epi == 1:
        ref = torch.relu(ref + bias.double())
        mag = mag + bias.double().abs()
    elif epi == 2:
        ref = ref * (mask > 0)
    outs = []
    for _ in range(2):
        assert lib.fmb_gemm_tc_strided(C.c_void_p(pa), sam, sak, C.c_void_p(pb), sbk, sbn, _p(Cbuf), scm, M, N, K, epi,
                                       _p(bias), None if mask is None else C.c_void_p(mask.data_ptr()), smm, _p(colsum),
                                       None) == 0, lib.fmb_last_error()
        torch.cuda.synchronize()
        outs.append((Cbuf.clone(), None if colsum is None else colsum.clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and (colsum is None or torch.equal(outs[0][1], outs[1][1])), case
    Cout = outs[0][0]
    out = Cout[:M, :N]
    edge = torch.ones_like(Cout, dtype=torch.bool)
    edge[:M, :N] = False
    assert bool((Cout[edge] == SENTINEL).all()), (case, "written outside C", int((Cout[edge] != SENTINEL).sum()))
    r = _within(out, ref, mag, tau, case)
    rs = 0.0
    if cs:
        c = outs[0][1]
        assert bool((c[M:] == SENTINEL).all()), (case, "written past the column sums")
        rs = _within(c[:M], A64.sum(1), A64.abs().sum(1), tau_sum, (case, "colsum"))
    return r, rs


def _mlp_offsets(k, L, H):
    offs, o = [], 0
    for l in range(L):
        nin = k if l == 0 else H
        offs.append((o, o + H * nin, nin))
        o += H * nin + H
    return offs, o


def _tower_tc_case(lib, B, H, k, L, seed, tau=TAU, tau_sum=TAU_SUM, hedge=False):
    """fmb_mlp_forward, then fmb_mlp_backward (or fmb_mlp_backward_hedge) on the same activations, against float64.
    Forward: each layer from the kernel's own input layer.  Backward: the reference gradient flows down from the top in
    float64 through the kernel's relu masks, and a first-order bound E on the kernel's error in it flows beside it, so
    every output (weight and bias gradients, gbi) is checked element by element.  Returns the forward's largest
    err / (|x| |W| + |c|) and the backward's largest err / bound."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    offs, n = _mlp_offsets(k, L, H)
    mlp = torch.empty(n, device="cuda")
    for o, c0, nin in offs:
        mlp[o:c0] = torch.randn(H * nin, generator=g, device="cuda") * (2.0 / nin) ** 0.5
        mlp[c0:c0 + H] = torch.randn(H, generator=g, device="cuda") * 0.1
    bi = torch.randn(B, k, generator=g, device="cuda")
    act = torch.empty(L, B, H, device="cuda")
    head = torch.empty(L, B, device="cuda")
    assert lib.fmb_mlp_forward(_p(bi), k, _p(mlp), B, k, L, H, _p(act), _p(head), None) == 0, lib.fmb_last_error()
    wsb = lib.fmb_mlp_bwd_workspace_bytes(B, H)
    ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
    gm = torch.full((n,), SENTINEL, device="cuda")
    if hedge:
        gtop = torch.randn(L, B, generator=g, device="cuda") / B
        alpha = torch.rand(L, generator=g, device="cuda") + 0.1
        alpha /= alpha.sum()
        assert lib.fmb_mlp_backward_hedge(_p(bi), k, _p(mlp), _p(act), _p(gtop), _p(alpha), B, k, L, H, _p(gm), _p(ws),
                                          wsb, None) == 0, lib.fmb_last_error()
    else:
        gtop = torch.randn(B, generator=g, device="cuda") / B
        gbi = torch.full((B, k), SENTINEL, device="cuda")
        assert lib.fmb_mlp_backward(_p(bi), k, _p(mlp), _p(act), _p(gtop), L - 1, B, k, L, H, _p(gm), _p(gbi), k, _p(ws),
                                    wsb, None) == 0, lib.fmb_last_error()
    torch.cuda.synchronize()
    assert lib.fmb_gemm_tc_error() == 0
    a64 = act.double()
    xs = [bi.double()] + [a64[l] for l in range(L - 1)]
    Ws = [mlp[o:c0].double().view(H, nin) for o, c0, nin in offs]
    cs = [mlp[c0:c0 + H].double() for o, c0, nin in offs]
    worst, worst_b = 0.0, 0.0
    for l in range(L):
        ref = torch.relu(xs[l] @ Ws[l].t() + cs[l])
        mag = xs[l].abs() @ Ws[l].abs().t() + cs[l].abs()
        worst = max(worst, _within(act[l], ref, mag, tau, ("forward", l)))
        hs = a64[l].sum(1)
        assert bool(((head[l].double() - hs).abs() <= H * EPS32 * a64[l].abs().sum(1) + FLOOR).all()), ("head", l)
    masks = [a64[l] > 0 for l in range(L)]
    if hedge:
        t = masks[L - 1] * (alpha[L - 1].double() * gtop[L - 1].double())[:, None]
        gp, E = t, EPS32 * t.abs()
    else:
        gp, E = masks[L - 1] * gtop.double()[:, None], torch.zeros(B, H, dtype=torch.float64, device="cuda")
    for l in range(L - 1, -1, -1):
        o, c0, nin = offs[l]
        x = xs[l]
        gW = gm[o:c0].view(H, nin)
        pa = gp.abs() + E
        worst_b = max(worst_b, _within(gW, gp.t() @ x, tau * (pa.t() @ x.abs()) + E.t() @ x.abs(), 1.0, ("dW", l)))
        worst_b = max(worst_b, _within(gm[c0:c0 + H], gp.sum(0), tau_sum * pa.sum(0) + E.sum(0), 1.0, ("dc", l)))
        gx = gp @ Ws[l]
        Ex = tau * (pa @ Ws[l].abs()) + E @ Ws[l].abs()
        if l > 0:
            gp, E = masks[l - 1] * gx, masks[l - 1] * Ex
            if hedge:
                t = masks[l - 1] * (alpha[l - 1].double() * gtop[l - 1].double())[:, None]
                E = E + 3 * EPS32 * masks[l - 1] * (gx.abs() + t.abs())
                gp = gp + t
        elif not hedge:
            worst_b = max(worst_b, _within(gbi, gx, Ex, 1.0, "gbi"))
    return worst, worst_b


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def _premise_cases():
    out = [("simt", kind, mode, H, k, L, B) for kind, mode, H, k, L, B in SIMT_CASES]
    out += [("hedge", kind, 0, H, k, L, B) for kind, H, k, L, B in HEDGE_CASES]
    out += [("cascade", kind, mode, H, k, L, B) for kind, mode, H, k, L, B in CASCADE_CASES]
    out += [("modes", "DeepFMAdam", 1, 511, 15, 3, 64), ("modes", "NFMAdam", 1, 511, 33, 3, 63)]
    return out


def test_simt_covering_set_reaches_every_edge():
    Hs = {c[2] for c in SIMT_CASES}
    assert Hs == {1, 3, 4, 31, 32, 33, 63, 64, 65, 127, 128, 129, 255, 256, 257, 400, 511}
    assert {c[3] for c in SIMT_CASES} == {1, 4, 15, 16, 17, 33, 124}
    assert {c[4] for c in SIMT_CASES} == {1, 2, 7}
    assert {1, 63, 64, 65} < {c[5] for c in SIMT_CASES}
    for kind in ("DeepFMAdam", "NFMAdam"):
        for mode in (0, 1):
            assert any(c[0] == kind and c[1] == mode for c in SIMT_CASES)
    assert {c[1] for c in HEDGE_CASES} == Hs - {3, 4}
    assert {c[2] for c in CASCADE_CASES} == {512, 1000, 2047} and max(c[5] for c in CASCADE_CASES) <= 3


@pytest.mark.parametrize("case", _premise_cases(), ids=lambda c: "-".join(str(v) for v in c))
def test_tower_case_premise(case):
    """each SIMT case's scaled tower has a top layer between 10 % and 90 % active on its first batch, and its largest
    product is below 2^24"""
    what, kind, mode, H, k, L, B = case
    kw = dict(batch_size=B) if kind.endswith("Onn") else {}
    orc = _bare_oracle(kind, k, L, H, mode, **kw)
    seed = 7 * H + L
    Xi, Xv, _ = _batches(B, seed)[0]
    _calib(orc, seed, (Xi, Xv))
    _premise(orc, Xi, Xv, B)


@pytest.mark.parametrize("kind", RUN_KINDS)
@pytest.mark.parametrize("L", [1, 3])
def test_run_experiment_premise(kind, L):
    for H in RUN_HS:
        orc = _bare_oracle(kind, _run_k(H, L), L, H, 1)
        Xi, Xv, _ = synth(SIZES, RUN_N, 50 + H + L, real_xv=True)
        _calib(orc, H + L, (Xi, Xv))
        _premise(orc, Xi, Xv, 1)


def test_tc_off_tower_premise():
    orc = _bare_oracle("DeepFMAdam", 10, 3, 256, 1)
    Xi, Xv, _ = _batches(2048, 3)[0]
    _calib(orc, 3, (Xi, Xv))
    _premise(orc, Xi, Xv, 2048, tc_side=True)


def test_online_largest_tower_by_the_200kb_rule():
    """the rule restated: at H = 511 the largest accepted L fills the 200 KB to within one layer; L + 1 exceeds it"""
    L = _online_largest_L(ONLINE_F, ONLINE_K, ONLINE_H)
    assert _online_smem_bytes(ONLINE_F, ONLINE_K, L, ONLINE_H) <= 200 * 1024 < _online_smem_bytes(ONLINE_F, ONLINE_K, L + 1,
                                                                                                   ONLINE_H)
    assert L == 97
    assert _online_smem_bytes(300, 124, 24, 500) > 200 * 1024       # the refusal test_gpu_fm_shapes already checks


def test_tc_launch_plan_reaches_every_branch():
    """the direct cases reach both tile widths, splits set by the one-wave rule, by the 1 024-term pass limit, capped by
    the four-slices rule, reduced by kchunk's rounding, a single split with a grid of more than half the SMs, a single
    partial slice, and column sums through both the split and the non-split reduction"""
    plans = {c: _tc_plan(*c[:3]) for c in GEMM_CASES}
    assert {p["tbn"] for p in plans.values()} == {128, 208}
    assert any(p["wave"] > 1 and p["splits"] == p["wave"] for p in plans.values())
    assert any(p["passes"] > p["wave"] and p["splits"] > 1 for p in plans.values())
    assert any(p["capped"] < p["passes"] for p in plans.values())
    assert any(p["splits"] < p["capped"] for p in plans.values())
    assert any(p["tiles"] * 2 > SMS and p["splits"] == 1 for p in plans.values())
    assert any(c[2] < TBK for c in GEMM_CASES)
    assert any(c[6] and p["splits"] == 1 and p["tiles"] * 2 > SMS for c, p in plans.items())
    assert any(c[6] and p["splits"] > 1 for c, p in plans.items())
    assert any(p["kchunk"] * (p["splits"] - 1) < c[2] < p["kchunk"] * p["splits"] for c, p in plans.items())
    for v, pos in (({1, 127, 128, 129, 8192}, 0), ({1, 4, 128, 129, 208, 209, 400, 417, 624}, 1),
                   ({1, 31, 32, 33, 1024, 1025, 4097}, 2)):
        assert v <= {c[pos] for c in GEMM_CASES}
    assert {c[3] for c in GEMM_CASES} | {c[4] for c in GEMM_CASES} == {"kc", "kc_odd", "off1", "rc"}
    assert {c[5] for c in GEMM_CASES} == {0, 1, 2}
    # the tower shapes: fmb_mlp_backward's dW at (300, 1500) takes the non-split column sums
    assert _tc_plan(1500, 1500, 300)["splits"] == 1 and _tc_plan(400, 400, 1024)["splits"] > 1
    for B, H, k, L in TOWER_TC_SHAPES:
        assert _largest_product(B, k, L, H) >= 1 << TC_LOG2


def test_elementwise_bound_catches_each_defect():
    """the bound with TAU / TAU_SUM is not vacuous at the largest K: one dropped 32-wide K-slice, an omitted bias, a
    flipped relu-mask entry and a column sum missing one split each leave it for most elements"""
    M, N, K = 129, 209, 4097
    g = torch.Generator().manual_seed(0)
    A = torch.randn(M, K, generator=g, dtype=torch.float64)
    Bm = torch.randn(K, N, generator=g, dtype=torch.float64)
    bias = torch.randn(N, generator=g, dtype=torch.float64)
    C0 = A @ Bm
    mag = A.abs() @ Bm.abs()
    caught = lambda d, m, tau=TAU: float(((d.abs() > tau * m + FLOOR)).double().mean())
    s = 64 * TBK
    assert caught(A[:, s:s + TBK] @ Bm[s:s + TBK], mag) > 0.9                                   # dropped K-slice
    ref, magb = torch.relu(C0 + bias), mag + bias.abs()
    live = ref > 0
    assert caught((torch.relu(C0) - ref)[live], magb[live]) > 0.9                               # omitted bias
    assert caught(C0, mag) > 0.9                                           # any one relu-mask entry flipped
    plan = _tc_plan(M, N, K)
    kc = plan["kchunk"]
    assert plan["splits"] > 1
    assert caught(A[:, kc:2 * kc].sum(1), A.abs().sum(1), TAU_SUM) > 0.9                        # colsum less a split


# ---------------------------------------------------------------------------------------------------------------------
# 1. SIMT towers and the per-example kernel, bit for bit
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind,mode,H,k,L,B", SIMT_CASES)
def test_simt_tower_fit_bit_exact(kind, mode, H, k, L, B):
    """forward, predict, fit (eager, captured, replayed) and update_embedding: V, w1, bias, tower after every step"""
    assert _lib().fmb_tensor_core_threshold_log2() == TC_LOG2
    batches = _batches(B, 7 * H + L)
    m, orc = _tower_pair(kind, mode, H, k, L, 7 * H + L, batches[0][:2])
    _premise(orc, batches[0][0], batches[0][1], B)
    _tower_steps(m, orc, batches)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,H,k,L,B", HEDGE_CASES)
def test_hedge_fit_l_pass_bit_exact(kind, H, k, L, B):
    """hedge backpropagation on the L-pass route (the products are SIMT): tower and alpha after every fit"""
    batches = _batches(B, 7 * H + L)
    m, orc = _tower_pair(kind, 0, H, k, L, 7 * H + L, batches[0][:2], batch_size=B)
    assert not m._hedge_single_pass(B)
    _premise(orc, batches[0][0], batches[0][1], B)
    _tower_steps(m, orc, batches)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,mode,H,k,L,B", CASCADE_CASES)
def test_head_sums_through_aten_cascade(kind, mode, H, k, L, B):
    """H >= 512: the head sums take ATen's multi-level cascade (fmb::aten_row_sum_warp), still bit-exact"""
    kw = dict(batch_size=B) if kind.endswith("Onn") else {}
    batches = _batches(B, 7 * H + L)
    m, orc = _tower_pair(kind, mode, H, k, L, 7 * H + L, batches[0][:2], **kw)
    _premise(orc, batches[0][0], batches[0][1], B)
    _tower_steps(m, orc, batches)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [3, 4])
def test_large_tower_adagrad_and_sparse_adam(mode):
    """modes 3 and 4 at H = 511, L = 3 (B * H * H just under 2^24) against their oracles: weights and optimizer state"""
    if mode == 3:
        import test_gpu_adagrad as t
        m, orc, st = t._model("DeepFMAdam", SIZES, 15, 3, 511)
        same = t._same_ada
    else:
        import test_gpu_sparse_adam as t
        m, orc, st = t._model("NFMAdam", SIZES, 33, 3, 511)
        same = t._same_sa
    B = 64 if mode == 3 else 63
    batches = _batches(B, 7 * 511 + 3)
    _calib(orc, 7 * 511 + 3, batches[0][:2])
    _push_padded(m, orc)
    _premise(orc, batches[0][0], batches[0][1], B)
    for i, (Xi, Xv, Y) in enumerate(batches):
        m.fit(Xi, Xv, Y)
        st.fit(Xi, Xv, Y)
        same(m, orc, st, ("fit", i))
        got = m.update_embedding(Xi, Xv, Y).item()
        assert np.float32(got) == np.float32(st.update_embedding(Xi, Xv, Y)), i
        same(m, orc, st, ("update_embedding", i))


@pytest.mark.gpu
def test_tower_above_threshold_with_tensor_cores_off_bit_exact():
    """B = 2048, H = 256, L = 3 is above 2^24; with the tensor cores switched off the tower stays on the SIMT kernel and
    is bit-identical to the oracle (the premise of test_gpu_deep's tensor-core-vs-SIMT comparisons)"""
    lib = _lib()
    lib.fmb_set_tensor_cores(0)
    batches = _batches(2048, 3)
    m, orc = _tower_pair("DeepFMAdam", 1, 256, 10, 3, 3, batches[0][:2])
    _premise(orc, batches[0][0], batches[0][1], 2048, tc_side=True)
    _tower_steps(m, orc, batches)


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 3])
@pytest.mark.parametrize("H", RUN_HS)
@pytest.mark.parametrize("kind", RUN_KINDS)
def test_run_experiment_tower_shapes(kind, H, L):
    """the per-example kernel at the warp edges of H, and H > 256 (two outputs per thread), with real-valued Xv"""
    kw = dict(batch_size=1) if kind.endswith("Onn") else {}
    Xi, Xv, Y = synth(SIZES, RUN_N, 50 + H + L, real_xv=True)
    m, orc = _tower_pair(kind, 1, H, _run_k(H, L), L, H + L, (Xi, Xv), **kw)
    _premise(orc, Xi, Xv, 1)
    _, _, _, conf = m.run_experiment(Xi, Xv, Y)
    oconf, opreds = orc.run_experiment(Xi, Xv, Y)
    assert conf == oconf
    assert np.array_equal(m._last_online_preds, opreds)
    _same(m, orc)


@pytest.mark.gpu
def test_run_experiment_largest_tower_and_refusal():
    """the largest L the 200 KB rule accepts at H = 511 runs bit-exact; L + 1 is refused with the shape in the message,
    and the process still trains"""
    import fm_for_online_recommendation_b200 as pkg
    F, k, H = ONLINE_F, ONLINE_K, ONLINE_H
    L = _online_largest_L(F, k, H)
    Xi, Xv, Y = synth(SIZES, 24, 12, real_xv=True)
    m, orc = _tower_pair("DeepFMAdam", 1, H, k, L, 11, (Xi, Xv))
    _premise(orc, Xi, Xv, 1)
    _, _, _, conf = m.run_experiment(Xi, Xv, Y)
    oconf, opreds = orc.run_experiment(Xi, Xv, Y)
    assert conf == oconf and np.array_equal(m._last_online_preds, opreds)
    _same(m, orc)
    del m, orc
    m = pkg.DeepFMAdam(SIZES, embedding_size=k, num_hidden_layers=L + 1, neuron_per_hidden_layer=H, n=0.01)
    _refused(m, lambda: m.run_experiment(Xi, Xv, Y), f"F={F}", f"k={k}", f"L={L + 1}", f"H={H}")
    del m
    _still_trains()


# ---------------------------------------------------------------------------------------------------------------------
# 2. tensor cores against float64, element by element
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("case", GEMM_CASES, ids=lambda c: "-".join(str(v) for v in c))
def test_tensor_core_gemm_elementwise(case):
    """fmb_gemm_tc_strided against float64 per element; nothing outside C or the column sums is written; a repeat launch
    is bit-identical.  Largest err / (|A| |B|)_ij measured on a B200: beside each case in GEMM_CASES"""
    lib = _lib()
    assert torch.cuda.get_device_properties(0).multi_processor_count == SMS
    _gemm_case(lib, case, GEMM_CASES.index(case))
    assert lib.fmb_gemm_tc_error() == 0


@pytest.mark.gpu
@pytest.mark.parametrize("B,H,k,L", TOWER_TC_SHAPES)
@pytest.mark.parametrize("hedge", [False, True])
def test_tower_tensor_cores_elementwise(B, H, k, L, hedge):
    """fmb_mlp_forward with fmb_mlp_backward or fmb_mlp_backward_hedge on the tensor cores, against float64.  Measured on
    the B200: forward err / (|x| |W| + |c|) at most 9.5e-7 (8192 x 130); the backward used at most 28 % of its bound
    (300 x 1500)"""
    _tower_tc_case(_lib(), B, H, k, L, B + H, hedge=hedge)


@pytest.mark.gpu
def test_tensor_core_dispatch_boundary():
    """H = 256: at B = 255 every product is below 2^24 and the tower is the same with the tensor cores on and off; at
    B = 256 the H x H products reach 2^24, go to the tensor cores, differ, and stay within the float64 bound"""
    lib = _lib()
    H, k, L = 256, 10, 3
    assert _largest_product(255, k, L, H) < 1 << TC_LOG2 <= _largest_product(256, k, L, H)

    def run(B, tc):
        lib.fmb_set_tensor_cores(tc)
        g = torch.Generator(device="cuda").manual_seed(B)
        offs, n = _mlp_offsets(k, L, H)
        mlp = torch.randn(n, generator=g, device="cuda") * 0.1
        bi = torch.randn(B, k, generator=g, device="cuda")
        gtop = torch.randn(B, generator=g, device="cuda") / B
        act, head = torch.empty(L, B, H, device="cuda"), torch.empty(L, B, device="cuda")
        gm, gbi = torch.empty(n, device="cuda"), torch.empty(B, k, device="cuda")
        wsb = lib.fmb_mlp_bwd_workspace_bytes(B, H)
        ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")
        assert lib.fmb_mlp_forward(_p(bi), k, _p(mlp), B, k, L, H, _p(act), _p(head), None) == 0
        assert lib.fmb_mlp_backward(_p(bi), k, _p(mlp), _p(act), _p(gtop), L - 1, B, k, L, H, _p(gm), _p(gbi), k, _p(ws),
                                    wsb, None) == 0
        torch.cuda.synchronize()
        return act, head, gm, gbi

    for x, y in zip(run(255, 1), run(255, 0)):
        assert torch.equal(x, y)
    on, off = run(256, 1), run(256, 0)
    assert not torch.equal(on[0][1], off[0][1]) and not torch.equal(on[2], off[2])
    lib.fmb_set_tensor_cores(1)
    _tower_tc_case(lib, 256, H, k, L, 256)
    assert lib.fmb_gemm_tc_error() == 0


# ---------------------------------------------------------------------------------------------------------------------
# 3. fit graphs across batch-size sequences
# ---------------------------------------------------------------------------------------------------------------------
_PATTERN = {torch.float32: -3.5, torch.int32: 0x5A5A5A5A, torch.uint8: 0xA5}


@pytest.mark.gpu
def test_fit_graphs_after_workspace_growth_simt():
    """DeepFMAdam.fit at B = 64, 64, 256, 256, 64, 64, 64: eager, capture, eager with growth, then captures and replays.
    The growth hands the B = 64 workspaces back to torch's allocator; tensors of exactly their sizes are taken and filled
    right after it, and a second model is built and stepped between the fits.  A graph still pointing at the replaced
    buffers would write into them: the pattern and both models against their oracles show it."""
    m, orc = _tower_pair("DeepFMAdam", 1, 16, 10, 2, 5)
    seq = [64, 64, 256, 256, 64, 64, 64]
    keep, m2 = [], None
    for i, B in enumerate(seq):
        Xi, Xv, Y = synth(SIZES, B, 900 + i, real_xv=True, zipf=(i % 3 == 0))   # one graph key per batch size
        before = {n: (t.data_ptr(), t.numel(), t.dtype) for n, t in m._ws.items()}
        m.fit(Xi, Xv, Y)
        orc.fit(Xi, Xv, Y)
        _same(m, orc, ("m", i, B))
        if i == 2:
            grown = [v for n, v in before.items() if m._ws[n].data_ptr() != v[0]]
            assert grown
            for _, numel, dt in grown:
                keep.append(torch.full((numel,), _PATTERN[dt], dtype=dt, device="cuda"))
            m2, orc2 = _tower_pair("DeepFMAdam", 1, 16, 10, 2, 6)
        if m2 is not None:
            b2 = synth(SIZES, 64, 950 + i, real_xv=True)
            m2.fit(*b2)
            orc2.fit(*b2)
            _same(m2, orc2, ("m2", i))
        torch.cuda.synchronize()
        for t in keep:
            assert bool((t == _PATTERN[t.dtype]).all()), ("freed workspace written", i, t.numel(), t.dtype)
    g = m._fit_graphs[(64, True, m._lr, 1, 1)]
    assert isinstance(g, tuple)


def _tc_graph_sequence():
    """body of test_fit_graphs_after_workspace_growth_tensor_cores, run in a fresh process so that the split-K workspace
    starts at the size the first B = 1024 products need and the B = 8192 fit grows it"""
    import fm_for_online_recommendation_b200 as pkg
    lib = pkg.require_cuda()
    sizes = [50, 3000, 20000, 7, 900]
    kw = dict(embedding_size=10, num_hidden_layers=3, neuron_per_hidden_layer=400, n=1e-3)

    def twins(cls, **extra):
        out = []
        for _ in range(2):
            torch.manual_seed(4)
            out.append(getattr(pkg, cls)(sizes, **kw, **extra))
        return out

    dfm, dfm_e = twins("DeepFMAdam")
    onn, onn_e = twins("DeepFMOnn", batch_size=1024)
    assert onn._hedge_single_pass(1024)

    def same(a, b, what):
        for x, y in ((a._table, b._table), (a.bias, b.bias), (a._mlp, b._mlp)):
            assert torch.equal(x, y), what
        if hasattr(a, "alpha"):
            assert torch.equal(a.alpha, b.alpha), what

    step = [0]

    def fit(m, me, B):
        Xi, Xv, Y = synth(sizes, B, 1000 + step[0], real_xv=True)   # one graph key per batch size
        step[0] += 1
        m.fit(Xi, Xv, Y)
        e = me.encode(Xi, Xv, Y)
        (me._hedge_fit if me._IS_ONN else me._deep_fit)(e)
        torch.cuda.synchronize()
        same(m, me, (type(m).__name__, B, step[0]))

    fit(onn, onn_e, 1024)          # eager
    fit(onn, onn_e, 1024)          # captured
    for B in (1024, 1024, 8192, 1024):
        fit(dfm, dfm_e, B)         # eager, captured, eager (grows both workspaces), eager (its graphs were dropped)
    fit(onn, onn_e, 1024)          # replayed: captured before the growth
    fit(dfm, dfm_e, 1024)          # captured after the growth
    fit(dfm, dfm_e, 1024)          # replayed
    fit(onn, onn_e, 1024)
    assert isinstance(onn._fit_graphs[("hedge", 1024, True, onn._lr)], tuple)
    assert lib.fmb_gemm_tc_error() == 0
    print("tc graph sequence ok")


@pytest.mark.gpu
def test_fit_graphs_after_workspace_growth_tensor_cores():
    """DeepFMAdam (H = 400) at B = 1024, 1024, 8192, 1024, 1024, 1024 and a single-pass-hedge DeepFMOnn (batch_size
    1024) captured before the B = 8192 fit grows the split-K workspace and replayed after it: each bit-identical to a
    twin that only ever calls _deep_fit / _hedge_fit eagerly (same kernels, same split order)"""
    code = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]; "
            "import test_gpu_tower_shapes as t; t._tc_graph_sequence()")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "tc graph sequence ok" in r.stdout, (r.stdout[-3000:], r.stderr[-6000:])
