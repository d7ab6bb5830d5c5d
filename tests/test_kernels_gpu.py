"""GPU parity tests of the individual CUDA kernels, called through the C ABI (ops.py -> libltgan.so), against the
CPU oracle (oracle/) or a plain torch fp32 restatement of the same op on the same seeded inputs.
Tolerances: bit-exact for integer/index work and RNG bits; bf16-operand/fp32-accumulate GEMMs within 2e-2 of the
fp32 product of the *bf16-rounded* operands scaled by sqrt(K) (the rounding of the inputs is shared)."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ltgan_oracle as orc  # noqa: E402
from oracle import philox  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    pkg = importlib.import_module("long-tail-gan_b200")
    pkg._lib.build()
    o = importlib.import_module("long-tail-gan_b200.ops")
    o.init()
    return o


def dev(x, dtype=None):
    t = torch.as_tensor(x)
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda().contiguous()


def rand_csr(rng, B, I, mean_nnz, min_nnz=1):
    indptr = [0]
    idx = []
    for _ in range(B):
        n = int(np.clip(rng.poisson(mean_nnz), min_nnz, I))
        it = np.sort(rng.choice(I, size=n, replace=False))
        idx.append(it)
        indptr.append(indptr[-1] + n)
    return np.asarray(indptr, dtype=np.int32), np.concatenate(idx).astype(np.int32)


# ----------------------------------------------------------------------------------------------------------------
# tcgen05 GEMM
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("a_mn,b_mn", [(False, False), (False, True), (True, False), (True, True)])
@pytest.mark.parametrize("bn", [64, 128, 192, 256])
def test_gemm_layouts(ops, a_mn, b_mn, bn):
    torch.manual_seed(1)
    M, N, K = 500, 600, 456  # ragged in every dimension (K tail handled by TMA zero fill)
    A = torch.randn(M, K, device="cuda").bfloat16()
    Bm = torch.randn(N, K, device="cuda").bfloat16()
    ref = A.float() @ Bm.float().t()
    # physical layouts with padded pitches (multiples of 8 elements)
    if a_mn:
        Ap = torch.zeros(K, 504, device="cuda", dtype=torch.bfloat16); Ap[:, :M] = A.t()
    else:
        Ap = torch.zeros(M, 456 + 8, device="cuda", dtype=torch.bfloat16); Ap[:, :K] = A
    if b_mn:
        Bp = torch.zeros(K, 608, device="cuda", dtype=torch.bfloat16); Bp[:, :N] = Bm.t()
    else:
        Bp = torch.zeros(N, 456 + 8, device="cuda", dtype=torch.bfloat16); Bp[:, :K] = Bm
    out = torch.full((M, 608), float("nan"), device="cuda")
    outb = torch.zeros(M, 608, device="cuda", dtype=torch.bfloat16)
    ops.gemm(Ap, Bp, M, N, K, a_mn=a_mn, b_mn=b_mn, bn=bn, out_f32=out, out_bf16=outb)
    torch.cuda.synchronize()
    err = (out[:, :N] - ref).abs().max().item()
    assert err < 2e-2 * np.sqrt(K), err
    assert torch.isnan(out[:, N:]).all()  # nothing written outside N
    assert (outb[:, :N].float() - ref).abs().max().item() < 0.02 * ref.abs().max().item() + 0.1
    for Me, Ke in GEMM_EDGE_CASES:
        _gemm_edge_case(ops, Me, 264, Ke, bn, a_mn, b_mn)


# (M, K): M sets the cluster size of launch_gemm (1, 2, 4 for 1, 2, 3-4 row blocks; 2 beyond), the K values the tails
GEMM_EDGE_CASES = [(100, 52),    # cluster 1
                   (200, 4100),  # cluster 2
                   (300, 1),     # cluster 4 with a zero-filled padding row block, K = 1 (a one-user batch's weight gradient)
                   (500, 500),   # cluster 4
                   (600, 52),    # cluster 2 with a padding block (dW_q1)
                   (1300, 500)]  # cluster 2, six groups, the last with a padding block


def _gemm_edge_case(ops, M, N, K, bn, a_mn, b_mn):
    """One GEMM shape through every epilogue path that stores fp32, per element against float64 (tests/helpers.py): plain store with
    the aux column diverted, split-K partials at split_stride with more splits than k blocks (the empty partials must store zeros, not
    leave the NaN they were filled with), split-K with atomics. Operand pitch padding holds NaN: TMA must never read it."""
    from helpers import TAU, TINY, gemm_ref, drop_last_kblock, assert_within, assert_detects
    g = torch.Generator(device="cuda").manual_seed(M * 7 + K + bn)
    A = torch.randn(M, K, device="cuda", generator=g).bfloat16()
    Bm = torch.randn(N, K, device="cuda", generator=g).bfloat16()

    def stored(X, mn):
        rows, cols = (X.shape[1], X.shape[0]) if mn else X.shape
        P = torch.full((rows, (cols + 7) // 8 * 8 + 8), float("nan"), device="cuda", dtype=torch.bfloat16)
        P[:, :cols] = X.t() if mn else X
        return P
    Ap, Bp = stored(A, a_mn), stored(Bm, b_mn)
    ref, mag = gemm_ref(A, Bm.t())
    bound = TAU * mag + TINY
    tag = "gemm M=%d N=%d K=%d bn=%d a_mn=%d b_mn=%d" % (M, N, K, bn, a_mn, b_mn)
    out = torch.full((M, N + 8), float("nan"), device="cuda")
    aux = torch.full((M,), float("nan"), device="cuda")
    ops.gemm(Ap, Bp, M, N, K, a_mn=a_mn, b_mn=b_mn, bn=bn, out_f32=out, aux_col=N - 1, aux_out=aux)
    kb = (K + 63) // 64
    splits = kb + 2
    parts = torch.full((splits, M, N + 8), float("nan"), device="cuda")
    ops.gemm(Ap, Bp, M, N, K, a_mn=a_mn, b_mn=b_mn, bn=bn, splits=splits, out_f32=parts, ld_f32=N + 8, split_stride=M * (N + 8))
    acc = torch.zeros(M, N + 8, device="cuda")
    ops.gemm(Ap, Bp, M, N, K, a_mn=a_mn, b_mn=b_mn, bn=bn, splits=3, atomic=True, out_f32=acc)
    torch.cuda.synchronize()
    assert_within(tag, out[:, :N - 1], ref[:, :N - 1], bound[:, :N - 1])
    assert_detects(tag + " minus last k block", out[:, :N - 1], drop_last_kblock(ref, A, Bm.t())[:, :N - 1], bound[:, :N - 1])
    assert_within(tag + " aux column", aux, ref[:, N - 1], bound[:, N - 1])
    assert torch.isnan(out[:, N - 1:]).all()   # the aux column and the pitch padding are not written
    per = (kb + splits - 1) // splits
    used = [s for s in range(splits) if s * per < kb]
    assert len(used) < splits
    for s in range(splits):
        if s not in used:
            assert (parts[s, :, :N] == 0).all(), "%s: empty split %d must store zeros" % (tag, s)
    assert torch.isnan(parts[:, :, N:]).all()
    got = parts[:, :, :N].double().sum(0)
    assert_within(tag + " split_stride", got, ref, bound)
    if len(used) > 1:
        assert_detects(tag + " without its last partial", got - parts[used[-1], :, :N].double(), ref, bound)
    assert_within(tag + " atomic split-K", acc[:, :N], ref, bound)
    assert (acc[:, N:] == 0).all()


def test_gemm_splitk_bias_act_aux(ops):
    torch.manual_seed(2)
    M, N, K = 300, 200, 4100
    A = (torch.randn(M, K, device="cuda") * 0.05).bfloat16()
    Bm = (torch.randn(N, K + 4, device="cuda") * 0.05).bfloat16()[:, :K]
    Bp = torch.zeros(N, K + 4, device="cuda", dtype=torch.bfloat16); Bp[:, :K] = Bm
    Ap = torch.zeros(M, K + 4, device="cuda", dtype=torch.bfloat16); Ap[:, :K] = A
    ref = A.float() @ Bm.float().t()
    out = torch.zeros(M, N, device="cuda")
    ops.gemm(Ap, Bp, M, N, K, splits=16, bn=128, out_f32=out, atomic=True, alpha=0.5)
    torch.cuda.synchronize()
    assert (out - 0.5 * ref).abs().max().item() < 5e-3
    # bias + tanh, bf16 out, aux column diverted
    bias = torch.randn(N, device="cuda")
    outb = torch.zeros(M, 208, device="cuda", dtype=torch.bfloat16)
    aux = torch.zeros(M, device="cuda")
    ops.gemm(Ap, Bp, M, N, K, bn=64, out_bf16=outb, bias=bias, act=1, aux_col=N - 1, aux_out=aux)
    torch.cuda.synchronize()
    want = torch.tanh(ref + bias)
    assert (outb[:, :N - 1].float() - want[:, :N - 1]).abs().max().item() < 1e-2
    assert (aux - want[:, N - 1]).abs().max().item() < 1e-2
    assert (outb[:, N - 1:] == 0).all()


def test_gemm_dropout_epilogue_bits(ops):
    torch.manual_seed(3)
    M, N, K = 260, 150, 128
    A = torch.randn(M, K, device="cuda").bfloat16()
    Bm = torch.randn(N, K, device="cuda").bfloat16()
    ref = torch.tanh(A.float() @ Bm.float().t())
    out = torch.zeros(M, 152, device="cuda")
    seed, step, keep = 0x1234567811, 7, 0.7
    step_dev = torch.tensor([3], dtype=torch.int32, device="cuda")
    ops.gemm(A, Bm, M, N, K, bn=128, out_f32=out, act=1, keep=keep, seed=seed, rng_stream=philox.STREAM_DISC_DROPOUT, rng_step=step,
             rng_step_dev=step_dev, rng_ld=152)
    torch.cuda.synchronize()
    mask = philox.hash_keep_mask(seed, philox.STREAM_DISC_DROPOUT, step + 3, M, N, 152, keep)
    assert abs(mask.mean() - keep) < 0.01
    got = out[:, :N].cpu().numpy()
    assert ((got != 0) == (mask & (ref.cpu().numpy() != 0))).all()  # RNG bits identical
    want = ref.cpu().numpy() * mask / np.float32(keep)
    assert np.abs(got - want).max() < 2e-2


# ----------------------------------------------------------------------------------------------------------------
# encoder gather, latent head, decoder statistics
# ----------------------------------------------------------------------------------------------------------------
def test_enc_gather_fwd_matches_oracle(ops):
    rng = np.random.RandomState(0)
    B, I = 37, 1000
    indptr, indices = rand_csr(rng, B, I, 20)
    indptr[-1]  # noqa
    # one long row to cross the 512-nnz chunk boundary
    W = (rng.randn(I, 600) * 0.05).astype(np.float32)
    b = (rng.randn(600) * 0.01).astype(np.float32)
    Wb = dev(W).bfloat16()
    seed, step, keep, uid0 = 42, 5, 0.75, 1000
    h1 = torch.zeros(B, 600, device="cuda", dtype=torch.bfloat16)
    coef = torch.zeros(len(indices), device="cuda")
    ops.enc_gather_fwd(dev(indptr), dev(indices), None, B, I, uid0, Wb, dev(b), keep, seed, step, None, h1, coef, int(np.diff(indptr).max()))
    torch.cuda.synchronize()
    X = np.zeros((B, I), dtype=np.float32)
    rows = np.repeat(np.arange(B), np.diff(indptr))
    X[rows, indices] = 1.0
    idx = (np.uint64(uid0) + np.arange(B, dtype=np.uint64))[:, None] * np.uint64(I) + np.arange(I, dtype=np.uint64)[None, :]
    mask = philox.keep_mask(seed, philox.STREAM_ENC_DROPOUT, step, idx, keep)
    params = [Wb.float().cpu(), None, None, None, torch.from_numpy(b)]
    Xt = torch.from_numpy(X)
    h = Xt * torch.rsqrt(torch.clamp((Xt * Xt).sum(1, keepdim=True), min=1e-12)) * torch.from_numpy(mask).float() / keep
    want = torch.tanh(h @ params[0] + params[4])
    assert (h1.float().cpu() - want).abs().max().item() < 1e-2
    # coefficients: exact mask bits, values to fp32 rounding
    want_coef = h.numpy()[rows, indices]
    got_coef = coef.cpu().numpy()
    assert ((got_coef != 0) == (want_coef != 0)).all()
    assert np.abs(got_coef - want_coef).max() < 1e-6


def test_enc_gather_long_row_and_values(ops):
    rng = np.random.RandomState(1)
    I = 3000
    n = 1300  # > 2 chunks of 512
    indices = np.sort(rng.choice(I, n, replace=False)).astype(np.int32)
    indptr = np.asarray([0, n, n, n + 0], dtype=np.int32)  # second and third rows empty
    vals = rng.randint(1, 3, size=n).astype(np.float32)
    W = (rng.randn(I, 600) * 0.05).astype(np.float32)
    Wb = dev(W).bfloat16()
    b = np.zeros(600, dtype=np.float32)
    h1 = torch.zeros(3, 600, device="cuda", dtype=torch.bfloat16)
    coef = torch.zeros(n, device="cuda")
    ws = torch.zeros(3, 600, device="cuda"); cn = torch.zeros(3, dtype=torch.int32, device="cuda")
    for _ in range(2):  # twice: the split-row workspace must come back zeroed
        ops.enc_gather_fwd(dev(indptr), dev(indices), dev(vals), 3, I, 0, Wb, dev(b), 1.0, 1, 0, None, h1, coef, n, ws, cn)
    torch.cuda.synchronize()
    assert ws.abs().max().item() == 0.0 and cn.abs().max().item() == 0
    x = np.zeros(I, dtype=np.float32); x[indices] = vals
    want = np.tanh((x / np.sqrt((x * x).sum())) @ Wb.float().cpu().numpy())
    assert np.abs(h1[0].float().cpu().numpy() - want).max() < 1e-2
    assert (h1[1:].float().abs().max().item()) == 0.0  # empty rows: tanh(0 + 0)
    # the same call over a host-built work list (one CTA per existing chunk instead of a rows x max-chunks grid)
    work = ops.enc_work_list(indptr)
    assert len(work) == 11 + 2 and sorted(int(w) & 0xFFFFF for w in work) == [0] * 11 + [1, 2]
    h1w = torch.full((3, 600), 7.0, device="cuda", dtype=torch.bfloat16)
    coefw = torch.zeros(n, device="cuda")
    ops.enc_gather_fwd(dev(indptr), dev(indices), dev(vals), 3, I, 0, Wb, dev(b), 1.0, 1, 0, None, h1w, coefw, n, ws, cn, work=dev(work))
    torch.cuda.synchronize()
    assert ws.abs().max().item() == 0.0 and cn.abs().max().item() == 0
    assert torch.equal(coefw, coef) and (h1w.float() - h1.float()).abs().max().item() < 4e-3   # (float atomics: order may differ)


def test_latent_fwd_bwd(ops):
    torch.manual_seed(5)
    B, L = 45, 200
    mulv = torch.randn(B, 2 * L, device="cuda") * 0.3
    eps = torch.randn(B, L, device="cuda")
    z = torch.zeros(B, L, device="cuda", dtype=torch.bfloat16)
    zmu = torch.zeros(B, L, device="cuda")
    scal = torch.zeros(16, device="cuda")
    ops.latent_fwd(mulv, eps, B, 0, 1.0, 0, 0, None, z, zmu, scal)
    torch.cuda.synchronize()
    mu, lv = mulv[:, :L], mulv[:, L:]
    kl = (0.5 * (-lv + lv.exp() + mu ** 2 - 1)).sum()
    assert abs(scal[0].item() - kl.item()) < 1e-3 * abs(kl.item())
    want_z = mu + eps * (0.5 * lv).exp()
    assert (z.float() - want_z).abs().max().item() < 2e-2
    assert (zmu - eps * (0.5 * lv).exp()).abs().max().item() < 1e-5
    # philox eps stream matches the numpy mirror
    ops.latent_fwd(mulv, None, B, 11, 1.0, 99, 4, None, z, zmu, scal)
    torch.cuda.synchronize()
    idx = (np.uint64(11) + np.arange(B, dtype=np.uint64))[:, None] * np.uint64(L) + np.arange(L, dtype=np.uint64)[None, :]
    e = philox.normal_eps(99, 4, idx)
    got_e = (zmu / (0.5 * lv).exp()).cpu().numpy()
    assert np.abs(got_e - e).max() < 1e-3
    # backward
    dz = torch.randn(B, L, device="cuda")
    dm = torch.zeros(B, 2 * L, device="cuda", dtype=torch.bfloat16)
    db = torch.zeros(2 * L, device="cuda")
    ops.latent_fwd(mulv, eps, B, 0, 1.0, 0, 0, None, z, zmu, scal)
    ops.latent_bwd(dz, mulv, zmu, B, B, 0.2, None, dm, db)
    torch.cuda.synchronize()
    mulv_r = mulv.clone().requires_grad_(True)
    mu_r, lv_r = mulv_r[:, :L], mulv_r[:, L:]
    loss = ((mu_r + eps * (0.5 * lv_r).exp()) * dz).sum() + 0.2 * (0.5 * (-lv_r + lv_r.exp() + mu_r ** 2 - 1)).sum(1).mean()
    g, = torch.autograd.grad(loss, mulv_r)
    assert (dm.float() - g).abs().max().item() < 2e-2
    assert (db - g.sum(0)).abs().max().item() < 5e-2


def test_decoder_logits_stats_and_dlogits(ops):
    torch.manual_seed(6)
    rng = np.random.RandomState(6)
    B, I = 70, 1203
    ld = 1208
    h2 = (torch.randn(B, 600, device="cuda") * 0.5).bfloat16()
    WdT = (torch.randn(I, 600, device="cuda") * 0.08).bfloat16()
    bd = torch.randn(I, device="cuda") * 0.1
    logits = torch.zeros(B, ld, device="cuda", dtype=torch.bfloat16)
    nblk = ops.dec_logits_nblk(B, I)
    assert 0 < nblk <= ops.dec_logits_nblk_max(I)
    partial = torch.zeros(nblk, B, 2, device="cuda")
    ops.dec_logits_fwd(h2, WdT, bd, B, I, logits, partial)
    ref = h2.float() @ WdT.float().t() + bd
    torch.cuda.synchronize()
    assert (logits[:, :I].float() - ref).abs().max().item() < 0.03 * ref.abs().max().item()
    indptr, indices = rand_csr(rng, B, I, 15)
    # sampled lists
    n_s = rng.randint(0, 6, size=B)
    samp_ptr = np.concatenate([[0], np.cumsum(n_s)]).astype(np.int32)
    samp_items = np.concatenate([np.sort(rng.choice(I, n, replace=False)) for n in n_s] + [np.zeros(0, dtype=np.int64)]).astype(np.int32)
    samp_valid = (rng.rand(len(samp_items)) < 0.8).astype(np.int32)
    lse = torch.zeros(B, device="cuda"); xw = torch.zeros(B, device="cuda"); su = torch.zeros(B, device="cuda")
    scal = torch.zeros(16, device="cuda")
    ops.dec_row_stats(partial, nblk, logits, B, dev(indptr), dev(indices), None, dev(samp_ptr), dev(samp_items), dev(samp_valid), lse, xw,
                      su, scal)
    torch.cuda.synchronize()
    want_lse = torch.logsumexp(ref, dim=1)
    assert (lse - want_lse).abs().max().item() < 2e-3
    X = torch.zeros(B, I); X[np.repeat(np.arange(B), np.diff(indptr)), indices] = 1.0
    lsm = torch.log_softmax(logits[:, :I].float().cpu(), dim=1)
    want_nll = -(lsm * X).sum().item()
    assert abs(scal[ops.S_NLL_SUM].item() - want_nll) < 1e-3 * abs(want_nll)
    probs = torch.softmax(logits[:, :I].float().cpu(), dim=1)
    m = torch.zeros(B, I)
    rows_s = np.repeat(np.arange(B), n_s)
    m[rows_s[samp_valid > 0], samp_items[samp_valid > 0]] = 1.0
    want_sp = (probs * m).sum().item()
    assert abs(scal[ops.S_SUM_P].item() - want_sp) < 2e-3 * abs(want_sp) + 1e-6
    # dlogits against autograd of the reference formula (on the stashed logits)
    lam = 1.0
    scal[ops.S_SUM_Y] = 3.3; scal[ops.S_CNT] = 7.0
    dl = torch.zeros(B, ld, device="cuda", dtype=torch.bfloat16)
    ops.dec_dlogits(logits, lse, xw, su, B, I, B, lam, scal, dev(indptr), dev(indices), None, dev(samp_ptr), dev(samp_items),
                    dev(samp_valid), dl)
    torch.cuda.synchronize()
    lg = logits[:, :I].float().cpu().requires_grad_(True)
    ls = torch.log_softmax(lg, dim=1)
    pr = torch.softmax(lg, dim=1)
    loss = -(ls * X).sum(1).mean() - lam * (3.3 / 7.0) * (pr * m).sum()
    g, = torch.autograd.grad(loss, lg)
    err = (dl[:, :I].float().cpu() - g).abs().max().item()
    assert err < 1e-2 * g.abs().max().item() + 1e-6, err
    assert (dl[:, I:] == 0).all()
    # fused per-user kernel (G step): same statistics and the same dlogits in one launch
    scal2 = torch.zeros(16, device="cuda"); scal2[ops.S_SUM_Y] = 3.3; scal2[ops.S_CNT] = 7.0
    lse2 = torch.zeros(B, device="cuda"); dl2 = torch.full((B, ld), 9.0, device="cuda", dtype=torch.bfloat16)
    ops.dec_row_bwd(partial, nblk, logits, B, I, B, lam, dev(indptr), dev(indices), None, dev(samp_ptr), dev(samp_items), dev(samp_valid),
                    lse2, scal2, dl2)
    torch.cuda.synchronize()
    assert (lse2 - lse).abs().max().item() < 1e-5
    assert abs(scal2[ops.S_NLL_SUM].item() - want_nll) < 1e-3 * abs(want_nll)
    assert abs(scal2[ops.S_SUM_P].item() - want_sp) < 2e-3 * abs(want_sp) + 1e-6
    assert (dl2.float() - dl.float()).abs().max().item() <= 2e-2 * g.abs().max().item()
    assert (dl2[:, :I].float().cpu() - g).abs().max().item() < 1e-2 * g.abs().max().item() + 1e-6
    # probabilities (compat path)
    out = torch.zeros(B, I, device="cuda")
    ops.dec_probs(logits, lse, B, I, out)
    torch.cuda.synchronize()
    assert (out.cpu() - probs).abs().max().item() < 1e-3 * probs.max().item() + 1e-7


# ----------------------------------------------------------------------------------------------------------------
# Adam, encoder sparse gradient
# ----------------------------------------------------------------------------------------------------------------
def test_adam_matches_tf_formula(ops):
    torch.manual_seed(7)
    n = 600 * 37 + 3
    p = torch.randn(n, device="cuda"); m = torch.randn(n, device="cuda") * 0.01; v = torch.rand(n, device="cuda") * 1e-4
    g = torch.randn(n, device="cuda") * 0.1
    p0, m0, v0 = p.cpu().clone(), m.cpu().clone(), v.cpu().clone()
    sh = torch.zeros(n + 5, device="cuda", dtype=torch.bfloat16)[:n]
    lr_t = orc.tf_adam_lr_t(1e-4, 17)
    ops.adam(p, m, v, g, sh, lr_t=lr_t)
    torch.cuda.synchronize()
    orc.tf_adam_step(p0, m0, v0, g.cpu(), lr_t)
    assert (p.cpu() - p0).abs().max().item() < 1e-6
    assert (m.cpu() - m0).abs().max().item() < 1e-7
    assert (v.cpu() - v0).abs().max().item() < 1e-8
    assert (sh.float().cpu() - p0).abs().max().item() < 2e-2
    # lr_t from the device step state
    words = torch.zeros(4, dtype=torch.int32, device="cuda"); scal = torch.zeros(16, device="cuda")
    for _ in range(3):
        ops.step_advance(words, scal, 2, 1e-4)
    torch.cuda.synchronize()
    assert words.cpu().tolist()[:3] == [3, 3, 3]
    assert abs(scal[ops.S_LR_T].item() - orc.tf_adam_lr_t(1e-4, 3)) < 1e-10
    assert abs(scal[ops.S_ANNEAL].item() - orc.anneal_value(2)) < 1e-9


@pytest.mark.parametrize("n_partials", [2, 5, 16, 17, 33, 34])
def test_adam_over_split_k_partials(ops, n_partials):
    """ltg_adam whose gradient is a sum of split-K partials (the discriminator update): the one-round kernel (<= 33 partials: eight
    warps x four partials per 32 float4, folded through shared memory) and the loop over rounds (34) against TF-Adam on the fp64
    sum of the partials; n % 4 != 0 exercises the scalar tail."""
    torch.manual_seed(20 + n_partials)
    n = 161001                      # the discriminator's parameter count (SURVEY a11): 161001 % 4 == 1
    stride = (n + 3) // 4 * 4 + 8
    p = torch.randn(n, device="cuda"); m = torch.randn(n, device="cuda") * 0.01; v = torch.rand(n, device="cuda") * 1e-4
    gp = torch.randn(n_partials, stride, device="cuda") * 0.1
    p0, m0, v0 = p.cpu().clone(), m.cpu().clone(), v.cpu().clone()
    sh = torch.zeros(stride, device="cuda", dtype=torch.bfloat16)[:n]
    lr_t = orc.tf_adam_lr_t(1e-4, 5)
    ops.adam(p, m, v, gp, sh, lr_t=lr_t, n_partials=n_partials, partial_stride=stride)
    torch.cuda.synchronize()
    g = gp[:, :n].double().sum(0).float().cpu()
    orc.tf_adam_step(p0, m0, v0, g, lr_t)
    # fp32 summation order of up to 34 terms with |sum| up to ~2.5: |g error| <~ 1e-5, so (1 - b1) dg ~ 1e-6 and (1 - b2) 2 g dg ~ 1e-7
    assert (m.cpu() - m0).abs().max().item() < 3e-6
    assert (v.cpu() - v0).abs().max().item() < 5e-7
    assert (p.cpu() - p0).abs().max().item() < 1e-5
    assert (sh.float().cpu() - p0).abs().max().item() < 2e-2


def test_enc_wgrad_and_enc_adam(ops):
    rng = np.random.RandomState(8)
    B, I = 50, 400
    indptr, indices = rand_csr(rng, B, I, 12)
    indices[: indptr[1]] = np.sort(rng.choice(I, indptr[1], replace=False))
    nnz = len(indices)
    coef = (rng.rand(nnz).astype(np.float32)) * (rng.rand(nnz) < 0.75)
    dh1 = rng.randn(B, 600).astype(np.float32)
    rows = np.repeat(np.arange(B), np.diff(indptr))
    order = np.lexsort((rows, indices))
    active, counts = np.unique(indices, return_counts=True)
    act_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    slot = np.full(I, -1, dtype=np.int32); slot[active] = np.arange(len(active))
    csc_row = rows[order].astype(np.int32); csc_pos = order.astype(np.int32)
    G = torch.full((len(active), 600), float("nan"), device="cuda")
    ops.enc_wgrad_compact(G, len(active), dev(act_ptr), dev(csc_row), dev(csc_pos), dev(coef), dev(dh1))
    dW = torch.full((I, 600), float("nan"), device="cuda")
    ops.enc_wgrad_expand(dW, I, dev(slot), G)
    torch.cuda.synchronize()
    Xc = np.zeros((B, I), dtype=np.float32); Xc[rows, indices] = coef
    want = Xc.T @ dh1
    assert np.abs(dW.cpu().numpy() - want).max() < 1e-4
    p = torch.randn(I, 600, device="cuda"); m = torch.zeros(I, 600, device="cuda"); v = torch.rand(I, 600, device="cuda") * 1e-2 + 1e-3
    m += 0.01  # rows without gradient must still move (dense Adam, F7)
    p0, m0, v0 = p.cpu().clone(), m.cpu().clone(), v.cpu().clone()
    p_init = p.cpu().clone()
    sh = torch.zeros(I, 600, device="cuda", dtype=torch.bfloat16)
    ops.enc_adam(p, m, v, sh, I, dev(slot), G, lr_t=1e-3)
    torch.cuda.synchronize()
    orc.tf_adam_step(p0, m0, v0, torch.from_numpy(want), 1e-3)
    assert (p.cpu() - p0).abs().max().item() < 1e-5
    assert (sh.float().cpu() - p0).abs().max().item() < 2e-2
    untouched = slot < 0
    assert untouched.any() and (p.cpu()[untouched] != p_init[untouched]).all()


# ----------------------------------------------------------------------------------------------------------------
# sampler
# ----------------------------------------------------------------------------------------------------------------
def _sampler_inputs(rng, B, I, ld):
    logits = (rng.randn(B, ld) * 1.5).astype(np.float32)
    niche = np.arange(I // 10, I)  # 90% of the catalog is "niche"
    cand, n_s, pops = [], [], []
    for u in range(B):
        n = int(rng.randint(0, 12)) if u % 7 else 0
        own = np.sort(rng.choice(niche, n, replace=False))
        others = np.setdiff1d(niche, own)
        extra = rng.choice(others, max(2 * n, 10 - n), replace=False)
        cand.append(np.sort(np.concatenate([own, extra])).astype(np.int32))
        n_s.append(n)
        pops.append(rng.choice(I // 10, size=rng.randint(1, 8), replace=False).astype(np.int32))
    return logits, cand, np.asarray(n_s), pops


def test_sampler_matches_gumbel_topk_oracle_bit_exact(ops):
    rng = np.random.RandomState(9)
    B, I, ld = 64, 1000, 1000
    logits, cand, n_s, pops = _sampler_inputs(rng, B, I, ld)
    lg = dev(logits).bfloat16()
    cand_ptr = np.concatenate([[0], np.cumsum([len(c) for c in cand])]).astype(np.int32)
    samp_ptr = np.concatenate([[0], np.cumsum(n_s)]).astype(np.int32)
    pop_ptr = np.concatenate([[0], np.cumsum([len(p) for p in pops])]).astype(np.int32)
    valid = np.ones(I, dtype=np.uint8); valid[[418, 447, 595]] = 0
    K = int(samp_ptr[-1])
    si = torch.full((K,), -7, dtype=torch.int32, device="cuda"); sp = torch.full((K,), -7, dtype=torch.int32, device="cuda")
    sv = torch.full((K,), -7, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    seed, step, uid0 = 777, 3, 500
    ops.sample_pairs(lg, B, I, uid0, dev(cand_ptr), dev(np.concatenate(cand)), dev(samp_ptr), dev(pop_ptr), dev(np.concatenate(pops)),
                     dev(valid), seed, step, None, si, sp, sv, cnt, int(max(len(c) for c in cand)),
                     dev(np.argsort(-np.diff(cand_ptr)).astype(np.int32)))
    torch.cuda.synchronize()
    si, sp, sv = si.cpu().numpy(), sp.cpu().numpy(), sv.cpu().numpy()
    lgf = lg.float().cpu().numpy()
    nvalid = 0
    for u in range(B):
        s0, s1 = samp_ptr[u], samp_ptr[u + 1]
        if s1 == s0:
            continue
        idx = np.uint64(uid0 + u) * np.uint64(I) + cand[u].astype(np.uint64)
        # device computes -log(-log(u)) with fast intrinsics; compare sets, allowing only near-ties to differ
        want = orc.gumbel_topk_sample(cand[u], lgf[u], n_s[u], philox.gumbel(seed, step, idx))
        got = si[s0:s1]
        assert (np.diff(got) > 0).all()
        if not np.array_equal(got, want):
            keys = lgf[u][cand[u]] + philox.gumbel(seed, step, idx)
            kth = np.sort(keys)[::-1][n_s[u] - 1:n_s[u] + 1]
            assert abs(kth[0] - kth[1]) < 1e-4, (u, got, want)
        r = philox.rand_u32(seed, philox.STREAM_PARTNER, step, np.uint64(uid0 + u) * np.uint64(I) + got.astype(np.uint64))
        want_p = pops[u][((r.astype(np.uint64) * np.uint64(len(pops[u]))) >> np.uint64(32)).astype(np.int64)]
        assert np.array_equal(sp[s0:s1], want_p)
        want_v = (valid[got] & valid[want_p]).astype(np.int32)
        assert np.array_equal(sv[s0:s1], np.where(want_v > 0, 1, -1))
        nvalid += int(want_v.sum())
    assert cnt.item() == nvalid


def test_sampler_distribution_chi_square(ops):
    """Distributional parity with sample.py:54 (np.random.choice without replacement): per-item inclusion counts of the
    device sampler vs the oracle's restatement over many draws (chi-square, alpha = 1e-3)."""
    from scipy import stats
    rng = np.random.RandomState(10)
    I = 64
    cand = np.sort(rng.choice(np.arange(8, I), 9, replace=False)).astype(np.int32)
    n_draw = 3
    logit_row = (rng.randn(I) * 1.2).astype(np.float32)
    R = 20000  # users all sharing the same candidate set / logits, distinct RNG keys
    lg = dev(np.tile(logit_row, (R, 1))).bfloat16()
    cand_ptr = (np.arange(R + 1) * len(cand)).astype(np.int32)
    samp_ptr = (np.arange(R + 1) * n_draw).astype(np.int32)
    pop_ptr = np.arange(R + 1).astype(np.int32)
    si = torch.zeros(R * n_draw, dtype=torch.int32, device="cuda"); sp = torch.zeros_like(si); sv = torch.zeros_like(si)
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.sample_pairs(lg, R, I, 0, dev(cand_ptr), dev(np.tile(cand, R)), dev(samp_ptr), dev(pop_ptr), dev(np.zeros(R, dtype=np.int32)),
                     dev(np.ones(I, dtype=np.uint8)), 2024, 1, None, si, sp, sv, cnt, len(cand))
    torch.cuda.synchronize()
    got = np.bincount(si.cpu().numpy(), minlength=I)[cand]
    p = np.exp(lg[0].float().cpu().numpy()[cand].astype(np.float64)); p /= p.sum()
    ref_rng = np.random.RandomState(11)
    ref = np.zeros(I, dtype=np.int64)
    for _ in range(R):
        _, ids = orc.sample_from_generator_new(cand, p, n_draw, I, ref_rng)
        ref[ids] += 1
    ref = ref[cand]
    chi2, pval, _, _ = stats.chi2_contingency(np.stack([got, ref]))
    assert pval > 1e-3, (pval, got, ref)


# ----------------------------------------------------------------------------------------------------------------
# top-k metrics
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,I", [("f32", 2500), ("bf16", 2500), ("f32", 20108), ("bf16", 20108), ("f32", 333)])
def test_topk_metrics_exact(ops, dtype, I):
    """Exact top-k index lists (ties: lowest index first), DCG and hit counts against NumPy. The rows cover both selection paths of
    the staged kernel: the candidate pre-filter (random rows; rows with a few hundred ties at the threshold) and its full-row path
    (a fully tied row and a row with half the catalog tied at the top overflow the 2,048-entry candidate list)."""
    from scipy import sparse
    rng = np.random.RandomState(12)
    n, k = 57, 100
    scores = rng.randn(n, I).astype(np.float32)
    scores[3, :] = 0.25           # a fully tied row
    scores[4, ::2] = 1.0          # half the row tied at the top
    scores[5, 7::40] = 5.0        # a few ties above everything else, fewer than k for small catalogs
    scores[6, :] = np.round(scores[6, :] * 4) / 4    # a coarse grid: hundreds of ties at every level, also at the threshold
    scores[7, :] = -np.abs(scores[7, :])             # all negative
    t = dev(scores)
    if dtype == "bf16":
        t = t.bfloat16()
        scores = t.float().cpu().numpy()
    seen_ptr, seen_items = rand_csr(rng, n, I, 30)
    held_ptr, held_items = rand_csr(rng, n, I, 10, min_nnz=0)
    topk = torch.zeros(n, k, dtype=torch.int32, device="cuda")
    dcg = torch.zeros(n, dtype=torch.float64, device="cuda")
    hits = torch.zeros(n, 2, dtype=torch.int32, device="cuda")
    ops.topk_metrics(t, n, I, dev(seen_ptr), dev(seen_items), dev(held_ptr), dev(held_items), k, [20, 50], topk, dcg, hits)
    torch.cuda.synchronize()
    masked = scores.copy()
    masked[np.repeat(np.arange(n), np.diff(seen_ptr)), seen_items] = -np.inf
    want = orc.topk_indices(masked, k)
    assert np.array_equal(topk.cpu().numpy(), want)  # bit-exact index lists (ties: lowest index first)
    held = sparse.csr_matrix((np.ones(len(held_items)), held_items, held_ptr), shape=(n, I))
    tp = 1.0 / np.log2(np.arange(2, k + 2))
    want_dcg = (held[np.arange(n)[:, None], want].toarray() * tp).sum(1)
    assert np.abs(dcg.cpu().numpy() - want_dcg).max() < 1e-12
    for j, kk in enumerate((20, 50)):
        want_hits = held[np.arange(n)[:, None], want[:, :kk]].toarray().sum(1)
        assert np.array_equal(hits.cpu().numpy()[:, j], want_hits.astype(np.int32))


# ----------------------------------------------------------------------------------------------------------------
# discriminator pieces
# ----------------------------------------------------------------------------------------------------------------
def test_disc_gather_head_and_backward(ops):
    torch.manual_seed(13)
    I, P, h3, ld = 500, 333, 300, 304
    E = torch.zeros(I, 128, device="cuda", dtype=torch.bfloat16); E[:, :100] = (torch.randn(I, 100, device="cuda") * 0.1).bfloat16()
    pop = torch.randint(0, I, (P,), dtype=torch.int32, device="cuda"); niche = torch.randint(0, I, (P,), dtype=torch.int32, device="cuda")
    Xp = torch.zeros(P, 128, device="cuda", dtype=torch.bfloat16); Xn = torch.zeros_like(Xp)
    ops.disc_gather(E, pop, niche, P, Xp, Xn)
    torch.cuda.synchronize()
    assert torch.equal(Xp, E[pop.long()]) and torch.equal(Xn, E[niche.long()])
    keep = 0.7
    t3 = torch.tanh(torch.randn(P, h3, device="cuda"))
    mask = (torch.rand(P, h3, device="cuda") < keep)
    Y3 = torch.zeros(P, ld, device="cuda", dtype=torch.bfloat16); Y3[:, :h3] = (t3 * mask / keep).bfloat16()
    w4 = torch.randn(h3, device="cuda") * 0.1; b4 = torch.tensor([0.05], device="cuda")
    label = torch.randint(-1, 2, (P,), dtype=torch.int32, device="cuda")
    y = torch.zeros(P, device="cuda"); scal = torch.zeros(16, device="cuda")
    dz3 = torch.full((P, ld), 7.0, device="cuda", dtype=torch.bfloat16); dz3[:, h3:] = 0
    dw4 = torch.zeros(h3, device="cuda"); db4 = torch.zeros(1, device="cuda")
    ops.disc_head(Y3, P, h3, w4, b4, label, keep, y, scal, dz3, dw4, db4)
    torch.cuda.synchronize()
    Yf = Y3[:, :h3].float()
    a = Yf.clone().requires_grad_(True); w4r = w4.clone().requires_grad_(True); b4r = b4.clone().requires_grad_(True)
    yr = torch.sigmoid(a @ w4r + b4r)
    real, gen = label == 0, label == 1
    loss = -torch.log(yr[real]).sum() - torch.log(1 - yr[gen]).sum()
    ga, gw, gb = torch.autograd.grad(loss, [a, w4r, b4r])
    assert (y - yr).abs().max().item() < 1e-5
    assert abs(scal[ops.S_D_LOSS].item() - loss.item()) < 1e-3 * abs(loss.item())
    assert abs(scal[ops.S_SUM_Y].item() - yr[gen].sum().item()) < 1e-3
    assert abs(db4.item() - gb.item()) < 1e-3
    assert scal[ops.S_CNT].item() == int(gen.sum().item())
    assert (dw4 - gw).abs().max().item() < 1e-3
    dact = torch.where(Yf != 0, (1 - (Yf * keep) ** 2) / keep, torch.zeros_like(Yf))
    want_dz3 = ga * dact
    assert (dz3[:, :h3].float() - want_dz3).abs().max().item() < 1e-2 * want_dz3.abs().max().item() + 1e-6
    assert (dz3[label.long() < 0][:, :h3] == 0).all()
    # backward through a dropout(tanh) layer, fused into the dgrad GEMM epilogue: dz = (dz3 W^T) * dact(Hact)
    K3 = 408
    W = (torch.randn(K3, ld, device="cuda") * 0.1).bfloat16(); W[:, h3:] = 0
    Hact = torch.zeros(P, K3, device="cuda", dtype=torch.bfloat16)
    t = torch.tanh(torch.randn(P, K3, device="cuda")); mk = torch.rand(P, K3, device="cuda") < keep
    Hact[:] = (t * mk / keep).bfloat16()
    dz = torch.zeros(P, K3, device="cuda", dtype=torch.bfloat16)
    ops.gemm(dz3, W, P, K3, h3, bn=256, out_bf16=dz, dact_src=Hact, dact_keep=keep)
    torch.cuda.synchronize()
    Hf = Hact.float()
    dact2 = torch.where(Hf != 0, (1 - (Hf * keep) ** 2) / keep, torch.zeros_like(Hf))
    want = (dz3[:, :h3].float() @ W[:, :h3].float().t()) * dact2
    assert (dz.float() - want).abs().max().item() < 2e-2 * want.abs().max().item() + 1e-6


@pytest.mark.parametrize("P,backward,sizes", [(333, True, (100, 150, 250, 300)), (1000, False, (100, 150, 250, 300)), (128, True, (100, 150, 250, 300)),
                                              (260, True, (40, 24, 56, 64)), (40000, True, (100, 150, 250, 300)), (40000, False, (100, 150, 250, 300))])
def test_disc_fused_forward_matches_unfused_chain(ops, P, backward, sizes):
    """disc_fused.cu (one tcgen05 kernel: branch layers -> fc1 -> head through TMEM / shared memory) against the chain of
    ltg_gemm_bf16 + ltg_disc_head launches it replaces. The dropout masks are the same counter hash, so the hidden activation
    must agree to bf16 rounding of tanh.approx inputs (accumulation order differs inside the tensor core only by k-block order:
    identical here), y / loss / gradients within 1e-3."""
    disc_mod = importlib.import_module("long-tail-gan_b200.discriminator")
    h0, h1, h2, h3 = sizes
    I = 700
    d = disc_mod.Discriminator(I, I, h0, h1, h2, h3, device="cuda", seed=5)
    assert ops.disc_fused_supported(d)
    with torch.no_grad():   # make the head weights and biases non-trivial
        prm = d.get_params()
        g = torch.Generator(device="cuda").manual_seed(3)
        prm = [p + 0.05 * torch.randn(p.shape, device="cuda", generator=g) for p in prm]
        d.set_params(d.E, prm)
    pop = torch.randint(0, I, (P,), dtype=torch.int32, device="cuda"); niche = torch.randint(0, I, (P,), dtype=torch.int32, device="cuda")
    label = torch.randint(-1, 2, (P,), dtype=torch.int32, device="cuda")
    bf = dict(device="cuda", dtype=torch.bfloat16)
    Xp = torch.zeros(P, 128, **bf); Xn = torch.zeros(P, 128, **bf)
    ops.disc_gather(d.E_b, pop, niche, P, Xp, Xn)
    words = torch.tensor([7, 0, 0, 0], dtype=torch.int32, device="cuda")
    keep, seed, st = 0.7, 1234, ops.STREAM_DISC_DROPOUT
    k1 = d.h0 + 1

    def run(fused):
        Hd = torch.zeros(P, d.k3, **bf); Hd[:, d.one3] = 1.0
        y = torch.zeros(P, device="cuda"); scal = torch.zeros(16, device="cuda")
        dz3 = torch.zeros(P, d.ld3, **bf) if backward else None
        dw4 = torch.zeros(d.ld3, device="cuda") if backward else None
        db4 = torch.zeros(4, device="cuda") if backward else None
        dz12 = torch.zeros(P, d.k3, **bf) if backward else None
        if fused:
            ops.disc_fwd_fused(Xp, Xn, P, d, label, keep, seed, st, words, Hd, y, scal, dz3, dw4, db4, dz12)
        else:
            Y3 = torch.zeros(P, d.ld3, **bf)
            ops.gemm(Xp, d.view("W1", "b"), P, d.h1, k1, lda=128, b_mn=True, bn=ops.pick_bn(P, d.h1), out_bf16=Hd, ld_bf16=d.k3, act=1,
                     keep=keep, seed=seed, rng_stream=st, rng_step_dev=words, rng_ld=d.ld1)
            ops.gemm(Xn, d.view("W2", "b"), P, d.h2, k1, lda=128, b_mn=True, bn=ops.pick_bn(P, d.h2), out_bf16=Hd[:, d.off2:], ld_bf16=d.k3,
                     act=1, keep=keep, seed=seed, rng_stream=st + 1, rng_step_dev=words, rng_ld=d.ld2)
            ops.gemm(Hd, d.view("W3", "b"), P, d.h3, d.k3, b_mn=True, bn=ops.pick_bn(P, d.h3), out_bf16=Y3, act=1, keep=keep, seed=seed,
                     rng_stream=st + 2, rng_step_dev=words, rng_ld=d.ld3)
            ops.disc_head(Y3, P, d.h3, d.view("w4"), d.view("b4"), label, keep, y, scal, dz3, dw4, db4)
            if backward:   # the backward GEMM the fused kernel's fourth MMA replaces
                ops.gemm(dz3, d.view("W3", "b"), P, d.k3, d.h3, bn=ops.pick_bn(P, d.k3), out_bf16=dz12, dact_src=Hd, dact_keep=keep)
        torch.cuda.synchronize()
        return Hd, y, scal, dz3, dw4, db4, dz12

    Hu, yu, su, dzu, dwu, dbu, d12u = run(False)
    Hf, yf, sf, dzf, dwf, dbf, d12f = run(True)
    # same dropout pattern and the ones column / padding layout
    assert torch.equal(Hu == 0, Hf == 0)
    assert (Hf[:, d.one3] == 1).all() and (Hf[:, d.one3 + 1:] == 0).all() and (Hf[:, d.h1:d.off2] == 0).all()
    assert (Hu.float() - Hf.float()).abs().max().item() <= 2e-2     # one bf16 ulp at |x| <= 1.43 (= 1/keep)
    assert (Hu.float() - Hf.float()).abs().mean().item() < 1e-4
    assert (yu - yf).abs().max().item() < 2e-3
    for slot in (ops.S_D_LOSS, ops.S_SUM_Y):
        assert abs(su[slot].item() - sf[slot].item()) < 1e-3 * max(1.0, abs(su[slot].item()))
    assert su[ops.S_CNT].item() == sf[ops.S_CNT].item() == int((label == 1).sum().item())
    if backward:
        scale = dzu.float().abs().max().item() + 1e-9
        assert (dzu.float() - dzf.float()).abs().max().item() < 3e-2 * scale
        assert (dzf[label.long() < 0] == 0).all()
        assert (dwu - dwf).abs().max().item() < 2e-3 * max(1.0, dwu.abs().max().item())
        assert abs(dbu[0].item() - dbf[0].item()) < 1e-3 * max(1.0, abs(dbu[0].item()))
        # dz12 = (dz3 W3^T) * dact(Hd): fused fourth MMA against the GEMM path, and against fp32 on the fused kernel's own dz3 / Hd
        used = list(range(d.h1)) + list(range(d.off2, d.off2 + d.h2))   # the columns the weight-gradient GEMMs read
        s12 = d12u.float()[:, used].abs().max().item() + 1e-9
        assert (d12u.float()[:, used] - d12f.float()[:, used]).abs().max().item() < 4e-2 * s12
        Hff = Hf.float()
        dact = torch.where(Hff != 0, (1 - (Hff * keep) ** 2) / keep, torch.zeros_like(Hff))
        want = (dzf[:, : d.h3].float() @ d.view("W3", "b").float()[:, : d.h3].t()) * dact
        assert (d12f.float()[:, used] - want[:, used]).abs().max().item() < 2e-2 * want[:, used].abs().max().item() + 1e-7
    # independent fp32 restatement of the head on the fused kernel's own hidden activation
    W3 = d.view("W3", "b").float()[:, : d.h3]
    a3 = torch.tanh(Hf.float() @ W3)
    y3 = torch.where(torch.from_numpy(philox.hash_keep_mask(seed, st + 2, 7, P, d.h3, d.ld3, keep)).cuda(), a3 / keep, torch.zeros_like(a3))
    yr = torch.sigmoid(y3.bfloat16().float() @ d.view("w4")[: d.h3] + d.view("b4")[0])
    assert (yr - yf).abs().max().item() < 5e-3


@pytest.mark.parametrize("P,Pr", [(1000, 333), (40000, 19001), (300, 128)])
def test_disc_fused_row_slices_equal_one_launch(ops, P, Pr):
    """ltg_disc_fwd_fused over rows [0, Pr) and [Pr, P) of a pair batch (pointers advanced, rng_row0 = first row) against ONE launch
    over all P rows: every per-row output (hidden activation with its dropout pattern, y, dz3) bit-identical -- a row's result does not
    depend on which 128-row tile it sits in --, the atomically accumulated sums equal up to summation order. This is what lets
    engine.run_step run the real pairs' half of the D forward beside phase A."""
    disc_mod = importlib.import_module("long-tail-gan_b200.discriminator")
    I = 700
    d = disc_mod.Discriminator(I, I, 100, 150, 250, 300, device="cuda", seed=5)
    with torch.no_grad():
        g = torch.Generator(device="cuda").manual_seed(3)
        d.set_params(d.E, [p + 0.05 * torch.randn(p.shape, device="cuda", generator=g) for p in d.get_params()])
    pop = torch.randint(0, I, (P,), dtype=torch.int32, device="cuda"); niche = torch.randint(0, I, (P,), dtype=torch.int32, device="cuda")
    label = torch.randint(-1, 2, (P,), dtype=torch.int32, device="cuda")
    bf = dict(device="cuda", dtype=torch.bfloat16)
    Xp = torch.zeros(P, 128, **bf); Xn = torch.zeros(P, 128, **bf)
    ops.disc_gather(d.E_b, pop, niche, P, Xp, Xn)
    words = torch.tensor([11, 0, 0, 0], dtype=torch.int32, device="cuda")
    keep, seed, st = 0.7, 99, ops.STREAM_DISC_DROPOUT

    def run(slices):
        Hd = torch.zeros(P, d.k3, **bf); y = torch.zeros(P, device="cuda"); scal = torch.zeros(16, device="cuda")
        dz3 = torch.zeros(P, d.ld3, **bf); dw4 = torch.zeros(d.ld3, device="cuda"); db4 = torch.zeros(4, device="cuda")
        for r0, r1 in slices:
            ops.disc_fwd_fused(Xp[r0:], Xn[r0:], r1 - r0, d, label[r0:], keep, seed, st, words, Hd[r0:], y[r0:], scal, dz3[r0:], dw4, db4, None,
                               rng_row0=r0)
        torch.cuda.synchronize()
        return Hd, y, scal, dz3, dw4, db4

    one = run([(0, P)])
    two = run([(0, Pr), (Pr, P)])
    assert (one[0] != 0).any() and (one[0] == 0).float().mean().item() > 0.2     # dropout is on
    assert torch.equal(one[0], two[0]) and torch.equal(one[1], two[1]) and torch.equal(one[3], two[3])
    for slot in (ops.S_D_LOSS, ops.S_SUM_Y):
        assert abs(one[2][slot].item() - two[2][slot].item()) < 1e-4 * max(1.0, abs(one[2][slot].item()))
    assert one[2][ops.S_CNT].item() == two[2][ops.S_CNT].item()
    assert (one[4] - two[4]).abs().max().item() < 1e-3 * max(1.0, one[4].abs().max().item())
    assert abs(one[5][0].item() - two[5][0].item()) < 1e-3 * max(1.0, abs(one[5][0].item()))
    # and without the row offset the second slice would draw different masks (the test can see the difference)
    Hd_wrong = torch.zeros(P, d.k3, **bf)
    ops.disc_fwd_fused(Xp[Pr:], Xn[Pr:], P - Pr, d, label[Pr:], keep, seed, st, words, Hd_wrong[Pr:], torch.zeros(P, device="cuda"),
                       torch.zeros(16, device="cuda"), rng_row0=0)
    torch.cuda.synchronize()
    assert not torch.equal(Hd_wrong[Pr:] == 0, one[0][Pr:] == 0)


def test_peer_exchange_kernels_on_one_device(ops):
    """peer_kernels.cu with pointer tables whose entries all live on this GPU (a table entry is just an address, so two "ranks"
    can be two local buffers): the pull-sum, the push, the Adam with fused reduce-scatter / all-gather, and the flag barrier with
    world = 1. The real 2-GPU check over NVLink is tools/dp_check.py."""
    torch.manual_seed(3)
    n = 600 * 37
    off = 600 * 5
    g0 = torch.randn(off + n + 8, device="cuda"); g1 = torch.randn(off + n + 8, device="cuda")
    tab_g = ops.peer_table([g0.data_ptr(), g1.data_ptr()])
    out = torch.zeros(n + 3, device="cuda")
    ops.peer_reduce(tab_g, off, n + 3, 2, out)
    torch.cuda.synchronize()
    assert torch.equal(out, g0[off: off + n + 3] + g1[off: off + n + 3])
    # Adam over the shard [off, off+n): gradient = g0 + g1 rows, bf16 result into both "ranks'" shadows; equals ltg_adam on the sum
    p = torch.randn(n, device="cuda"); m = torch.randn(n, device="cuda") * 0.01; v = torch.rand(n, device="cuda") * 1e-3
    p2, m2, v2 = p.clone(), m.clone(), v.clone()
    sh0 = torch.zeros(off + n, device="cuda", dtype=torch.bfloat16); sh1 = torch.zeros_like(sh0)
    ref_sh = torch.zeros(n, device="cuda", dtype=torch.bfloat16)
    scal = torch.zeros(16, device="cuda")
    ops.adam_peer(p, m, v, tab_g, ops.peer_table([sh0.data_ptr(), sh1.data_ptr()]), off, 2, lr_t=1e-3, scal=scal)
    ops.adam(p2, m2, v2, (g0 + g1)[off: off + n].contiguous(), ref_sh, lr_t=1e-3, scal=scal)
    torch.cuda.synchronize()
    assert torch.equal(p, p2) and torch.equal(m, m2) and torch.equal(v, v2)
    assert torch.equal(sh0[off:], ref_sh) and torch.equal(sh1[off:], ref_sh) and (sh0[:off] == 0).all()
    # encoder variant: compact gradient rows through slot_of_item, bf16 rows into both shadows
    items, H = 37, 600
    slot = torch.full((items,), -1, dtype=torch.int32, device="cuda"); slot[::3] = torch.arange(len(slot[::3]), dtype=torch.int32, device="cuda")
    G = torch.randn(int((slot >= 0).sum()), H, device="cuda")
    p = torch.randn(items, H, device="cuda"); m = torch.zeros_like(p); v = torch.zeros_like(p)
    p2, m2, v2 = p.clone(), m.clone(), v.clone()
    sh0.zero_(); sh1.zero_(); ref2 = torch.zeros(items, H, device="cuda", dtype=torch.bfloat16)
    ops.enc_adam_peer(p, m, v, ops.peer_table([sh0.data_ptr(), sh1.data_ptr()]), off, items, slot, G, 2, lr_t=1e-3, scal=scal)
    ops.enc_adam(p2, m2, v2, ref2, items, slot, G, lr_t=1e-3, scal=scal)
    torch.cuda.synchronize()
    assert torch.equal(p, p2) and torch.equal(sh0[off: off + items * H].view(items, H), ref2) and torch.equal(sh0, sh1)
    # push: one source block into slot 1 of two destination buffers
    src = torch.randn(256, device="cuda")
    d0 = torch.zeros(3, 256, device="cuda"); d1 = torch.zeros(3, 256, device="cuda")
    ops.peer_push(src, 1024, ops.peer_table([d0.data_ptr(), d1.data_ptr()]), 1024, 2)
    torch.cuda.synchronize()
    assert torch.equal(d0[1], src) and torch.equal(d1[1], src) and (d0[0] == 0).all() and (d0[2] == 0).all()
    # barrier / small all-reduce with a single rank: must not hang, must leave the values alone, must advance the epochs
    pads = torch.zeros(ops.PEER_SLOTS * 8, dtype=torch.int32, device="cuda"); epochs = torch.zeros(ops.PEER_SLOTS, dtype=torch.int32, device="cuda")
    tab_p = ops.peer_table([pads.data_ptr()])
    vals = torch.arange(16, dtype=torch.float32, device="cuda")
    ops.peer_barrier(tab_p, 0, 1, 2, epochs)
    ops.peer_allreduce_small(ops.peer_table([vals.data_ptr()]), 3, 2, tab_p, 0, 1, 0, epochs)
    torch.cuda.synchronize()
    assert torch.equal(vals, torch.arange(16, dtype=torch.float32, device="cuda"))
    assert epochs.tolist() == [2, 0, 1, 0]


def test_wgrad_adam_epilogue_matches_gemm_then_adam(ops):
    """EpiAdam (decoder weight-gradient GEMM whose epilogue applies TF-Adam) against the two kernels it replaces: the same GEMM
    storing the fp32 gradient, then ltg_adam. Same accumulators, same formula: equal up to FMA contraction (1e-6)."""
    torch.manual_seed(21)
    K, M, H = 500, 1300, 600
    A = (torch.randn(K, M + 4, device="cuda") * 0.05).bfloat16()            # stored [K, lda]: dlogits-like
    Bm = torch.zeros(K, 608, device="cuda", dtype=torch.bfloat16)
    Bm[:, :H] = torch.tanh(torch.randn(K, H, device="cuda")).bfloat16(); Bm[:, H] = 1.0
    p = torch.randn(M, H, device="cuda") * 0.1; m = torch.randn(M, H, device="cuda") * 1e-3; v = torch.rand(M, H, device="cuda") * 1e-4
    p2, m2, v2 = p.clone(), m.clone(), v.clone()
    sh = torch.zeros(M, H, device="cuda", dtype=torch.bfloat16); sh2 = torch.zeros_like(sh)
    aux = torch.zeros(M, device="cuda"); aux2 = torch.zeros(M, device="cuda")
    scal = torch.zeros(16, device="cuda"); scal[ops.S_LR_T] = 3e-4
    ops.wgrad_adam(A, Bm, M, H + 1, K, p, m, v, sh, H, aux_col=H, aux_out=aux, scal=scal)
    G = torch.zeros(M, H, device="cuda")
    ops.gemm(A, Bm, M, H + 1, K, a_mn=True, b_mn=True, bn=128, out_f32=G, ld_f32=H, aux_col=H, aux_out=aux2)
    ops.adam(p2, m2, v2, G, sh2, scal=scal)
    torch.cuda.synchronize()
    assert torch.equal(aux, aux2)
    want = A[:, :M].float().t() @ Bm[:, :H].float()
    assert (G - want).abs().max().item() < 2e-2 * want.abs().max().item()
    for a, b in ((p, p2), (m, m2), (v, v2)):
        assert (a - b).abs().max().item() <= 1e-6 * max(1.0, b.abs().max().item())
    assert (sh.float() - sh2.float()).abs().max().item() <= 1e-2 * 0.5 and (sh != sh2).float().mean().item() < 1e-3


# ----------------------------------------------------------------------------------------------------------------
# VAE middle on tcgen05 (mid_tc.cu) against a torch fp32 restatement of MultiVAE.py:151-181 / its autodiff, and against the
# mma.sync kernels (mid_kernels.cu) on the same inputs
# ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [500, 77, 128, 1])
def test_vae_mid_tc_forward_backward(ops, B):
    torch.manual_seed(5 + B)
    H, L = 600, 200
    h1 = (torch.randn(B, H, device="cuda") * 0.5).tanh().bfloat16()
    Wq1 = (torch.randn(H, 2 * L, device="cuda") * 0.05).bfloat16(); bq1 = torch.randn(2 * L, device="cuda") * 0.01
    Wp0 = (torch.randn(L, H, device="cuda") * 0.08).bfloat16(); bp0 = torch.randn(H, device="cuda") * 0.01
    eps = torch.randn(B, L, device="cuda")
    outs = {}
    for tc in (False, True):
        mulv = torch.zeros(B, 2 * L, device="cuda"); z = torch.zeros(B, L, device="cuda", dtype=torch.bfloat16)
        zmu = torch.zeros(B, L, device="cuda"); h2 = torch.zeros(B, 608, device="cuda", dtype=torch.bfloat16); scal = torch.zeros(16, device="cuda")
        ops.vae_mid_fwd(h1, Wq1, bq1, Wp0, bp0, eps, B, 0, 1.0, 0, 0, None, mulv, z, zmu, h2, scal, tc=tc)
        torch.cuda.synchronize()
        outs[tc] = (mulv, z, zmu, h2, scal)
    # fp32 reference on the bf16-rounded operands
    mv = h1.float() @ Wq1.float() + bq1
    mu, lv = mv[:, :L], mv[:, L:]
    kl = (0.5 * (-lv + lv.exp() + mu * mu - 1.0)).sum()
    d = eps * (0.5 * lv).exp()
    zr = (mu + d)
    h2r = (zr.bfloat16().float() @ Wp0.float() + bp0).tanh()
    for tc in (False, True):
        mulv, z, zmu, h2, scal = outs[tc]
        assert (mulv - mv).abs().max().item() < 2e-3, tc
        assert (zmu - d).abs().max().item() < 2e-3, tc
        assert (z.float() - zr).abs().max().item() < 2e-2, tc
        assert (h2[:, :H].float() - h2r).abs().max().item() < 2e-2, tc
        assert abs(scal[ops.S_KL_SUM].item() - kl.item()) < 1e-3 * abs(kl.item()) + 1e-3, tc
    # tensor-core version against the mma.sync version: same operands, same accumulation type
    assert (outs[True][0] - outs[False][0]).abs().max().item() < 1e-4
    assert (outs[True][3].float() - outs[False][3].float()).abs().max().item() < 1e-2
    # inference mode (phase A / evaluation): z = mu, Philox path not taken
    mulv, z, zmu, h2, scal = [torch.zeros_like(t) for t in outs[True]]
    ops.vae_mid_fwd(h1, Wq1, bq1, Wp0, bp0, None, B, 7, 0.0, 3, 1, None, mulv, z, zmu, h2, scal, tc=True)
    assert (z.float() - mu).abs().max().item() < 2e-2 and zmu.abs().max().item() == 0.0

    # ---- backward
    mulv, z, zmu, h2, scal = outs[True]
    dh2pre = (torch.randn(B, H, device="cuda") * 0.01).bfloat16()
    anneal, Bg = 0.13, max(B, 2)
    res = {}
    for tc in (False, True):
        dmulv = torch.zeros(B, 2 * L, device="cuda", dtype=torch.bfloat16); dh1pre = torch.zeros(B, H, device="cuda")
        dh1pre_b = torch.zeros(B, H, device="cuda", dtype=torch.bfloat16); dbq1 = torch.zeros(2 * L, device="cuda"); dbq0 = torch.zeros(H, device="cuda")
        ops.vae_mid_bwd(dh2pre, Wp0, Wq1, mulv, zmu, h1, B, Bg, anneal, scal, dmulv, dh1pre, dh1pre_b, dbq1, dbq0, tc=tc)
        torch.cuda.synchronize()
        res[tc] = (dmulv, dh1pre, dh1pre_b, dbq1, dbq0)
    dz = dh2pre.float() @ Wp0.float().t()
    dmu = dz + anneal * mulv[:, :L] / Bg
    dlv = dz * zmu * 0.5 + anneal * 0.5 * (mulv[:, L:].exp() - 1.0) / Bg
    dmv = torch.cat([dmu, dlv], 1)
    dh1 = dmv.bfloat16().float() @ Wq1.float().t()
    dh1p = dh1 * (1.0 - h1.float() ** 2)
    sc = dh1p.abs().max().item()
    for tc in (False, True):
        dmulv, dh1pre, dh1pre_b, dbq1, dbq0 = res[tc]
        assert (dmulv.float() - dmv).abs().max().item() < 1e-2 * dmv.abs().max().item() + 1e-6, tc
        assert (dh1pre - dh1p).abs().max().item() < 2e-2 * sc + 1e-7, tc
        assert (dh1pre_b.float() - dh1pre).abs().max().item() < 1e-2 * sc + 1e-7, tc
        assert (dbq1 - dmv.sum(0)).abs().max().item() < 2e-2 * dmv.sum(0).abs().max().item() + 1e-6, tc
        assert (dbq0 - dh1p.sum(0)).abs().max().item() < 2e-2 * dh1p.sum(0).abs().max().item() + 1e-6, tc
    assert (res[True][1] - res[False][1]).abs().max().item() < 1e-3 * sc + 1e-8
