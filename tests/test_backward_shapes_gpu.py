"""The backward pass of the assembled GAN step at the shapes it trains at, stage by stage against float64.

One GanEngine (graphs off, lam = 1) on the ML-20M-shaped catalog (I = 20,108) with batch 500: one full batch (500 users, 4 row
blocks: 4-CTA clusters) and one ragged batch (383 users, 3 row blocks plus a zero-filled padding block), and a second engine whose
only batch holds ONE user (every weight-gradient GEMM contracts over K = 1; the discriminator's P = 20 pairs give one k block for
16 split-K partials, 15 of which are empty). Each batch runs phase A, the D update and the G update without the optimizer step;
every stage is then checked against float64 computed from THAT STAGE's own device inputs, so a kernel is tested in isolation and
an error cannot hide behind an upstream one.

Bounds (tests/helpers.py): GEMM-shaped stages |got - ref| <= 2^-14 (|A| |B|) per element from the exact bf16 operands; bf16
outputs add half a bf16 ulp; element-wise kernels a few fp32 ulps, derived next to each assert; index and bit outputs exact. Every
GEMM-shaped bound is also shown to FAIL for a reference with its last k block, or its last split partial, missing.
"""
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
from helpers import TAU, U32, HALF_BF16, TINY, gemm_ref, drop_last_kblock, assert_within, assert_detects  # noqa: E402

pytestmark = pytest.mark.gpu

H, L = 600, 200
CASES = ["b500", "b383", "b1"]


def _mods():
    names = ("synthetic", "generator", "discriminator", "engine", "ops")
    return [importlib.import_module("long-tail-gan_b200." + n) for n in names]


def _engine(n_users, first_batch=0):
    syn, gen, dis, eng, ops = _mods()
    I = syn.CONFIGS["ml20m"][1]
    tabs = syn.make_config("ml20m", n_users=n_users)
    params = orc.init_vae_params(I, seed=1)
    params[3] = params[3] * 4.0           # decoder weights large enough for a peaked softmax
    E, dparams = orc.init_disc_params(I, 100, 150, 250, 300, seed=2)
    vae = gen.MultiVAE([200, 600, I], lam=0.0, random_seed=1)
    vae.set_params(params); vae.reset_optimizer()
    disc = dis.Discriminator(I, I, 100, 150, 250, 300, seed=1)
    disc.set_params(E, dparams)
    data = eng.TrainData(batch_size=500, first_batch=first_batch, **tabs)
    engine = eng.GanEngine(vae, disc, data.max_B, data.max_P, seed=4711, lr=1e-4, lam=1.0, use_graphs=False, max_active=data.max_active)
    return engine, data, tabs


def _snapshot_d(engine, data, bi):
    """phase A and the D forward/backward of batch bi; returns the D stage's device tensors (before the D optimizer step)."""
    d = engine.disc
    bt = data.batches[bi]
    engine.phase_a(data, bi)
    # the regions the weight-gradient GEMMs own (every split writes its partial, empty splits zeros): poisoned with NaN first
    for name, nsp, rows, ld, cols in (("W1", engine.d_sp, d.h0 + 1, d.ld1, d.h1), ("W2", engine.d_sp, d.h0 + 1, d.ld2, d.h2),
                                      ("W3", engine.d_sp3, d.k3, d.ld3, d.h3)):
        o = d._off[name][0]
        engine.arena_gp[:nsp, o:o + rows * ld].view(nsp, rows, ld)[:, :, :cols] = float("nan")
    engine._d_fwd_bwd(data, bi)
    torch.cuda.synchronize()
    P = bt["P"]
    snap = dict(P=P, parts=engine._d_parts, sp=engine.d_sp, sp3=engine.d_sp3, Xp=engine.Xp[:P].clone(), Xn=engine.Xn[:P].clone(),
                Hd=engine.Hd[:P].clone(), dz3=engine.dz3[:P].clone(), dz12=engine.dz12[:P].clone(), gp=engine.arena_gp.clone(),
                W3b=d.view("W3", "b").clone())
    engine._d_update()
    return snap


def _snapshot_g(engine, data, bi):
    """g_step(update=False) of batch bi (after phase A and the D update); returns the G stage's device tensors."""
    v = engine.vae
    bt = data.batches[bi]
    B, I = bt["B"], engine.I
    engine.dh2_part.fill_(float("nan"))     # every split partial of the dgrad GEMM is written for the batch rows
    engine.g_step(data, bi, update=False)
    torch.cuda.synchronize()
    nb = engine.dgrad_splits
    c = lambda t: t.clone()  # noqa: E731
    return dict(
        B=B, I=I, bt=bt, step=int(engine.w_g.item()), scal=c(engine.scal),
        logits=c(engine.logits[:B]), lse=c(engine.lse[:B]), dl=c(engine.dl[:B]), h2=c(engine.h2[:B]), z=c(engine.z[:B]), h1=c(engine.h1[:B]),
        mulv=c(engine.mulv[:B]), zmu=c(engine.zmu[:B]), dh2_part=c(engine.dh2_part[:, :B]), splits=nb, dh2pre=c(engine.dh2pre[:B]),
        dmulv=c(engine.dmulv[:B]), dh1pre=c(engine.dh1pre[:B]), dh1pre_b=c(engine.dh1pre_b[:B]), coef=c(data.coef[bt["e0"]:bt["e1"]]),
        G_enc=c(engine.G_enc[:bt["n_active"]]), Xc_absmax=engine.Xc.float().abs().max().item(), dWdT=c(engine.dWdT),
        g=dict((k, c(v.view(k, "g"))) for k in ("W_p0", "W_q1", "b_q0", "b_q1", "b_p0", "b_p1")),
        WdT_b=c(v.WdT_b), Wp0_b=c(v.view("W_p0", "b")), Wq1_b=c(v.view("W_q1", "b")), b_p1=c(v.view("b_p1")),
        indptr=data.h_indptr[bt["b0"]: bt["b0"] + B + 1] - data.h_indptr[bt["b0"]], indices=data.h_indices[bt["e0"]:bt["e1"]],
        samp_ptr=bt["samp_ptr"].cpu().numpy(), pair_niche=bt["pair_niche"].cpu().numpy(), label=bt["label"].cpu().numpy(),
        slot_of_item=bt["slot_of_item"], keep=engine.keep_vae, seed=engine.seed, lam=engine.lam if bt["K"] > 0 else 0.0)


@pytest.fixture(scope="module")
def runs():
    _, _, _, _, ops = _mods()
    ops.init()
    out = {}
    engine, data, _ = _engine(883)
    assert [bt["B"] for bt in data.batches] == [500, 383]
    for bi, key in ((0, "b500"), (1, "b383")):
        dsnap = _snapshot_d(engine, data, bi)
        out[key] = (dsnap, _snapshot_g(engine, data, bi))
    one, data1, _ = _engine(501, first_batch=1)
    assert [bt["B"] for bt in data1.batches] == [1] and data1.batches[0]["P"] > 0 and data1.batches[0]["K"] > 0
    dsnap = _snapshot_d(one, data1, 0)
    out["b1"] = (dsnap, _snapshot_g(one, data1, 0))
    out["_engine"] = (engine, data)
    return out


def _gemm_stage(name, got, A, B, tau=TAU):
    """GEMM-shaped fp32 stage: per-element bound from the exact operands, and the bound's sensitivity to a missing k block."""
    ref, mag = gemm_ref(A, B)
    bound = tau * mag + TINY
    assert_within(name, got, ref, bound)
    assert_detects(name + " minus last k block", got, drop_last_kblock(ref, A, B), bound)
    return ref, mag


def _sampled_mask(s):
    """m[u, i] = 1 for the valid generated pairs of user u (train.py:316 generated_tags)."""
    B, I = s["B"], s["I"]
    bt = s["bt"]
    Pr = bt["Pr"]
    m = torch.zeros(B, I, dtype=torch.float64, device="cuda")
    sp = s["samp_ptr"]
    rows = np.repeat(np.arange(B), np.diff(sp))
    lab = s["label"][Pr:Pr + len(rows)]
    items = s["pair_niche"][Pr:Pr + len(rows)]
    sel = lab > 0
    m[torch.from_numpy(rows[sel]).cuda(), torch.from_numpy(items[sel].astype(np.int64)).cuda()] = 1.0
    return m


def _dense_x(s):
    B, I = s["B"], s["I"]
    X = torch.zeros(B, I, dtype=torch.float64, device="cuda")
    rows = np.repeat(np.arange(B), np.diff(s["indptr"]))
    X[torch.from_numpy(rows).cuda(), torch.from_numpy(s["indices"].astype(np.int64)).cuda()] = 1.0
    return X


# ------------------------------------------------------------------------------------------------------------------------------------
# G update
# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_decoder_softmax_statistics(runs, case):
    """lse of ltg_dec_row_bwd from the forward's fp32 softmax partials against logsumexp of the float64 logits h2 WdT_b^T + b_p1."""
    s = runs[case][1]
    I = s["I"]
    A = s["h2"][:, :H]
    logits, mag = gemm_ref(A, s["WdT_b"].t())
    logits = logits + s["b_p1"][:I].double()
    want = torch.logsumexp(logits, dim=1)
    # a logit is off by at most TAU |h2||W| (+ its bias add); the max-shifted sums take ex2.approx / __expf (relative 2^-21 plus the
    # rounding of the argument, |x| 2^-23) over <= 64-term chains and a 256-thread tree (<= 2^-18 relative), logf and the final
    # add a few ulps of |lse|
    bound = TAU * mag.max(dim=1).values + 2.0 ** -18 + 2.0 ** -21 * (want.abs() + logits.abs().max(dim=1).values)
    assert_within("lse [%s]" % case, s["lse"], want, bound)


@pytest.mark.parametrize("case", CASES)
def test_decoder_dlogits(runs, case):
    """dl of ltg_dec_row_bwd (ltgan.h: dl = pi (xw/Bg + lam Ybar s_u) - x/Bg - lam Ybar pi m) from the bf16 logit stash, the device
    lse, X, the sampled mask and Ybar = scal[SUM_Y] / scal[CNT]."""
    _, _, _, _, ops = _mods()
    s = runs[case][1]
    B, I = s["B"], s["I"]
    lg = s["logits"][:, :I].double()
    lse = s["lse"].double()[:, None]
    X, m = _dense_x(s), _sampled_mask(s)
    sc = s["scal"].double()
    cnt = sc[ops.S_CNT].item()
    ybar = np.float32(np.float32(sc[ops.S_SUM_Y].item()) / np.float32(cnt)) if (cnt > 0 and s["lam"] != 0) else 0.0
    lam = s["lam"]
    pi = torch.exp(lg - lse)
    su = (pi * m).sum(1, keepdim=True)
    xw = X.sum(1, keepdim=True)
    a = xw / B + lam * ybar * su
    dense = pi * a
    fix_x = X / B
    fix_m = lam * ybar * pi * m
    want = dense - fix_x - fix_m
    # fp32 arithmetic of the kernel: __expf(x) relative 2^-21 + |x| 2^-22; a = xw inv_bg + lam ybar sp (sp: a sum of such terms over
    # a block tree, a few ulps): relative 2^-19 on top of the largest __expf error of the row
    e_el = 2.0 ** -21 + (lg - lse).abs() * 2.0 ** -22
    e_row = (e_el * m).max(dim=1, keepdim=True).values
    acc = dense.abs() * (e_el + e_row + 2.0 ** -19)
    acc = acc + HALF_BF16 * (dense.abs() + acc)                       # dense pass rounded to bf16
    acc = torch.where(X > 0, acc + HALF_BF16 * ((dense - fix_x).abs() + acc) + U32 / B, acc)   # fix-up: bf16(dl - x/Bg)
    acc = torch.where(m > 0, acc + fix_m.abs() * (e_el + 2 * U32), acc)
    acc = torch.where(m > 0, acc + HALF_BF16 * (want.abs() + acc), acc)                       # fix-up: bf16(dl - lam Ybar pi)
    assert_within("dlogits [%s]" % case, s["dl"][:, :I], want, acc + TINY)
    assert (s["dl"][:, I:] == 0).all()    # pitch padding stays zero: the weight-gradient GEMMs read whole 64-column boxes


@pytest.mark.parametrize("case", CASES)
def test_decoder_dgrad_split_k(runs, case):
    """dh2 = dl WdT_b as `dgrad_splits` fp32 partials (split-K over the catalog, split_stride): their sum against float64, every
    partial whose k range is empty exactly 0, and the bound blind to nothing: the sum without its last non-empty partial fails."""
    s = runs[case][1]
    I, S = s["I"], s["splits"]
    A, Bm = s["dl"][:, :I], s["WdT_b"]
    parts = s["dh2_part"]
    kb = (I + 63) // 64
    per = (kb + S - 1) // S
    used = [sp for sp in range(S) if sp * per < kb]
    for sp in range(S):
        if sp not in used:
            assert (parts[sp] == 0).all(), "empty split %d must store zeros" % sp
    got = parts.double().sum(0)
    ref, mag = gemm_ref(A, Bm)
    bound = TAU * mag + TINY
    assert_within("dgrad sum of %d partials [%s]" % (S, case), got, ref, bound)
    assert_detects("dgrad minus last k block", got, drop_last_kblock(ref, A, Bm), bound)
    if len(used) > 1:
        assert_detects("dgrad without its last partial", got - parts[used[-1]].double(), ref, bound)


@pytest.mark.parametrize("case", CASES)
def test_tanh_backward_of_decoder_input(runs, case):
    """ltg_tanh_bwd: dh2pre = (sum of the fp32 partials) (1 - h2^2) as bf16, and the b_p0 gradient (column sums)."""
    s = runs[case][1]
    B = s["B"]
    parts = s["dh2_part"].double()
    t = s["h2"][:, :H].double()
    want = parts.sum(0) * (1 - t * t)
    # fp32: <= S - 1 additions of the partials (relative (S) u of sum |p|), then 1 - t^2 and the product (3 u)
    e = parts.shape[0] * U32 * parts.abs().sum(0) * (1 - t * t).abs() + 3 * U32 * want.abs()
    assert_within("dh2pre [%s]" % case, s["dh2pre"], want, e + HALF_BF16 * (want.abs() + e) + TINY)
    # column sums of the fp32 values: the element errors plus (B + 8) u of sum |.| (per-CTA chains of 4 rows, then float atomics)
    assert_within("b_p0 grad [%s]" % case, s["g"]["b_p0"], want.sum(0), e.sum(0) + (B + 8) * U32 * want.abs().sum(0) + TINY)


@pytest.mark.parametrize("case", CASES)
def test_wgrad_W_p0(runs, case):
    """dW_p0 = z^T dh2pre (M = 200: CTA pairs; K = the batch)."""
    s = runs[case][1]
    _gemm_stage("dW_p0 [%s]" % case, s["g"]["W_p0"], s["z"].t(), s["dh2pre"])


@pytest.mark.parametrize("case", CASES)
def test_vae_mid_backward(runs, case):
    """ltg_vae_mid_bwd: dmulv, dh1pre (fp32 and bf16), the b_q1 / b_q0 gradients; formulas of test_vae_mid_tc_forward_backward with the
    anneal weight the device wrote into scal. The second half is checked from the device's own dmulv."""
    _, _, _, _, ops = _mods()
    s = runs[case][1]
    B = s["B"]
    anneal = s["scal"][ops.S_ANNEAL].double().item()
    mulv, zmu = s["mulv"].double(), s["zmu"].double()
    mu, lv = mulv[:, :L], mulv[:, L:]
    dz, dz_mag = gemm_ref(s["dh2pre"], s["Wp0_b"].t())
    e_dz = TAU * dz_mag + TINY
    t1 = dz * zmu * 0.5
    t2 = anneal * 0.5 * (lv.exp() - 1.0) / B
    dmv = torch.cat([dz + anneal * mu / B, t1 + t2], 1)
    # dmu: the dz error plus 3 roundings; dlogvar: dz error x |zmu|/2, expf (2 ulp) and 5 roundings of the two terms
    e_mu = e_dz + 4 * U32 * (dz.abs() + (anneal * mu / B).abs())
    e_lv = e_dz * zmu.abs() * 0.5 + 8 * U32 * (t1.abs() + anneal * 0.5 * (lv.exp() + 1.0) / B)
    e = torch.cat([e_mu, e_lv], 1)
    assert_within("dmulv [%s]" % case, s["dmulv"], dmv, e + HALF_BF16 * (dmv.abs() + e) + TINY)
    assert_detects("dmulv minus last k block", s["dmulv"], torch.cat(
        [drop_last_kblock(dz, s["dh2pre"], s["Wp0_b"].t()) + anneal * mu / B, t1 + t2], 1), e + HALF_BF16 * (dmv.abs() + e) + TINY)
    assert_within("b_q1 grad [%s]" % case, s["g"]["b_q1"], dmv.sum(0), e.sum(0) + (B + 16) * U32 * dmv.abs().sum(0) + TINY)
    # second half from the device's dmulv: dh1pre = (dmulv W_q1^T) (1 - h1^2)
    dh1, dh1_mag = gemm_ref(s["dmulv"], s["Wq1_b"].t())
    h1 = s["h1"].double()
    g1 = 1 - h1 * h1
    want = dh1 * g1
    e1 = TAU * dh1_mag * g1.abs() + 3 * U32 * want.abs() + TINY
    assert_within("dh1pre [%s]" % case, s["dh1pre"], want, e1)
    assert_detects("dh1pre minus last k block", s["dh1pre"], drop_last_kblock(dh1, s["dmulv"], s["Wq1_b"].t()) * g1, e1)
    assert_within("dh1pre bf16 [%s]" % case, s["dh1pre_b"], want, e1 + HALF_BF16 * (want.abs() + e1))
    assert_within("b_q0 grad [%s]" % case, s["g"]["b_q0"], want.sum(0), e1.sum(0) + (B + 16) * U32 * want.abs().sum(0) + TINY)


@pytest.mark.parametrize("case", CASES)
def test_wgrad_W_q1(runs, case):
    """dW_q1 = h1^T dmulv (M = 600: CTA pairs with a zero-filled padding row block)."""
    s = runs[case][1]
    _gemm_stage("dW_q1 [%s]" % case, s["g"]["W_q1"], s["h1"].t(), s["dmulv"])


@pytest.mark.parametrize("case", CASES)
def test_encoder_coefficients(runs, case):
    """coef = x rsqrt(|x|^2) mask / keep per interaction of the batch: the dropout bits exactly (Philox mirror), values to 4 ulps
    (rsqrtf: 2 ulps, then one division)."""
    s = runs[case][1]
    bt = s["bt"]
    B, I = s["B"], s["I"]
    deg = np.diff(s["indptr"])
    rows = np.repeat(np.arange(B), deg)
    idx = (np.uint64(bt["uid0"]) + rows.astype(np.uint64)) * np.uint64(I) + s["indices"].astype(np.uint64)
    mask = philox.keep_mask(s["seed"], philox.STREAM_ENC_DROPOUT, s["step"], idx, s["keep"])
    assert len(mask) < 1000 or 0.7 < mask.mean() < 0.8
    got = s["coef"]
    assert np.array_equal(got.cpu().numpy() != 0, mask)
    want = torch.from_numpy(np.where(mask, 1.0 / np.sqrt(deg[rows].astype(np.float64)) / np.float64(np.float32(s["keep"])), 0.0)).cuda()
    assert_within("coef [%s]" % case, got, want, 4 * 2 * U32 * want.abs() + TINY)


@pytest.mark.parametrize("case", CASES)
def test_encoder_weight_gradient_and_xc_cleared(runs, case):
    """G_enc[:n_active] = Xc^T dh1pre_b with Xc[row, slot_of_item[item]] = bf16(coef) rebuilt from the device coefficients; and the
    dense Xc matrix all-zero again after the G step (else the next step's encoder gradient is polluted)."""
    s = runs[case][1]
    B = s["B"]
    n_act = s["G_enc"].shape[0]
    rows = torch.from_numpy(np.repeat(np.arange(B), np.diff(s["indptr"]))).cuda()
    slots = s["slot_of_item"].long()[torch.from_numpy(s["indices"].astype(np.int64)).cuda()]
    assert int(slots.min()) >= 0 and int(slots.max()) < n_act
    Xc = torch.zeros(B, n_act, dtype=torch.float64, device="cuda")
    Xc[rows, slots] = s["coef"].bfloat16().double()
    _gemm_stage("G_enc [%s]" % case, s["G_enc"], Xc.t(), s["dh1pre_b"])
    assert s["Xc_absmax"] == 0.0


@pytest.mark.parametrize("case", CASES)
def test_wgrad_decoder(runs, case):
    """dWdT = dl^T [h2 | 1] (M = 20,108, N = 601, K = the batch): columns < 600 to dWdT, the ones column to the b_p1 gradient."""
    s = runs[case][1]
    I = s["I"]
    A = s["dl"][:, :I].t()
    Bm = s["h2"][:, :H + 1]
    ref, mag = gemm_ref(A, Bm)
    bound = TAU * mag + TINY
    got = torch.cat([s["dWdT"], s["g"]["b_p1"][:I, None]], 1)
    assert_within("dWdT | b_p1 grad [%s]" % case, got, ref, bound)
    assert_detects("dWdT minus last k block", got, drop_last_kblock(ref, A, Bm), bound)


# ------------------------------------------------------------------------------------------------------------------------------------
# decoder update paths with the optimizer step: EpiAdam epilogue and the chunked GEMM + Adam pipeline, against float64 TF-Adam
# ------------------------------------------------------------------------------------------------------------------------------------
def _adam_bound(g, dg, m0, v0, p0, lr_t, b1=0.9, b2=0.999, eps=1e-8):
    """float64 TF-Adam of (p0, m0, v0) on gradient g and per-element bounds on m, v, p when the gradient is known to within dg:
    m: (1-b1) dg; v: (1-b2)(2|g| dg + dg^2); r = m/(sqrt v + eps): dm/s_lo + |m| (1/s_lo - 1/s_hi) with s = sqrt(v -/+ dv) + eps;
    plus 4 fp32 ulps of each quantity for the kernel's own arithmetic."""
    m = b1 * m0 + (1 - b1) * g
    v = b2 * v0 + (1 - b2) * g * g
    r = m / (v.sqrt() + eps)
    p = p0 - lr_t * r
    dm = (1 - b1) * dg + 8 * U32 * (b1 * m0.abs() + (1 - b1) * g.abs())
    dv = (1 - b2) * (2 * g.abs() * dg + dg * dg) + 8 * U32 * (b2 * v0 + (1 - b2) * g * g)
    s_lo = (v - dv).clamp_min(0).sqrt() + eps
    s_hi = (v + dv).sqrt() + eps
    dr = dm / s_lo + m.abs() * (1 / s_lo - 1 / s_hi) + 8 * U32 * r.abs()
    dp = lr_t * dr + 8 * U32 * (p0.abs() + lr_t * r.abs())
    return (p, dp), (m, dm), (v, dv)


@pytest.mark.parametrize("path", ["epi_adam", "chunked"])
def test_decoder_update_paths(runs, path):
    _, _, _, _, ops = _mods()
    engine, data = runs["_engine"]
    v = engine.vae
    bi = 0 if path == "epi_adam" else 1
    engine.fused_wgrad_adam = path == "epi_adam"
    engine.dec_chunks = 1 if path == "epi_adam" else 4
    try:
        engine.phase_a(data, bi)
        engine.d_step(data, bi)
        torch.cuda.synchronize()
        p0, m0, v0 = v.WdT.double(), v.WdT_m.double(), v.WdT_v.double()
        engine.g_step(data, bi, update=True)
        torch.cuda.synchronize()
    finally:
        engine.fused_wgrad_adam, engine.dec_chunks = False, 1
    B, I = data.batches[bi]["B"], engine.I
    lr_t = engine.scal[ops.S_LR_T].double().item()
    assert lr_t > 0
    g, mag = gemm_ref(engine.dl[:B, :I].t(), engine.h2[:B, :H])      # this step's own dl and h2 (the Adam step does not touch them)
    (p, dp), (m, dm), (vv, dv) = _adam_bound(g, TAU * mag + TINY, m0, v0, p0, lr_t)
    assert_within("WdT m [%s]" % path, v.WdT_m, m, dm + TINY)
    assert_within("WdT v [%s]" % path, v.WdT_v, vv, dv + TINY)
    assert_within("WdT [%s]" % path, v.WdT, p, dp + TINY)
    assert_within("WdT bf16 shadow [%s]" % path, v.WdT_b, p, dp + HALF_BF16 * (p.abs() + dp) + TINY)
    assert (v.WdT.double() != p0).float().mean().item() > 0.5     # the step did move the weights


# ------------------------------------------------------------------------------------------------------------------------------------
# D update
# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_disc_dz12(runs, case):
    """dz12 = (dz3 W3^T) dact(Hd) (the dgrad GEMM with the fused dropout-tanh backward) on the columns the weight gradients read."""
    snap = runs[case][0]
    engine, _ = runs["_engine"]
    d = engine.disc
    keep = engine.keep_d
    A, Bm = snap["dz3"][:, :d.h3], snap["W3b"][:, :d.h3].t()
    ref, mag = gemm_ref(A, Bm)
    y = snap["Hd"].double()
    dact = torch.where(y != 0, (1 - (y * keep) ** 2) / keep, torch.zeros_like(y))
    used = torch.tensor(list(range(d.h1)) + list(range(d.off2, d.off2 + d.h2)), device="cuda")
    want = (ref * dact)[:, used]
    # the GEMM bound scaled by |dact|, 5 roundings of the dact arithmetic and the product, then the bf16 store
    e = (TAU * mag * dact.abs())[:, used] + 5 * U32 * want.abs() + TINY
    bound = e + HALF_BF16 * (want.abs() + e)
    got = snap["dz12"][:, used]
    assert_within("dz12 [%s]" % case, got, want, bound)
    assert_detects("dz12 minus last k block", got, (drop_last_kblock(ref, A, Bm) * dact)[:, used], bound)


@pytest.mark.parametrize("case", CASES)
def test_disc_weight_gradients_split_k(runs, case):
    """The split-K partials of the three discriminator weight-gradient GEMMs (arena_gp, summed by the Adam kernel): W3 (+b3) = Hd^T
    dz3, W1 (+b1) = Xp^T dz1, W2 (+b2) = Xn^T dz2 with dz2 = the dz12[:, off2:] slice read at pitch k3. The sum over every partial
    the Adam step reads against float64; partials whose k range is empty exactly 0 (they were NaN before the step); the sum without
    the last non-empty partial fails the bound."""
    snap = runs[case][0]
    engine, _ = runs["_engine"]
    d = engine.disc
    P = snap["P"]
    k1 = d.h0 + 1
    kb = (P + 63) // 64
    stages = (("W3", snap["sp3"], d.k3, d.ld3, d.h3, snap["Hd"][:, :d.k3], snap["dz3"][:, :d.h3]),
              ("W1", snap["sp"], k1, d.ld1, d.h1, snap["Xp"][:, :k1], snap["dz12"][:, :d.h1]),
              ("W2", snap["sp"], k1, d.ld2, d.h2, snap["Xn"][:, :k1], snap["dz12"][:, d.off2:d.off2 + d.h2]))
    if case == "b1":
        assert kb < snap["sp"]    # empty splits are exercised
    for name, sp, rows, ld, cols, X, dz in stages:
        o = d._off[name][0]
        parts = snap["gp"][:snap["parts"], o:o + rows * ld].view(snap["parts"], rows, ld)[:, :, :cols]
        per = (kb + sp - 1) // sp
        used = [s for s in range(sp) if s * per < kb]
        for s in range(sp, snap["parts"]):
            assert (parts[s] == 0).all(), (name, s)     # partials the GEMM does not own: the Adam kernel reads them as zeros
        for s in range(sp):
            if s not in used:
                assert (parts[s] == 0).all(), "%s: empty split %d must store zeros" % (name, s)
        got = parts.double().sum(0)
        ref, mag = gemm_ref(X.t(), dz)
        bound = TAU * mag + TINY
        assert_within("d%s sum of %d partials [%s]" % (name, sp, case), got, ref, bound)
        assert_detects("d%s minus last k block" % name, got, drop_last_kblock(ref, X.t(), dz), bound)
        if len(used) > 1:
            assert_detects("d%s without its last partial" % name, got - parts[used[-1]].double(), ref, bound)
