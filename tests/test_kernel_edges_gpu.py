"""Kernel entry points at the configurations and edges the training step reaches, called directly, against float64 or bit-exact
references: the decoder forward at every tile shape a batch <= 500 selects, the split-K tanh backward (vector and scalar kernels),
the partial-sum kernel, the one-launch step advance, the dense encoder coefficient matrix (gather, clear, data-parallel rebuild),
the sampler with explicit candidate logits and the bf16 cast. (The generic GEMM's instantiations are swept in
test_kernels_gpu.py::test_gemm_layouts.) Bounds as in tests/helpers.py."""
import importlib
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers  # noqa: E402
from helpers import TAU, U32, HALF_BF16, TINY, gemm_ref, assert_within, assert_detects  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    pkg = importlib.import_module("long-tail-gan_b200")
    pkg._lib.build()
    o = importlib.import_module("long-tail-gan_b200.ops")
    o.init()
    return o


def dev(x):
    return torch.as_tensor(x).cuda().contiguous()


# ------------------------------------------------------------------------------------------------------------------------------------
# decoder forward: tile shape per (B, I), logits stash and softmax partials
# ------------------------------------------------------------------------------------------------------------------------------------
def logits_tile_shape(B, n_items, sms):
    """Mirror of gemm_ops.cu logits_tile_shape: (tile width, cluster size) of the decoder forward."""
    m_blocks = (B + 127) // 128
    best, out = -1, None
    for bn, cm in ((256, 4), (256, 2), (192, 2), (128, 2), (256, 1), (192, 1), (128, 1)):
        if (cm > 1 and m_blocks < cm) or (cm == 1 and m_blocks > 1) or (cm == 4 and m_blocks not in (3, 4)):
            continue
        clusters = sms * 33 // 148 if cm == 4 else sms // cm
        tiles = ((m_blocks + cm - 1) // cm) * ((n_items + bn - 1) // bn)
        cost = ((tiles + clusters - 1) // clusters) * (bn + 48)
        if best < 0 or cost < best:
            best, out = cost, (bn, cm)
    return out


DEC_B = (1, 96, 129, 257, 383, 500)


@pytest.mark.parametrize("I", [20108, 17769])
def test_decoder_forward_tile_shapes(ops, I):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    reachable = {logits_tile_shape(B, I, sms) for B in range(1, max(DEC_B) + 1)}
    swept = {logits_tile_shape(B, I, sms) for B in DEC_B}
    assert swept == reachable, (swept, reachable)
    g = torch.Generator(device="cuda").manual_seed(I)
    W = (torch.randn(I, 600, device="cuda", generator=g) * 0.3).bfloat16()
    bias = torch.randn(I, device="cuda", generator=g) * 0.5
    ld = (I + 7) // 8 * 8
    for B in DEC_B:
        bn, cm = logits_tile_shape(B, I, sms)
        nblk = ops.dec_logits_nblk(B, I)
        assert nblk == 4 * ((I + bn - 1) // bn), (B, bn, cm, nblk)
        h2 = torch.zeros(B, 608, device="cuda", dtype=torch.bfloat16)
        h2[:, :600] = torch.tanh(torch.randn(B, 600, device="cuda", generator=g)).bfloat16()
        logits = torch.full((B, ld), float("nan"), device="cuda", dtype=torch.bfloat16)
        partial = torch.full((ops.dec_logits_nblk_max(I), B, 2), float("nan"), device="cuda")
        ops.dec_logits_fwd(h2, W, bias, B, I, logits, partial)
        lse = torch.full((B,), float("nan"), device="cuda")
        ops.dec_row_stats(partial, nblk, logits, B, None, None, None, None, None, None, lse, None, None, torch.zeros(16, device="cuda"))
        torch.cuda.synchronize()
        ref, mag = gemm_ref(h2[:, :600], W.t())
        ref = ref + bias.double()
        e = TAU * mag + U32 * ref.abs() + TINY          # fp32 accumulation, then the bias add (one rounding)
        tag = "B=%d I=%d bn=%d cm=%d" % (B, I, bn, cm)
        assert_within("logits " + tag, logits[:, :I], ref, e + HALF_BF16 * (ref.abs() + e))
        assert torch.isnan(logits[:, I:]).all()        # nothing written beyond the catalog
        want = torch.logsumexp(ref, dim=1)
        # as test_backward_shapes_gpu.test_decoder_softmax_statistics: logit error, ex2 / __expf and fp32 sums, logf
        bound = e.max(dim=1).values + 2.0 ** -18 + 2.0 ** -21 * (want.abs() + ref.abs().max(dim=1).values)
        assert_within("lse " + tag, lse, want, bound)


# ------------------------------------------------------------------------------------------------------------------------------------
# ltg_tanh_bwd: split-K partials summed on the fly, vector (N % 4 == 0, <= 8 partials) and scalar kernels
# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,n_partials", [(600, 6), (600, 1), (602, 3), (600, 12)])
@pytest.mark.parametrize("B", [1, 3, 500])
def test_tanh_bwd_partials(ops, B, N, n_partials):
    g = torch.Generator(device="cuda").manual_seed(B * 100 + N + n_partials)
    ld_dy = N + 6 if N % 4 else N + 8                  # the partials' pitch differs from N
    stride = (B + 1) * ld_dy
    dy = torch.randn(n_partials * stride + 8, device="cuda", generator=g) * 0.1
    parts = dy[: n_partials * stride].view(n_partials, B + 1, ld_dy)[:, :B, :N].double()
    y = torch.zeros(B, N + 8, device="cuda", dtype=torch.bfloat16)
    y[:, :N] = torch.tanh(torch.randn(B, N, device="cuda", generator=g) * 2).bfloat16()
    dxb = torch.full((B, N + 8), float("nan"), device="cuda", dtype=torch.bfloat16)
    dxf = torch.full((B, N + 4), float("nan"), device="cuda")
    db = torch.zeros(N + 4, device="cuda")
    ops.tanh_bwd(dy, y, B, N, dx_bf16=dxb, dx_f32=dxf, dbias=db, n_partials=n_partials, partial_stride=stride, ld_dy=ld_dy)
    torch.cuda.synchronize()
    t = y[:, :N].double()
    want = parts.sum(0) * (1 - t * t)
    # fp32: n_partials - 1 additions (relative n_partials u of sum |p|), then 1 - t^2 and the product: 3 u
    e = n_partials * U32 * parts.abs().sum(0) * (1 - t * t).abs() + 3 * U32 * want.abs() + TINY
    tag = "B=%d N=%d parts=%d" % (B, N, n_partials)
    assert_within("tanh_bwd fp32 " + tag, dxf[:, :N], want, e)
    assert_within("tanh_bwd bf16 " + tag, dxb[:, :N], want, e + HALF_BF16 * (want.abs() + e))
    assert_within("tanh_bwd dbias " + tag, db[:N], want.sum(0), e.sum(0) + (B + 8) * U32 * want.abs().sum(0) + TINY)
    assert torch.isnan(dxf[:, N:]).all() and torch.isnan(dxb[:, N:]).all() and (db[N:] == 0).all()
    if n_partials > 1:   # the bound sees a partial that was not summed
        assert_detects("tanh_bwd without last partial", dxf[:, :N], (parts[:-1].sum(0)) * (1 - t * t), e)


# ------------------------------------------------------------------------------------------------------------------------------------
# ltg_sum_partials
# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_partials", [1, 12, 16, 32])
def test_sum_partials(ops, n_partials):
    disc_mod = importlib.import_module("long-tail-gan_b200.discriminator")
    d = disc_mod.Discriminator(700, 700, 100, 150, 250, 300, device="cuda", seed=5)
    n = (d.arena_n + 3) // 4 * 4
    stride = n + 4
    g = torch.Generator(device="cuda").manual_seed(n_partials)
    src = torch.randn(n_partials, stride, device="cuda", generator=g)
    out = torch.full((n + 4,), float("nan"), device="cuda")
    ops.sum_partials(src, n_partials, stride, n, out)
    torch.cuda.synchronize()
    p = src[:, :n].double()
    want = p.sum(0)
    assert_within("sum_partials %d" % n_partials, out[:n], want, n_partials * U32 * p.abs().sum(0) + TINY)
    assert torch.isnan(out[n:]).all()
    if n_partials > 1:
        assert_detects("sum_partials without last", out[:n], p[:-1].sum(0), n_partials * U32 * p.abs().sum(0) + TINY)


# ------------------------------------------------------------------------------------------------------------------------------------
# ltg_step_advance3 == ltg_step_advance kinds 0, 1, 2
# ------------------------------------------------------------------------------------------------------------------------------------
def test_step_advance3_equals_three_advances(ops):
    g = torch.Generator(device="cuda").manual_seed(3)
    words0 = torch.tensor([41, 17, 9, 5, 0, 0, 0, 0], dtype=torch.int32, device="cuda")
    scal0 = torch.randn(3, 16, device="cuda", generator=g)
    lens = (1500, 2049, 777)                           # distinct, none a multiple of 1,024
    lr, cap, total = 3e-4, 0.2, 50.0

    def bufs():
        return [torch.randint(1, 1 << 30, (n,), dtype=torch.int32, device="cuda", generator=g) for n in lens]

    w1, s1, z1 = words0.clone(), scal0.clone(), bufs()
    ops.step_advance3(w1, s1[0], s1[1], s1[2], lr, z1[0], z1[1], z1[2], w1[4:5], w1[5:6], w1[6:7], anneal_cap=cap, total_anneal_steps=total)
    w2, s2, z2 = words0.clone(), scal0.clone(), bufs()
    for kind in range(3):
        ops.step_advance(w2, s2[kind], kind, lr, anneal_cap=cap, total_anneal_steps=total, zero=z2[kind], snap=w2[4 + kind:5 + kind])
    torch.cuda.synchronize()
    assert torch.equal(w1, w2), (w1.tolist(), w2.tolist())
    assert w1[:3].tolist() == [44, 19, 10] and w1[4:7].tolist() == [42, 43, 44]
    assert torch.equal(s1, s2)
    for q in range(3):
        assert (z1[q] == 0).all() and (z2[q] == 0).all(), q
    assert (s1[:, :8] == 0).all() and torch.equal(s1[:, 10:], scal0[:, 10:]) and torch.equal(s1[0, 8:10], scal0[0, 8:10])


# ------------------------------------------------------------------------------------------------------------------------------------
# the dense coefficient matrix Xc: forward gather output, self-cleaning, data-parallel rebuild
# ------------------------------------------------------------------------------------------------------------------------------------
def _xc_case(rng, I=3000, B=40):
    indptr, idx = [0], []
    for u in range(B):
        n = 300 if u % 9 == 4 else (0 if u == 7 else int(rng.randint(1, 60)))    # split rows (> 128 nonzeros) and an empty row
        idx.append(np.sort(rng.choice(I, n, replace=False)))
        indptr.append(indptr[-1] + n)
    indptr = np.asarray(indptr, dtype=np.int32); indices = np.concatenate(idx).astype(np.int32)
    active = np.unique(indices)
    slot = np.full(I, -1, dtype=np.int32); slot[active] = np.arange(len(active))
    return indptr, indices, slot, len(active)


def test_enc_gather_xc_and_clear(ops):
    rng = np.random.RandomState(4)
    I, B = 3000, 40
    indptr, indices, slot, n_act = _xc_case(rng, I, B)
    W = dev((rng.randn(I, 600) * 0.05).astype(np.float32)).bfloat16()
    bq0 = torch.zeros(600, device="cuda")
    ld_xc = (n_act + 7) // 8 * 8 + 8
    max_nnz = int(np.diff(indptr).max())
    assert max_nnz > 128
    ws = torch.zeros(B, 600, device="cuda"); cn = torch.zeros(B, dtype=torch.int32, device="cuda")
    rows = np.repeat(np.arange(B), np.diff(indptr))
    for work in (None, dev(ops.enc_work_list(indptr))):
        xc = torch.zeros(B, ld_xc, device="cuda", dtype=torch.bfloat16)
        coef = torch.zeros(len(indices), device="cuda")
        h1 = torch.zeros(B, 600, device="cuda", dtype=torch.bfloat16)
        ops.enc_gather_fwd(dev(indptr), dev(indices), None, B, I, 100, W, bq0, 0.75, 77, 3, None, h1, coef, max_nnz, ws, cn,
                           slot_of_item=dev(slot), xc=xc, work=work)
        torch.cuda.synchronize()
        want = torch.zeros(B, ld_xc, device="cuda", dtype=torch.bfloat16)
        want[torch.from_numpy(rows).cuda(), torch.from_numpy(slot[indices].astype(np.int64)).cuda()] = coef.bfloat16()
        assert (coef == 0).any() and (coef != 0).any()
        assert torch.equal(xc, want), "xc must hold bf16(coef) at slot_of_item and 0 elsewhere"
        ops.enc_xc_clear(dev(indptr), dev(indices), B, len(indices), dev(slot), xc)
        torch.cuda.synchronize()
        assert (xc == 0).all()
        assert (ws == 0).all() and (cn == 0).all()


def test_enc_coef_scatter_matches_forward_and_clears(ops):
    """Data-parallel encoder gradient on one device (world 1, shard = whole catalog): ltg_enc_coef_scatter rebuilds from host tables
    (1/sqrt(deg) computed on the host) the coefficients ltg_enc_gather_fwd wrote (rsqrtf on the device): the same dropout pattern,
    values within one bf16 ulp; ltg_enc_coef_clear restores zeros."""
    eng = importlib.import_module("long-tail-gan_b200.engine")
    rng = np.random.RandomState(5)
    I, N, Bsz = 3000, 150, 64
    tabs = helpers.synth_side_tables(rng, N, I, mean_nnz=40)
    data = eng.TrainData(batch_size=Bsz, **tabs)
    tables = eng.build_dp_shard_tables(data, tabs["indptr"], tabs["indices"], world=1, rank=0, nb_per_rank=len(data.batches), R=I)
    W = dev((rng.randn(I, 600) * 0.05).astype(np.float32)).bfloat16()
    bq0 = torch.zeros(600, device="cuda")
    keep, seed = 0.75, 99
    step_dev = torch.tensor([6], dtype=torch.int32, device="cuda")
    for bi, bt in enumerate(data.batches):
        tb = tables[bi]
        B = bt["B"]
        assert tb["n_entries"] == bt["nnz"] and tb["n_active"] == bt["n_active"]
        ld_xc = (bt["n_active"] + 7) // 8 * 8
        xc = torch.zeros(Bsz, ld_xc, device="cuda", dtype=torch.bfloat16)
        h1 = torch.zeros(B, 600, device="cuda", dtype=torch.bfloat16)
        ws = torch.zeros(B, 600, device="cuda"); cn = torch.zeros(B, dtype=torch.int32, device="cuda")
        ops.enc_gather_fwd(data.indptr[bt["b0"]: bt["b0"] + B + 1], data.indices, None, B, I, bt["uid0"], W, bq0, keep, seed, 2, step_dev, h1,
                           data.coef, bt["max_nnz"], ws, cn, slot_of_item=bt["slot_of_item"], xc=xc)
        xc2 = torch.zeros_like(xc)
        ops.enc_coef_scatter(tb["e_row"], tb["e_item"], tb["e_slot"], tb["row_uid"], tb["row_rnorm"], tb["n_entries"], I, keep, seed, 2,
                             step_dev, xc2)
        torch.cuda.synchronize()
        assert torch.equal(xc != 0, xc2 != 0), "dropout pattern of the rebuilt coefficients"
        a, b = xc.double(), xc2.double()
        assert_within("coef rebuild batch %d" % bi, b, a, 2 * HALF_BF16 * torch.maximum(a.abs(), b.abs()) + TINY)   # one bf16 ulp
        ops.enc_coef_clear(tb["e_row"], tb["e_slot"], tb["n_entries"], xc2)
        torch.cuda.synchronize()
        assert (xc2 == 0).all()


# ------------------------------------------------------------------------------------------------------------------------------------
# ltg_sample_pairs_vals with the candidates' logits given explicitly == ltg_sample_pairs on the logits
# ------------------------------------------------------------------------------------------------------------------------------------
def test_sample_pairs_vals_equals_sample_pairs(ops):
    _lib = importlib.import_module("long-tail-gan_b200._lib")
    rng = np.random.RandomState(9)
    B, I = 300, 2000
    lg = dev((rng.randn(B, I) * 1.5).astype(np.float32)).bfloat16()
    niche = np.arange(I // 10, I)
    cand, n_s, pops = [], [], []
    for u in range(B):
        n = int(rng.randint(0, 12)) if u % 7 else 0
        own = np.sort(rng.choice(niche, n, replace=False))
        extra = rng.choice(np.setdiff1d(niche, own), max(2 * n, 10 - n), replace=False)
        cand.append(np.sort(np.concatenate([own, extra])).astype(np.int32)); n_s.append(n)
        pops.append(rng.choice(I // 10, size=rng.randint(1, 8), replace=False).astype(np.int32))
    cand_ptr = np.concatenate([[0], np.cumsum([len(c) for c in cand])]).astype(np.int32)
    samp_ptr = np.concatenate([[0], np.cumsum(n_s)]).astype(np.int32)
    pop_ptr = np.concatenate([[0], np.cumsum([len(p) for p in pops])]).astype(np.int32)
    valid = np.ones(I, dtype=np.uint8); valid[rng.choice(I, 40, replace=False)] = 0
    cand_items = np.concatenate(cand)
    K = int(samp_ptr[-1])
    order = dev(np.argsort(-np.diff(cand_ptr), kind="stable").astype(np.int32))
    args = [dev(cand_ptr), dev(cand_items), dev(samp_ptr), dev(pop_ptr), dev(np.concatenate(pops)), dev(valid)]
    outs = []
    for explicit in (False, True):
        si, sp, sv = [torch.full((K,), -7, dtype=torch.int32, device="cuda") for _ in range(3)]
        cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
        if explicit:
            rows = torch.from_numpy(np.repeat(np.arange(B), np.diff(cand_ptr))).cuda()
            vals = lg[rows, torch.from_numpy(cand_items.astype(np.int64)).cuda()].float().contiguous()
            ops.sample_pairs(None, B, I, 500, *args, 777, 3, None, si, sp, sv, cnt, int(np.diff(cand_ptr).max()), order, cand_vals=vals)
        else:
            p = _lib.ptr
            s = torch.cuda.current_stream().cuda_stream
            _lib.check(ops.lib().ltg_sample_pairs(p(lg), lg.stride(0), B, I, 500, *[p(a) for a in args], 777, 3, None, p(si), p(sp), p(sv),
                                                  p(cnt), int(np.diff(cand_ptr).max()), p(order), s))
        torch.cuda.synchronize()
        outs.append((si, sp, sv, cnt))
    for a, b in zip(*outs):
        assert torch.equal(a, b)
    assert (outs[0][0] >= 0).all() and 0 < outs[0][3].item() <= K


# ------------------------------------------------------------------------------------------------------------------------------------
# ltg_cast_bf16 == torch's round-to-nearest-even conversion
# ------------------------------------------------------------------------------------------------------------------------------------
def test_cast_bf16_bit_exact(ops):
    rows, cols, ld_src, ld_dst = 37, 203, 211, 216
    g = torch.Generator(device="cuda").manual_seed(11)
    src = torch.randn(rows, ld_src, device="cuda", generator=g) * 100
    flat = src[:, :cols].reshape(-1)
    special = torch.tensor([0.0, -0.0, float("inf"), float("-inf"), 1e-40, -1e-40, 3e-39, 1.17549435e-38, 3.4e38, -3.4e38],
                           device="cuda")
    flat = flat.clone()
    flat[: len(special)] = special
    # exact ties between two bf16 values, with an even and an odd lower neighbour (ties go to the even one), and just off the ties
    hi = torch.randint(0, 1 << 15, (400,), dtype=torch.int32, device="cuda", generator=g) | (0x3F << 8)
    ties = ((hi << 16) | 0x8000).view(torch.float32)
    near = ((hi << 16) | 0x8001).view(torch.float32)
    below = ((hi << 16) | 0x7FFF).view(torch.float32)
    n0 = len(special)
    flat[n0: n0 + 400] = ties; flat[n0 + 400: n0 + 800] = -near; flat[n0 + 800: n0 + 1200] = below
    src[:, :cols] = flat.view(rows, cols)
    dst = torch.full((rows, ld_dst), 5.0, device="cuda", dtype=torch.bfloat16)
    ops.cast_bf16(src, dst, rows, cols)
    torch.cuda.synchronize()
    want = src[:, :cols].bfloat16()
    assert torch.equal(dst[:, :cols].view(torch.int16), want.view(torch.int16))
    assert (dst[:, cols:] == 5.0).all()
    assert (want.view(torch.int16)[0, :2] == torch.tensor([0, -32768], dtype=torch.int16, device="cuda")).all()   # +0, -0 kept
