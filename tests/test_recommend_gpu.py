"""GPU checks of top-k recommendation: the ltg_topk_recommend kernel (staged and streaming paths) against a float64 oracle on the same
fp32 logits, GanEngine.recommend against GanEngine.evaluate and the oracle forward, the niche-only filter, the catalog-sharded engine,
and the recommend.py CLI on a short training run."""
import importlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
from scipy import sparse
from scipy.special import logsumexp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle import ltgan_oracle as orc  # noqa: E402
import helpers  # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden", "askubuntu_sample.npz")


@pytest.fixture(scope="module")
def ops():
    m = importlib.import_module("long-tail-gan_b200.ops")
    m.init()
    return m


@pytest.fixture(scope="module")
def eng():
    return importlib.import_module("long-tail-gan_b200.engine")


# ---------------------------------------------------------------------------------------------------------------------------------
# kernel
# ---------------------------------------------------------------------------------------------------------------------------------
def _scores(rows, n, rng, values=None):
    """[rows, n] fp32 logits in a device buffer whose row pitch exceeds n; the padding columns hold NaN (they must never be read)."""
    ld = (n + 7) // 8 * 8 + 8
    buf = torch.full((rows, ld), float("nan"), dtype=torch.float32, device="cuda")
    if values is None:
        base = np.linspace(-8.0, 8.0, n, dtype=np.float32)
        values = np.stack([base[rng.permutation(n)] + np.float32(0.01 * (r % 7)) for r in range(rows)])
    buf[:, :n] = torch.from_numpy(values).cuda()
    return buf, values


def _seen(rows, n, rng, max_len=200):
    ptr, idx = [0], []
    for r in range(rows):
        s = np.sort(rng.choice(n, rng.randint(0, max_len + 1) if r % 5 else 0, replace=False))
        idx.append(s); ptr.append(ptr[-1] + len(s))
    return np.asarray(ptr, dtype=np.int32), np.concatenate(idx).astype(np.int32)


def _run(ops, eng, buf, n, seen, allow, k, with_prob=True):
    rows = buf.shape[0]
    dev = lambda a: torch.as_tensor(a).cuda()  # noqa: E731
    sp, si = (None, None) if seen is None else (dev(seen[0]), dev(seen[1] if len(seen[1]) else np.zeros(1, np.int32)))
    bits = None if allow is None else dev(eng.allow_bits(allow, n).view(np.int32))
    idx = torch.empty(rows, k, dtype=torch.int32, device="cuda")
    logit = torch.empty(rows, k, dtype=torch.float32, device="cuda")
    prob = torch.empty(rows, k, dtype=torch.float32, device="cuda") if with_prob else None
    lse = torch.empty(rows, dtype=torch.float32, device="cuda")
    ops.topk_recommend(buf, rows, n, sp, si, bits, k, idx, logit, prob, lse)
    torch.cuda.synchronize()
    return idx.cpu().numpy(), logit.cpu().numpy(), (prob.cpu().numpy() if with_prob else None), lse.cpu().numpy()


def _oracle(values, seen, allow, k):
    """float64: eligible items ordered by (logit desc, id asc), -1 padded; lse over every column."""
    rows, n = values.shape
    x = values.astype(np.float64)
    lse = logsumexp(x, axis=1)
    base = np.ones(n, dtype=bool)
    if allow is not None:
        base[:] = False; base[np.asarray(allow)] = True
    out = np.full((rows, k), -1, dtype=np.int64)
    for r in range(rows):
        el = base.copy()
        if seen is not None:
            el[seen[1][seen[0][r]: seen[0][r + 1]]] = False
        ids = np.nonzero(el)[0]
        top = ids[np.lexsort((ids, -x[r, ids]))[:k]]
        out[r, :len(top)] = top
    return out, lse


def _check(got, values, want_idx, lse64):
    idx, logit, prob, lse = got
    assert np.array_equal(idx, want_idx)
    valid = idx >= 0
    r, j = np.nonzero(valid)
    assert np.array_equal(logit[r, j].view(np.uint32), values[r, idx[r, j]].view(np.uint32))        # bit-equal to the input
    assert np.all(np.isneginf(logit[~valid]))
    assert np.abs(lse.astype(np.float64) - lse64).max() <= 1e-5
    if prob is not None:
        p64 = np.exp(values[r, idx[r, j]].astype(np.float64) - lse64[r])
        assert np.all(np.abs(prob[r, j] - p64) <= 1e-5 * p64)
        assert np.all(prob[~valid] == 0.0)


@pytest.mark.parametrize("n", [1000, 20108, 49152])
def test_kernel_staged_matches_oracle(ops, eng, n):
    rng = np.random.RandomState(n)
    rows = 300
    buf, values = _scores(rows, n, rng)
    assert all(len(np.unique(values[r])) == n for r in range(0, rows, 37))     # tie-free
    seen = _seen(rows, n, rng)
    allow30 = np.sort(rng.choice(n, int(0.3 * n), replace=False))
    for allow in (None, allow30):
        want, lse64 = _oracle(values, seen, allow, 128)
        for k in (1, 100, 128):
            _check(_run(ops, eng, buf, n, seen, allow, k), values, want[:, :k], lse64)


def test_kernel_streaming_matches_oracle(ops, eng):
    n, rows = 100003, 64
    rng = np.random.RandomState(7)
    buf, values = _scores(rows, n, rng)
    seen = _seen(rows, n, rng, max_len=2000)
    allow30 = np.sort(rng.choice(n, int(0.3 * n), replace=False))
    for allow in (None, allow30):
        want, lse64 = _oracle(values, seen, allow, 128)
        for k in (1, 100, 128):
            _check(_run(ops, eng, buf, n, seen, allow, k, with_prob=(k != 100)), values, want[:, :k], lse64)


@pytest.mark.parametrize("n", [1000, 20108, 100003])
def test_kernel_ties_padding_and_filters(ops, eng, n):
    """Constant rows and rows of equal-score blocks list the lowest eligible ids in order (a constant 20 k-item row overflows the
    pre-filter's candidate list and takes the full-row selection); rows with fewer eligible items than k pad with (-1, -inf, 0); no
    excluded id is listed; the log-sum-exp does not depend on the filters."""
    rng = np.random.RandomState(n + 1)
    rows = 6
    vals = np.empty((rows, n), dtype=np.float32)
    vals[0] = 0.5
    vals[1] = -3.0
    vals[2] = np.floor(rng.rand(n) * 8).astype(np.float32) / 4           # eight values, blocks of equal scores
    nb = (n + 99) // 100
    vals[3] = (np.repeat(np.arange(nb, dtype=np.float32), 100)[:n][::-1] * np.float32(8.0 / nb)).astype(np.float32)   # descending blocks of 100
    vals[4] = rng.randn(n).astype(np.float32)
    vals[5] = 0.0
    buf, _ = _scores(rows, n, rng, vals)
    seen = _seen(rows, n, rng)
    allow30 = np.sort(rng.choice(n, int(0.3 * n), replace=False))
    plain = _run(ops, eng, buf, n, None, None, 128)
    for allow in (None, allow30):
        want, lse64 = _oracle(vals, seen, allow, 128)
        got = _run(ops, eng, buf, n, seen, allow, 128)
        _check(got, vals, want, lse64)
        assert np.array_equal(got[3].view(np.uint32), plain[3].view(np.uint32))      # filters do not change the normaliser
        for r in range(rows):
            listed = got[0][r][got[0][r] >= 0]
            assert not np.isin(listed, seen[1][seen[0][r]: seen[0][r + 1]]).any()
            if allow is not None:
                assert np.isin(listed, allow).all()
    for r in (0, 1, 5):                                                               # constant rows: lowest eligible ids
        el = np.setdiff1d(np.arange(n), seen[1][seen[0][r]: seen[0][r + 1]])
        assert np.array_equal(plain[0][r], np.arange(128)) and np.array_equal(_run(ops, eng, buf, n, seen, None, 128)[0][r], el[:128])
    # ten allowed items, four of them (and many others) seen: six eligible, the rest padding; a row with all ten seen lists nothing
    allow10 = np.sort(rng.choice(n, 10, replace=False))
    others = np.setdiff1d(np.arange(n), allow10)
    sp, si = [0], []
    for r in range(rows):
        s = np.union1d(rng.choice(others, 300, replace=False), allow10 if r == 5 else allow10[:4]).astype(np.int32)
        si.append(s); sp.append(sp[-1] + len(s))
    seen10 = (np.asarray(sp, dtype=np.int32), np.concatenate(si))
    got = _run(ops, eng, buf, n, seen10, allow10, 100)
    want, lse64 = _oracle(vals, seen10, allow10, 100)
    _check(got, vals, want, lse64)
    assert ((got[0] >= 0).sum(1) == [6, 6, 6, 6, 6, 0]).all()
    assert np.all(got[0][:, 6:] == -1) and np.all(np.isneginf(got[1][:, 6:])) and np.all(got[2][:, 6:] == 0.0)
    assert np.array_equal(got[3].view(np.uint32), plain[3].view(np.uint32))


def test_kernel_rejects_bad_arguments(ops, eng):
    buf, _ = _scores(2, 100, np.random.RandomState(0))
    lib_err = importlib.import_module("long-tail-gan_b200._lib").LtgError
    for k in (0, 129):
        with pytest.raises(lib_err):
            _run(ops, eng, buf, 100, None, None, k)


# ---------------------------------------------------------------------------------------------------------------------------------
# engine
# ---------------------------------------------------------------------------------------------------------------------------------
I, N_TRAIN, BATCH, SEED = 1000, 230, 100, 20240607


@pytest.fixture(scope="module")
def setup(ops, eng):
    gen = importlib.import_module("long-tail-gan_b200.generator")
    dis = importlib.import_module("long-tail-gan_b200.discriminator")
    tabs = helpers.synth_side_tables(np.random.RandomState(5), N_TRAIN, I)
    vae = gen.MultiVAE([200, 600, I], lam=0.0, random_seed=98765)
    params = orc.init_vae_params(I, seed=98765)
    params[3] = params[3] * 3.0
    vae.set_params(params); vae.reset_optimizer()
    disc = dis.Discriminator(I, I, 100, 150, 250, 300, seed=1)
    E, dparams = orc.init_disc_params(I, 100, 150, 250, 300, seed=77)
    disc.set_params(E, dparams)
    data = eng.TrainData(batch_size=BATCH, **tabs)
    engine = eng.GanEngine(vae, disc, data.max_B, data.max_P, seed=SEED, lr=1e-4, lam=1.0, use_graphs=False, max_active=data.max_active)
    engine.run_phase_a(data, 0); engine.run_d_step(data, 0); engine.run_g_step(data, 0)     # a non-zero rng step and trained weights
    # fold-in rows of 6-40 items: under one 128-nonzero encoder chunk, so the scores are free of float atomics (deterministic)
    rng = np.random.RandomState(21)
    tr_ptr, tr_idx, te_ptr, te_idx = [0], [], [0], []
    for u in range(150):
        items = rng.choice(I, rng.randint(6, 41), replace=False)
        cut = 0 if u % 17 == 3 else max(1, len(items) // 5)
        te, tr = np.sort(items[:cut]), np.sort(items[cut:])
        tr_idx.append(tr); tr_ptr.append(tr_ptr[-1] + len(tr)); te_idx.append(te); te_ptr.append(te_ptr[-1] + len(te))
    ev = (np.asarray(tr_ptr), np.concatenate(tr_idx), np.asarray(te_ptr), np.concatenate(te_idx))
    return dict(vae=vae, engine=engine, ev=ev)


def _pred_from_lists(items, n_items):
    """A score matrix whose top-k under eval_functions.py is exactly the given ordered lists."""
    pred = np.full((items.shape[0], n_items), -np.inf)
    k = items.shape[1]
    for r in range(items.shape[0]):
        pred[r, items[r]] = np.arange(k, 0, -1)
    return pred


def test_recommend_ranks_what_evaluate_ranks_and_leaves_the_engine_state(setup):
    engine = setup["engine"]
    tr_ptr, tr_idx, te_ptr, te_idx = setup["ev"]
    words0, scal0 = engine.words.clone(), engine.scal_all.clone()
    rec = engine.recommend(tr_ptr, tr_idx, k=100, keep=None, uid_start=5000, batch=64)
    torch.cuda.synchronize()
    assert torch.equal(engine.words, words0) and torch.equal(engine.scal_all, scal0)
    got = engine.evaluate(tr_ptr, tr_idx, te_ptr, te_idx, k=100, recall_ks=(20, 50), uid_start=5000, batch=64)   # keep_vae: dropout live
    assert not torch.equal(engine.words, words0)
    n = len(tr_ptr) - 1
    held = sparse.csr_matrix((np.ones(len(te_idx)), te_idx, te_ptr), shape=(n, I))
    assert rec["items"].shape == (n, 100) and (rec["items"] >= 0).all()
    for r in range(n):
        assert not np.isin(rec["items"][r], tr_idx[tr_ptr[r]: tr_ptr[r + 1]]).any()
    pred = _pred_from_lists(rec["items"], I)
    nd = orc.ndcg_binary_at_k_batch(pred, held, k=100)
    r20, _ = orc.recall_at_k_batch(pred, held, k=20)
    r50, _ = orc.recall_at_k_batch(pred, held, k=50)
    assert len(nd) == len(got["ndcg@100"]) and len(r20) == len(got["recall@20"])
    assert np.abs(np.asarray(nd) - got["ndcg@100"]).max() <= 1e-12
    assert np.abs(np.asarray(r20) - got["recall@20"]).max() <= 1e-12
    assert np.abs(np.asarray(r50) - got["recall@50"]).max() <= 1e-12


def test_recommend_probabilities_match_oracle_forward(setup):
    engine, vae = setup["engine"], setup["vae"]
    tr_ptr, tr_idx = setup["ev"][:2]
    rec = engine.recommend(tr_ptr, tr_idx, k=100)               # keep = 1.0: no dropout
    n = len(tr_ptr) - 1
    params = [p.detach().cpu().float().contiguous() for p in vae.params]
    X = torch.from_numpy(helpers.dense_rows(tr_ptr, tr_idx, 0, n, I))
    ref = orc.vae_forward(params, X, None, 1.0, None, 0.0, 1.0)["probs"].numpy()
    p = rec["probs"]
    want = np.take_along_axis(ref, rec["items"], 1)
    assert np.all(np.abs(p - want) <= 3e-2 * ref.max(1, keepdims=True))
    assert np.all(np.diff(p, axis=1) <= 0)
    assert np.all(p.sum(1) <= 1.0) and np.all(p > 0)
    assert rec["lse"].shape == (n,) and np.isfinite(rec["lse"]).all()


def test_niche_only_lists(setup):
    engine = setup["engine"]
    tr_ptr, tr_idx = setup["ev"][:2]
    niche = np.sort(np.random.RandomState(99).choice(I, 300, replace=False))
    full = engine.recommend(tr_ptr, tr_idx, k=100)
    mask = np.zeros(I, dtype=bool); mask[niche] = True
    for allow in (niche, mask):
        nic = engine.recommend(tr_ptr, tr_idx, k=100, allow=allow)
        assert np.isin(nic["items"], niche).all()
        assert np.array_equal(nic["lse"].view(np.uint32), full["lse"].view(np.uint32))
        for r in range(len(tr_ptr) - 1):
            f_items, f_probs = full["items"][r], full["probs"][r]
            inset = np.isin(f_items, niche)
            pre = f_items[inset]
            assert np.array_equal(nic["items"][r][:len(pre)], pre)                     # the unfiltered list's niche items, a prefix
            assert np.array_equal(nic["probs"][r][:len(pre)].view(np.uint32), f_probs[inset].view(np.uint32))


# ---------------------------------------------------------------------------------------------------------------------------------
# catalog-sharded engine
# ---------------------------------------------------------------------------------------------------------------------------------
def test_catalog_sharded_one_shard(ops):
    vrc = _load_tool()
    res = vrc.run_check(2400, 96, 0, 1)
    _check_sharded(res)


def _load_tool():
    import importlib.util
    spec = importlib.util.spec_from_file_location("vp_recommend_check", os.path.join(ROOT, "tools", "vp_recommend_check.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _check_sharded(res):
    assert res["items_equal_evaluate_topk"], res
    assert res["words_unchanged"], res
    assert res["max_prob_diff_rel"] < 3e-2, res
    assert res["niche_only_ok"], res


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_catalog_sharded_two_shards(tmp_path):
    out = str(tmp_path / "vpr.json")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port",
           "29623", os.path.join(ROOT, "tools", "vp_recommend_check.py"), out]
    r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    res = json.load(open(out))
    assert res["world"] == 2
    _check_sharded(res)


# ---------------------------------------------------------------------------------------------------------------------------------
# CLI
# ---------------------------------------------------------------------------------------------------------------------------------
def _read_tsv(path):
    lines = open(path).read().splitlines()
    assert lines[0] == "uid\trank\tsid\tprob"
    rows = [l.split("\t") for l in lines[1:]]
    return (np.asarray([int(r[0]) for r in rows]), np.asarray([int(r[1]) for r in rows]), np.asarray([int(r[2]) for r in rows]),
            np.asarray([float(r[3]) for r in rows]))


def test_recommend_cli_after_training(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    train = importlib.import_module("long-tail-gan_b200.train")
    rec = importlib.import_module("long-tail-gan_b200.recommend")
    cfg = dict(h0_size=100, h1_size=150, h2_size=250, h3_size=300, NUM_EPOCH=8, NUM_SUB_EPOCHS=1, BATCH_SIZE=100, DISPLAY_ITER=50,
               LEARNING_RATE=1e-3, to_restore=0, model_name="LT_GAN", dataset=GOLD, GANLAMBDA=1.0)
    train.train_GAN(max_epochs=2, quiet=True, seed=3, **cfg)
    ck = os.path.join("chkpt", "askubuntu_sample_LT_GAN_1.0", "model_1")
    g = np.load(GOLD)
    ip, idx, start = g["tst_tr_indptr"].astype(np.int64), g["tst_tr_indices"].astype(np.int64), int(g["tst_start"])
    niche = set(g["niche_tags"].tolist())
    for niche_only in (False, True):
        out = str(tmp_path / ("rec_niche.tsv" if niche_only else "rec.tsv"))
        rec.main([GOLD, ck, "--split", "test", "--k", "20", "--out", out] + (["--niche-only"] if niche_only else []))
        uid, rank, sid, prob = _read_tsv(out)
        users, first = np.unique(uid, return_index=True)
        assert len(users) == len(ip) - 1 and users.min() == start and users.max() == start + len(ip) - 2
        assert np.all(np.diff(uid) >= 0)                                                  # one block per user
        bounds = list(first) + [len(uid)]
        for b, u in enumerate(users):
            s = slice(bounds[b], bounds[b + 1])
            r = u - start
            assert 1 <= bounds[b + 1] - bounds[b] <= 20
            assert np.array_equal(rank[s], np.arange(1, bounds[b + 1] - bounds[b] + 1))
            assert np.all(np.diff(prob[s]) <= 0)
            assert not np.isin(sid[s], idx[ip[r]: ip[r + 1]]).any()
            if niche_only:
                assert all(int(i) in niche for i in sid[s])
        assert np.all((prob > 0) & (prob <= 1))
