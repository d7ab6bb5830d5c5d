"""GPU checks of long-tail evaluation: ltg_topk_longtail against ltg_topk_metrics (bit-identical shared outputs) and a float64 NumPy
oracle on both kernel paths, GanEngine.evaluate(niche=..., item_pop=...) against the lists of GanEngine.recommend on the bundled
fixture and at the ML-20M shape, and the train.py / test.py CLIs."""
import ctypes
import importlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
pytestmark = pytest.mark.gpu
GOLD = os.path.join(ROOT, "tests", "golden", "askubuntu_sample.npz")
PKG = "long-tail-gan_b200"


@pytest.fixture(scope="module")
def ops():
    m = importlib.import_module(PKG + ".ops")
    m.init()
    return m


@pytest.fixture(scope="module")
def eng():
    return importlib.import_module(PKG + ".engine")


# ---------------------------------------------------------------------------------------------------------------------------------
# kernel
# ---------------------------------------------------------------------------------------------------------------------------------
def _case(n, rows, dtype, seed):
    """Scores [rows, n] (fp32 or bf16, row pitch > n) with deliberate ties, seen lists (some leaving fewer than 128 eligible items),
    held-out lists (some empty, many drawn from the row's best items), a niche mask and popularity counts up to 2**20."""
    rng = np.random.RandomState(seed)
    x = rng.randn(rows, n).astype(np.float32)
    x[1::7] = np.round(x[1::7] * 2) / 2 + np.float32(0)   # a handful of values: long runs of equal scores (+ 0: no -0.0, which ranks
                                                          # below +0.0 on the device and equal to it in NumPy)
    x[2::7] = 0.25                                        # constant rows
    x[3::7, : n // 2] = x[3::7, n // 2: 2 * (n // 2)]     # pairs of equal scores
    ld = (n + 7) // 8 * 8 + 8
    buf = torch.full((rows, ld), float("nan"), dtype=torch.float32, device="cuda")
    buf[:, :n] = torch.from_numpy(x).cuda()
    if dtype == torch.bfloat16:
        buf = buf.to(torch.bfloat16)
    vals = buf[:, :n].float().cpu().numpy()               # exactly the values the kernel ranks
    seen_ptr, seen = [0], []
    for r in range(rows):
        m = n - 60 if r % 10 == 4 else rng.randint(0, 200)
        s = np.sort(rng.choice(n, m, replace=False))
        seen.append(s); seen_ptr.append(seen_ptr[-1] + m)
    held_ptr, held = [0], []
    for r in range(rows):
        if r % 9 == 5:
            h = np.zeros(0, np.int64)
        else:
            best = np.argsort(-vals[r], kind="stable")[:160]
            h = np.union1d(rng.choice(best, rng.randint(1, 40), replace=False), rng.choice(n, rng.randint(0, 20), replace=False))
        held.append(h); held_ptr.append(held_ptr[-1] + len(h))
    niche = rng.rand(n) < 0.4
    pop = rng.randint(0, 2 ** 20 + 1, n)
    pop[rng.choice(n, 50, replace=False)] = 2 ** 20
    return dict(buf=buf, vals=vals, seen=(np.asarray(seen_ptr, np.int32), np.concatenate(seen).astype(np.int32)),
                held=(np.asarray(held_ptr, np.int32), np.concatenate(held).astype(np.int32)), niche=niche, pop=pop.astype(np.int64))


def _oracle_lists(c, k):
    """float64: seen items as -inf, order (score desc, id asc), first min(k, n) ids of every row."""
    vals, (sp, si) = c["vals"], c["seen"]
    rows, n = vals.shape
    ids = np.arange(n)
    out = np.empty((rows, min(k, n)), dtype=np.int64)
    for r in range(rows):
        x = vals[r].astype(np.float64)
        x[si[sp[r]: sp[r + 1]]] = -np.inf
        out[r] = np.lexsort((ids, -x))[: min(k, n)]
    return out


def _oracle_counts(c, lists, rks):
    hp, hi = c["held"]
    rows, kk = lists.shape
    hit = np.zeros((rows, kk), dtype=bool)
    for r in range(rows):
        hit[r] = np.isin(lists[r], hi[hp[r]: hp[r + 1]])
    nh = hit & c["niche"][lists]
    w = 1.0 / np.log2(np.arange(kk) + 2.0)
    return dict(dcg_niche=(nh * w).sum(1), hits_niche=np.asarray([nh[:, :rk].sum(1) for rk in rks], dtype=np.int64).reshape(len(rks), rows).T,
                n_niche_top=c["niche"][lists].sum(1), pop_sum=c["pop"][lists].sum(1),
                rec_count=np.bincount(lists[np.diff(hp) > 0].reshape(-1), minlength=c["vals"].shape[1]))


def _launch(ops, eng, c, k, rks, longtail, r0, r1, rec_count=None):
    """One launch over rows [r0, r1) (row slices as GanEngine.evaluate takes them: absolute CSR offsets)."""
    dev = lambda a: torch.as_tensor(a).cuda()  # noqa: E731
    n = c["vals"].shape[1]
    B = r1 - r0
    sp, si = dev(c["seen"][0]), dev(c["seen"][1])
    hp, hi = dev(c["held"][0]), dev(c["held"][1])
    idx = torch.full((B, k), -7, dtype=torch.int32, device="cuda")
    dcg = torch.full((B,), float("nan"), dtype=torch.float64, device="cuda")
    hits = torch.full((B, max(1, len(rks))), -7, dtype=torch.int32, device="cuda")
    out = dict(idx=idx, dcg=dcg, hits=hits)
    if not longtail:
        ops.topk_metrics(c["buf"][r0:r1], B, n, sp[r0:], si, hp[r0:], hi, k, rks, idx, dcg, hits)
    else:
        out.update(dcg_niche=torch.full((B,), float("nan"), dtype=torch.float64, device="cuda"),
                   hits_niche=torch.full((B, max(1, len(rks))), -7, dtype=torch.int32, device="cuda"),
                   n_niche_top=torch.full((B,), -7, dtype=torch.int32, device="cuda"),
                   pop_sum=torch.full((B,), -7, dtype=torch.int64, device="cuda"))
        ops.topk_longtail(c["buf"][r0:r1], B, n, sp[r0:], si, hp[r0:], hi, k, rks, idx, dcg, hits,
                          dev(eng.allow_bits(c["niche"], n).view(np.int32)), dev(c["pop"].astype(np.int32)), out["dcg_niche"],
                          out["hits_niche"], out["n_niche_top"], out["pop_sum"], rec_count)
    torch.cuda.synchronize()
    res = {key: v.cpu().numpy() for key, v in out.items()}
    res["hits"] = np.ascontiguousarray(res["hits"][:, :len(rks)])
    if longtail:
        res["hits_niche"] = np.ascontiguousarray(res["hits_niche"][:, :len(rks)])
    return res


def _rk_sets(k):
    return [tuple(min(k, r) for r in (5, 20, 50, 128)[:m]) for m in range(5)]


def _check_kernel(ops, eng, c):
    rows, n = c["vals"].shape
    lists128 = _oracle_lists(c, 128)
    half = rows // 2
    for k in (1, 100, 128):
        kk = min(k, n)
        lists = lists128[:, :kk]
        for rks in _rk_sets(k):
            base = _launch(ops, eng, c, k, rks, False, 0, rows)
            rec = torch.zeros(n, dtype=torch.int32, device="cuda")
            a = _launch(ops, eng, c, k, rks, True, 0, half, rec)          # two launches accumulate into one rec_count
            b = _launch(ops, eng, c, k, rks, True, half, rows, rec)
            got = {key: np.concatenate([a[key], b[key]]) for key in a}
            for key in ("idx", "dcg", "hits"):                          # bit-identical to ltg_topk_metrics
                assert np.array_equal(got[key].view(np.uint8), base[key].view(np.uint8)), (n, k, rks, key)
            assert np.array_equal(got["idx"][:, :kk], lists), (n, k)
            want = _oracle_counts(c, lists, rks)
            assert np.abs(got["dcg_niche"] - want["dcg_niche"]).max() <= 1e-12
            for key in ("hits_niche", "n_niche_top", "pop_sum"):
                assert np.array_equal(got[key], want[key]), (n, k, rks, key)
            assert np.array_equal(rec.cpu().numpy(), want["rec_count"]), (n, k, rks)
    assert (want["n_niche_top"] > 0).any() and (want["dcg_niche"] > 0).any()       # the cases exercise what they check
    assert (np.diff(c["held"][0]) == 0).any() and (c["pop"][lists128] == 2 ** 20).any()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("n", [1000, 20108, 49152])
def test_kernel_staged_matches_metrics_and_oracle(ops, eng, n, dtype):
    _check_kernel(ops, eng, _case(n, 120, dtype, seed=n))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_kernel_streaming_matches_metrics_and_oracle(ops, eng, dtype):
    _check_kernel(ops, eng, _case(100003, 40, dtype, seed=3))


def test_kernel_rejects_missing_long_tail_pointers(ops):
    """Every long-tail pointer is required: a call with one of them NULL returns an argument error before any launch."""
    lib = importlib.import_module(PKG + "._lib").load()
    n, rows = 64, 2
    t = lambda dt, m: torch.zeros(m, dtype=dt, device="cuda")  # noqa: E731
    scores = t(torch.float32, rows * n)
    hp, hi = torch.zeros(rows + 1, dtype=torch.int32, device="cuda"), t(torch.int32, 1)
    rk = np.asarray([5], dtype=np.int32)
    dcg, hits = t(torch.float64, rows), t(torch.int32, rows)
    bufs = [t(torch.int32, 2), t(torch.int32, n), t(torch.float64, rows), t(torch.int32, rows), t(torch.int32, rows), t(torch.int64, rows),
            t(torch.int32, n)]

    def call(ptrs):
        return lib.ltg_topk_longtail(scores.data_ptr(), 0, n, rows, n, None, None, hp.data_ptr(), hi.data_ptr(), 10, rk.ctypes.data, 1,
                                     None, dcg.data_ptr(), hits.data_ptr(), *ptrs, torch.cuda.current_stream().cuda_stream)
    assert call([b.data_ptr() for b in bufs]) == 0
    torch.cuda.synchronize()
    for j in range(len(bufs)):
        ptrs = [b.data_ptr() for b in bufs]
        ptrs[j] = None
        assert call(ptrs) != 0
        assert b"bad argument" in ctypes.string_at(lib.ltg_last_error())


# ---------------------------------------------------------------------------------------------------------------------------------
# engine
# ---------------------------------------------------------------------------------------------------------------------------------
def _oracle_keys(lists, te_ptr, te_idx, niche, pop, k, recall_ks):
    """The long-tail keys of evaluate from explicit lists [N, kk], float64, user by user."""
    n_items = len(niche)
    kk = lists.shape[1]
    out = {key: [] for key in ["niche_ndcg@%d" % k] + ["niche_recall@%d" % rk for rk in recall_ks] + ["niche_share@%d" % k, "avg_pop@%d" % k]}
    c = np.zeros(n_items, dtype=np.int64)
    for u in range(len(te_ptr) - 1):
        H = set(te_idx[te_ptr[u]: te_ptr[u + 1]].tolist())
        if not H:
            continue
        L = lists[u].tolist()
        for i in L:
            c[i] += 1
        out["niche_share@%d" % k].append(sum(bool(niche[i]) for i in L) / kk)
        out["avg_pop@%d" % k].append(sum(int(pop[i]) for i in L) / kk)
        HN = {i for i in H if niche[i]}
        if not HN:
            continue
        dcg = sum(1.0 / np.log2(j + 2) for j, i in enumerate(L) if i in HN)
        idcg = sum(1.0 / np.log2(j + 2) for j in range(min(len(HN), k)))
        out["niche_ndcg@%d" % k].append(dcg / idcg)
        for rk in recall_ks:
            out["niche_recall@%d" % rk].append(sum(1 for i in L[:rk] if i in HN) / min(rk, len(HN)))
    cs = np.sort(c)
    num = sum((2 * j - n_items - 1) * int(cs[j - 1]) for j in range(1, n_items + 1))
    out["coverage@%d" % k] = np.count_nonzero(c) / n_items
    out["niche_coverage@%d" % k] = np.count_nonzero(c[niche]) / int(niche.sum())
    out["gini@%d" % k] = float(num) / float(n_items * int(c.sum())) if c.sum() else 0.0
    return out


def _compare_engine(e, tr, te, niche, pop, batch=None):
    plain = e.evaluate(tr[0], tr[1], te[0], te[1], k=100, recall_ks=(20, 50), keep=1.0, batch=batch)
    got = e.evaluate(tr[0], tr[1], te[0], te[1], k=100, recall_ks=(20, 50), keep=1.0, batch=batch, niche=niche, item_pop=pop)
    for key, v in plain.items():
        assert got[key] == v, key                                        # existing keys: the same values
    rec = e.recommend(tr[0], tr[1], k=100, keep=1.0, batch=batch)          # keep = 1.0: the lists evaluate ranks
    mask = np.zeros(e.I, dtype=bool); mask[niche] = True
    want = _oracle_keys(rec["items"], np.asarray(te[0], np.int64), np.asarray(te[1], np.int64), mask, pop, 100, (20, 50))
    assert set(got) == set(plain) | set(want)
    for key, v in want.items():
        if isinstance(v, list):
            assert len(got[key]) == len(v), key
            assert len(v) == 0 or np.abs(np.asarray(got[key]) - np.asarray(v)).max() <= 1e-12, key
        else:
            assert got[key] == v, (key, got[key], v)
    return got


def _cap_rows(ptr, idx, cap=128):
    """Fold-in rows cut to their first `cap` items: one encoder chunk per row, so the scores carry no float atomics and two passes over
    the same users rank bit-identical scores."""
    ptr = np.asarray(ptr, np.int64)
    keep = np.concatenate([np.arange(a, min(b, a + cap)) for a, b in zip(ptr[:-1], ptr[1:])])
    return np.concatenate([[0], np.cumsum(np.minimum(np.diff(ptr), cap))]), np.asarray(idx)[keep].astype(np.int32)


def test_evaluate_long_tail_on_fixture(ops, eng):
    gen = importlib.import_module(PKG + ".generator"); dis = importlib.import_module(PKG + ".discriminator")
    g = np.load(GOLD)
    I = int(g["n_items"])
    vae = gen.MultiVAE([200, 600, I], lam=0.0, random_seed=98765); vae.init_weights(98765)
    disc = dis.Discriminator(I, I, 100, 150, 250, 300, seed=5)
    e = eng.GanEngine(vae, disc, 512, 1, seed=77, use_graphs=False, max_active=1)
    tr = _cap_rows(g["vad_tr_indptr"], g["vad_tr_indices"])
    te = (g["vad_te_indptr"].astype(np.int64), g["vad_te_indices"].astype(np.int32))
    pop = np.bincount(g["train_indices"].astype(np.int64), minlength=I)
    got = _compare_engine(e, tr, te, np.sort(g["niche_tags"].astype(np.int64)), pop, batch=1500)   # several batches
    assert 0 < len(got["niche_ndcg@100"]) < len(got["ndcg@100"]) == len(got["niche_share@100"])
    with pytest.raises(ValueError):
        e.evaluate(tr[0], tr[1], te[0], te[1], niche=[I], item_pop=pop)
    with pytest.raises(ValueError):
        e.evaluate(tr[0], tr[1], te[0], te[1], niche=[1], item_pop=-pop)


def test_evaluate_long_tail_ml20m_shape(ops, eng):
    """10,000 users of a 20,108-item catalog: three 3,334-row batches (staged kernel) accumulate one rec_count."""
    syn = importlib.import_module(PKG + ".synthetic")
    gen = importlib.import_module(PKG + ".generator"); dis = importlib.import_module(PKG + ".discriminator")
    _, I, deg = syn.CONFIGS["ml20m"]
    tr_p, tr_i, te_p, te_i = syn.make_eval_split(10000, I, deg)
    tr = _cap_rows(tr_p, tr_i)
    vae = gen.MultiVAE([200, 600, I], lam=0.0, random_seed=98765); vae.init_weights(98765)
    disc = dis.Discriminator(I, I, 100, 150, 250, 300, seed=4242)
    e = eng.GanEngine(vae, disc, 500, 1, seed=2026, use_graphs=False, max_active=1)
    assert e._eval_batch(10000, None) == 3334
    rng = np.random.RandomState(11)
    niche = np.sort(rng.choice(I, I // 3, replace=False))
    pop = np.bincount(syn.make_interactions(20000, I, deg, 99)[1].astype(np.int64), minlength=I)
    got = _compare_engine(e, tr, (te_p, te_i), niche, pop)
    assert 0 < got["gini@100"] < 1 and 0 < got["coverage@100"] <= 1


# ---------------------------------------------------------------------------------------------------------------------------------
# CLI
# ---------------------------------------------------------------------------------------------------------------------------------
LT_FIELDS = ["niche_ndcg", "niche_r20", "niche_r50", "niche_share", "avg_pop", "coverage", "niche_coverage", "gini"]


def test_cli_long_tail(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    train = importlib.import_module(PKG + ".train")
    test = importlib.import_module(PKG + ".test")
    cfg = dict(h0_size=100, h1_size=150, h2_size=250, h3_size=300, NUM_EPOCH=8, NUM_SUB_EPOCHS=1, BATCH_SIZE=100, DISPLAY_ITER=50,
               LEARNING_RATE=1e-3, to_restore=0, model_name="LT_GAN", dataset=GOLD, GANLAMBDA=1.0)
    h = train.train_GAN(max_epochs=2, quiet=True, seed=3, **cfg)["history"]
    assert len(h) == 2
    for rec in h:
        assert all(f in rec and np.isfinite(rec[f]) for f in LT_FIELDS), rec
        assert all(0 <= rec[f] <= 1 for f in ("niche_ndcg", "niche_r20", "niche_r50", "niche_share", "coverage", "niche_coverage")), rec
        assert 0 <= rec["gini"] < 1 and rec["avg_pop"] > 0, rec
    ck = os.path.join(str(tmp_path), "chkpt", "askubuntu_sample_LT_GAN_1.0", "model_1")
    # the test split with fold-in rows of at most 128 items (scores free of float atomics: both runs rank identical scores)
    g = dict(np.load(GOLD))
    g["tst_tr_indptr"], g["tst_tr_indices"] = _cap_rows(g["tst_tr_indptr"], g["tst_tr_indices"])
    data = str(tmp_path / "fixture_cap128.npz")
    np.savez(data, **g)
    with open(os.path.join(ROOT, PKG, "config.ini")) as src, open(tmp_path / "config.ini", "w") as dst:
        dst.write(src.read())
    script = os.path.join(ROOT, PKG, "test.py")
    runs = [subprocess.run([sys.executable, script, data, ck] + extra, cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
            for extra in ([], ["--long-tail"])]
    for r in runs:
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    plain, lt = runs[0].stdout.splitlines(), runs[1].stdout.splitlines()
    assert lt[:-1] == plain and len(plain[-1].split("\t")) == 3       # the reference's line unchanged, then one more line
    fields = lt[-1].split("\t")
    assert len(fields) == 8
    res = test.test_GAN(output_path=ck, quiet=True, long_tail=True, **dict(cfg, dataset=data))
    assert len(res) == 4 and list(res[3]) == LT_FIELDS
    assert [float(f) for f in fields] == list(res[3].values())
    assert test.test_GAN(output_path=ck, quiet=True, **dict(cfg, dataset=data))[:3] == res[:3]
