"""CPU checks of the recommendation host layer: the allow-set -> bitmap packing of ltg_topk_recommend (whole catalog and catalog
shards), the TSV writer of recommend.py, and the fold-in / niche-set loading of every --split from the committed fixture and from a
dataset directory."""
import importlib
import io
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "askubuntu_sample.npz")


@pytest.fixture(scope="module")
def eng():
    return importlib.import_module("long-tail-gan_b200.engine")


@pytest.fixture(scope="module")
def rec():
    return importlib.import_module("long-tail-gan_b200.recommend")


def _unpack(words, n):
    w = np.asarray(words, dtype=np.uint32)
    i = np.arange(len(w) * 32)
    bits = ((w[i // 32] >> (i % 32).astype(np.uint32)) & 1).astype(bool)
    return bits[:n], bits[n:]


@pytest.mark.parametrize("n_items", [1000, 1003, 64, 5])
def test_allow_bits_from_ids_and_mask(eng, n_items):
    rng = np.random.RandomState(n_items)
    mask = rng.rand(n_items) < 0.3
    mask[n_items - 1] = True          # the last item sits in the last, partial word
    ids = np.nonzero(mask)[0]
    for allow in (ids, list(ids), set(ids.tolist()), mask):
        w = eng.allow_bits(allow, n_items)
        assert w.dtype == np.uint32 and len(w) == (n_items + 31) // 32
        got, tail = _unpack(w, n_items)
        assert np.array_equal(got, mask) and not tail.any()
    assert not _unpack(eng.allow_bits([], n_items), n_items)[0].any()


def test_allow_bits_rejects_bad_input(eng):
    with pytest.raises(ValueError):
        eng.allow_bits([0, 1000], 1000)
    with pytest.raises(ValueError):
        eng.allow_bits([-1], 1000)
    with pytest.raises(ValueError):
        eng.allow_bits(np.ones(999, dtype=bool), 1000)


def test_shard_bitmaps_follow_the_global_set(eng):
    vp = importlib.import_module("long-tail-gan_b200.vocab_parallel")
    n_items = 1003
    rng = np.random.RandomState(3)
    ids = np.sort(rng.choice(n_items, 300, replace=False))
    mask = np.zeros(n_items, dtype=bool); mask[ids] = True
    bounds = vp.shard_bounds(n_items, 3)
    assert any(lo % 32 for lo, _ in bounds)          # a shard starts inside a word of the global bitmap
    for lo, hi in bounds:
        w = eng.allow_bits(ids, n_items, lo, hi)
        got, tail = _unpack(w, hi - lo)
        assert len(w) == (hi - lo + 31) // 32
        assert np.array_equal(got, mask[lo:hi]) and not tail.any()


def test_tsv_writer_adds_uid_offset_and_skips_padding(rec):
    items = np.array([[7, 3, -1], [-1, -1, -1], [0, 9, 4]])
    probs = np.array([[0.5, 0.25, 0.0], [0.0, 0.0, 0.0], [0.125, 1e-7, 3.0e-3]], dtype=np.float32)
    f = io.StringIO()
    rec.write_tsv(f, items, probs, 100)
    lines = f.getvalue().splitlines()
    assert lines[0] == "uid\trank\tsid\tprob"
    rows = [l.split("\t") for l in lines[1:]]
    assert [(int(a), int(b), int(c)) for a, b, c, _ in rows] == [(100, 1, 7), (100, 2, 3), (102, 1, 0), (102, 2, 9), (102, 3, 4)]
    assert np.array_equal(np.float32([float(r[3]) for r in rows]), probs[[0, 0, 2, 2, 2], [0, 1, 0, 1, 2]])   # float32 round trip
    f = io.StringIO()
    rec.write_tsv(f, -np.ones((2, 4), dtype=np.int64), np.zeros((2, 4), dtype=np.float32), 0)
    assert f.getvalue() == "uid\trank\tsid\tprob\n"


@pytest.mark.parametrize("split,prefix,start", [("test", "tst_tr", "tst_start"), ("validation", "vad_tr", "vad_start"),
                                                 ("train", "train", "uid_start")])
def test_split_loading_from_fixture(rec, split, prefix, start):
    g = np.load(GOLD)
    n_items = rec.n_items_of(GOLD)
    assert n_items == int(g["n_items"])
    ip, idx, uid0 = rec.load_split(GOLD, split, n_items)
    assert uid0 == int(g[start])
    want_ip = g[prefix + "_indptr"].astype(np.int64)[uid0 if split == "train" else 0:]
    assert np.array_equal(ip, want_ip - want_ip[0])
    assert np.array_equal(idx, g[prefix + "_indices"][want_ip[0]:want_ip[-1]].astype(np.int32))
    assert ip[-1] == len(idx) and idx.min() >= 0 and idx.max() < n_items
    assert np.array_equal(rec.load_niche(GOLD, n_items), np.sort(g["niche_tags"]))


def _write(path, text):
    with open(path, "w") as f:
        f.write(text)


def _csv(path, rows):
    _write(path, "uid,sid\n" + "".join("%d,%d\n" % r for r in rows))


@pytest.mark.parametrize("split", ["test", "validation", "train"])
def test_split_and_niche_loading_from_dataset_dir(rec, tmp_path, split):
    """A dataset directory in the reference's layout: splits with their own uid ranges, item names mapped to ids by item2id.txt."""
    n_items = 40
    d = str(tmp_path)
    _write(os.path.join(d, "unique_item_id.txt"), "".join("%d\n" % i for i in range(n_items)))
    _write(os.path.join(d, "item2id.txt"), "".join("tag%d\t%d\n" % (i, i) for i in range(n_items)))
    _write(os.path.join(d, "item_list.txt"), "".join("tag%d\n" % i for i in range(n_items) if i != 33))
    _write(os.path.join(d, "niche_items.txt"), "".join("tag%d\n" % i for i in (2, 5, 33, 39, 17)))
    rng = np.random.RandomState(1)
    ranges = dict(train=(5, 13), validation=(20, 26), test=(30, 35))
    fold = {}
    for name, (u0, u1) in ranges.items():
        fold[name] = {u: np.sort(rng.choice(n_items, rng.randint(1, 8), replace=False)) for u in range(u0, u1)}
        pairs = [(u, int(i)) for u in range(u0, u1) for i in rng.permutation(fold[name][u])]   # file order is not sorted
        if name == "train":
            _csv(os.path.join(d, "train_GAN.csv"), pairs)
        else:
            _csv(os.path.join(d, name + "_tr.csv"), pairs)
            _csv(os.path.join(d, name + "_te.csv"), [(u, (u * 7) % n_items) for u in range(u0, u1)])
    assert rec.n_items_of(d) == n_items
    ip, idx, uid0 = rec.load_split(d, split, n_items)
    u0, u1 = ranges[split]
    assert uid0 == u0 and len(ip) - 1 == u1 - u0
    for r in range(u1 - u0):
        assert np.array_equal(idx[ip[r]: ip[r + 1]], fold[split][u0 + r])
    assert rec.load_niche(d, n_items).tolist() == [2, 5, 17, 39]       # tag33 is not in item_list.txt


def test_cli_rejects_k_out_of_range(rec):
    with pytest.raises(SystemExit):
        rec.main([GOLD, "nochk", "--k", "129"])
    with pytest.raises(SystemExit):
        rec.main([GOLD, "nochk", "--split", "dev"])
