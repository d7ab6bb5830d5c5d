"""Top-k recommendations from a trained checkpoint:

    python recommend.py <dataset_dir | fixture.npz> <checkpoint> [--split test|validation|train] [--k 100] [--keep 1.0]
                        [--niche-only] [--include-seen] [--out FILE]

Restores the checkpoint written by train.py the way test.py does, folds in the chosen split's interactions (`<split>_tr.csv`, or
train_GAN.csv for `train`) and writes, per user, the k items with the highest generator probability as TSV: a header
`uid  rank  sid  prob`, then one line per listed item (rank 1 first). `uid` is the dataset's user id, `sid` the item id of the
dataset's CSV files, `prob` the generator's softmax probability over the whole catalog (MultiVAE.py:143). By default the user's fold-in
items are never listed (--include-seen lists them too); --niche-only lists niche items only (niche_items.txt, the set the training
samples generated items from). Scoring, filtering and ranking run on the device (GanEngine.recommend)."""
from __future__ import print_function

import argparse
import importlib
import os
import sys

import numpy as np
import torch

if __package__ in (None, ""):
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    _pkg = importlib.import_module("long-tail-gan_b200")
    __package__ = _pkg.__name__

from . import data_processing as dp          # noqa: E402
from .discriminator import Discriminator     # noqa: E402
from .engine import GanEngine                # noqa: E402
from .generator import MultiVAE              # noqa: E402

SPLITS = ("test", "validation", "train")
_NPZ_PREFIX = {"test": ("tst_tr", "tst_start"), "validation": ("vad_tr", "vad_start"), "train": ("train", "uid_start")}


def n_items_of(dataset):
    if dataset.endswith(".npz"):
        return int(np.load(dataset)["n_items"])
    return sum(1 for _ in open(os.path.join(dataset, "unique_item_id.txt")))


def load_split(dataset, split, n_items):
    """Fold-in rows of a split: (indptr, indices) CSR with ascending item ids within a row, and the uid of row 0. For a dataset
    directory the rows are those of <split>_tr.csv (uid offset as load_tr_te_data removes it) or, for `train`, of train_GAN.csv from
    its smallest uid on; for the .npz fixture the same arrays as saved by the reference's loaders."""
    if split not in SPLITS:
        raise ValueError("split must be one of %s, got %r" % (", ".join(SPLITS), split))
    if dataset.endswith(".npz"):
        g = np.load(dataset)
        prefix, start = _NPZ_PREFIX[split]
        uid0 = int(g[start])
        ip = g[prefix + "_indptr"].astype(np.int64)
        if split == "train":   # rows are uids from 0 on
            ip = ip[uid0:]
        return ip - ip[0], g[prefix + "_indices"][ip[0]: ip[-1]].astype(np.int32), uid0
    if split == "train":
        csr, uid0 = dp.load_train_data(os.path.join(dataset, "train_GAN.csv"), n_items)
        csr = csr[uid0:]
    else:
        csr, _, uid0 = dp.load_tr_te_data(os.path.join(dataset, split + "_tr.csv"), os.path.join(dataset, split + "_te.csv"), n_items)
    csr = csr.tocsr()
    csr.sort_indices()
    return csr.indptr.astype(np.int64), csr.indices.astype(np.int32), int(uid0)


def load_niche(dataset, n_items):
    """The niche item ids, ascending: niche_items.txt through load_pop_niche_tags, or the fixture's niche_tags."""
    if dataset.endswith(".npz"):
        return np.sort(np.load(dataset)["niche_tags"].astype(np.int64))
    _, _, niche, _, _ = dp.load_pop_niche_tags(os.path.join(dataset, "item2id.txt"), os.path.join(dataset, "item_list.txt"),
                                               os.path.join(dataset, "niche_items.txt"), n_items)
    return np.asarray(sorted(niche), dtype=np.int64)


def write_tsv(f, items, probs, uid0):
    """items / probs [N, k] (item -1 = padding, not written) -> `uid  rank  sid  prob` lines; row r is user uid0 + r, rank 1 first."""
    items = np.asarray(items); probs = np.asarray(probs)
    f.write("uid\trank\tsid\tprob\n")
    r, j = np.nonzero(items >= 0)
    if len(r):
        cols = np.stack([r + int(uid0), j + 1, items[r, j]], 1).astype(np.int64)
        lines = ["%d\t%d\t%d\t%.9g\n" % (a, b, c, p) for (a, b, c), p in zip(cols.tolist(), probs[r, j].tolist())]
        f.write("".join(lines))


def recommend_GAN(dataset, checkpoint, split="test", k=100, keep=1.0, niche_only=False, include_seen=False, out=None):
    """Returns (items [N, k], probs [N, k], uid of row 0) and writes the TSV to `out` (a path; None: stdout)."""
    n_items = n_items_of(dataset)
    ip, idx, uid0 = load_split(dataset, split, n_items)
    allow = load_niche(dataset, n_items) if niche_only else None
    ck = torch.load(checkpoint, map_location="cpu")
    vae = MultiVAE(ck["p_dims"], lam=0.0, random_seed=98765)
    vae.load_state_dict(ck["vae"])
    hs = ck["hs"]
    disc = Discriminator(n_items, n_items, hs[0], hs[1], hs[2], hs[3], seed=0)
    disc.load_state_dict(ck["disc"])
    engine = GanEngine(vae, disc, 2048, 1, seed=int(ck["words"][0]) + 1, use_graphs=False, max_active=1)
    rec = engine.recommend(ip, idx, k=k, keep=keep, exclude_seen=not include_seen, allow=allow)
    if out is None:
        write_tsv(sys.stdout, rec["items"], rec["probs"], uid0)
        sys.stdout.flush()
    else:
        with open(out, "w") as f:
            write_tsv(f, rec["items"], rec["probs"], uid0)
    return rec["items"], rec["probs"], uid0


def main(argv=None):
    ap = argparse.ArgumentParser(description="Top-k item recommendations from a Long-Tail-GAN checkpoint (TSV: uid, rank, sid, prob).")
    ap.add_argument("dataset", help="dataset directory (as for train.py / test.py) or a .npz fixture")
    ap.add_argument("checkpoint", help="model_<epoch> file written by train.py")
    ap.add_argument("--split", default="test", choices=SPLITS, help="users to recommend for (fold-in rows of this split)")
    ap.add_argument("--k", type=int, default=100, help="items per user, 1..128")
    ap.add_argument("--keep", type=float, default=1.0, help="encoder dropout keep probability (1.0: deterministic lists)")
    ap.add_argument("--niche-only", action="store_true", help="list niche items only")
    ap.add_argument("--include-seen", action="store_true", help="also list the user's fold-in items")
    ap.add_argument("--out", default=None, help="output file (default: stdout)")
    a = ap.parse_args(argv)
    if not 1 <= a.k <= 128:
        ap.error("--k must lie in 1..128")
    recommend_GAN(a.dataset, a.checkpoint, split=a.split, k=a.k, keep=a.keep, niche_only=a.niche_only, include_seen=a.include_seen, out=a.out)


if __name__ == "__main__":
    main()
