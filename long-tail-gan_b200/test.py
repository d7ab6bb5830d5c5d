"""Drop-in for Codes/test.py:  python test.py <dataset_dir> <checkpoint_path> [--long-tail]   (run from the directory holding config.ini).
Rebuilds the networks, restores the checkpoint written by train.py and prints `NDCG@100<TAB>R@20<TAB>R@50` over the test
users (test.py:138-173); scoring, seen-item masking and ranking run on the device.
--long-tail (ours) adds a second line from the same ranked lists: niche NDCG@100, niche R@20, niche R@50, niche share@100,
avg pop@100, coverage@100, niche coverage@100 and Gini@100 (engine.longtail_from_counts; niche items: niche_items.txt,
popularity: training interactions per item in train_GAN.csv)."""
from __future__ import print_function

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
from .engine import GanEngine, longtail_summary   # noqa: E402
from .generator import MultiVAE              # noqa: E402
from .recommend import load_niche            # noqa: E402
from .train import read_config               # noqa: E402


def test_GAN(h0_size, h1_size, h2_size, h3_size, NUM_EPOCH, NUM_SUB_EPOCHS, BATCH_SIZE, DISPLAY_ITER, LEARNING_RATE, to_restore,
             model_name, dataset, GANLAMBDA, output_path, quiet=False, long_tail=False):
    """Returns (NDCG@100, R@20, R@50); with long_tail=True also a dict of the long-tail numbers (engine.longtail_summary)."""
    if dataset.endswith(".npz"):
        g = np.load(dataset)
        n_items = int(g["n_items"])
        tr = (g["tst_tr_indptr"], g["tst_tr_indices"].astype(np.int32)); te = (g["tst_te_indptr"], g["tst_te_indices"].astype(np.int32))
        train_indices = g["train_indices"] if long_tail else None
    else:
        pro_dir = dataset + "/"
        n_items = sum(1 for _ in open(os.path.join(pro_dir, "unique_item_id.txt")))
        t_tr, t_te, _ = dp.load_tr_te_data(os.path.join(pro_dir, "test_tr.csv"), os.path.join(pro_dir, "test_te.csv"), n_items)
        t_tr.sort_indices(); t_te.sort_indices()
        tr = (t_tr.indptr, t_tr.indices); te = (t_te.indptr, t_te.indices)
        train_indices = dp.load_train_data(os.path.join(pro_dir, "train_GAN.csv"), n_items)[0].indices if long_tail else None
    ck = torch.load(output_path, map_location="cpu")
    vae = MultiVAE(ck["p_dims"], lam=0.0, random_seed=98765)
    vae.load_state_dict(ck["vae"])
    hs = ck["hs"]
    disc = Discriminator(n_items, n_items, hs[0], hs[1], hs[2], hs[3], seed=0)
    disc.load_state_dict(ck["disc"])
    if not quiet:
        print("Model Loaded")
    batch_size_test = 2048   # test.py:76 uses 20000-row dense batches; the device path streams 2048 rows at a time
    engine = GanEngine(vae, disc, batch_size_test, 1, seed=int(ck["words"][0]) + 1, lr=LEARNING_RATE, lam=GANLAMBDA, use_graphs=False,
                       max_active=1)
    if not long_tail:
        m = engine.evaluate(tr[0], tr[1], te[0], te[1], k=100, recall_ks=(20, 50), batch=batch_size_test)
    else:
        pop = np.bincount(np.asarray(train_indices, dtype=np.int64), minlength=n_items)
        m = engine.evaluate(tr[0], tr[1], te[0], te[1], k=100, recall_ks=(20, 50), batch=batch_size_test, niche=load_niche(dataset, n_items),
                            item_pop=pop)
    n100, r20, r50 = np.mean(m["ndcg@100"]), np.mean(m["recall@20"]), np.mean(m["recall@50"])
    print(str(n100) + "\t" + str(r20) + "\t" + str(r50))   # test.py:173
    if not long_tail:
        return n100, r20, r50
    lt = longtail_summary(m)
    print("\t".join(str(v) for v in lt.values()))
    return n100, r20, r50, lt


if __name__ == "__main__":
    cfg = read_config("config.ini")
    args = [a for a in sys.argv[1:] if a != "--long-tail"]
    cfg["dataset"] = args[0]
    cfg["output_path"] = args[1]
    test_GAN(long_tail="--long-tail" in sys.argv[1:], **cfg)
