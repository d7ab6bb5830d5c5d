"""CatalogShardedEngine.recommend against that engine's evaluate and against GanEngine.recommend on the same weights
(the set-up of long-tail-gan_b200/vp_check.py, without training steps).
    python tools/vp_recommend_check.py [out.json]                       (one shard, one GPU)
    torchrun --nproc-per-node N tools/vp_recommend_check.py [out.json]  (N item shards)"""
import importlib
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "long-tail-gan_b200"


def run_check(n_items, batch, rank, world, seed=11, n_eval=96):
    gen = importlib.import_module(PKG + ".generator"); dis = importlib.import_module(PKG + ".discriminator")
    eng = importlib.import_module(PKG + ".engine"); vp = importlib.import_module(PKG + ".vocab_parallel")
    dpc = importlib.import_module(PKG + ".dp_check")
    I, B = int(n_items), int(batch)
    tabs = dpc.small_problem(1, batch_per_rank=B, n_items=I, seed=7)
    g = torch.Generator().manual_seed(123)
    lim = float(np.sqrt(6.0 / (I + 600)))
    params = [(torch.rand(I, 600, generator=g) * 2 - 1) * lim, (torch.rand(600, 400, generator=g) * 2 - 1) * 0.077, (torch.rand(200, 600, generator=g) * 2 - 1) * 0.087,
              (torch.rand(600, I, generator=g) * 2 - 1) * lim * 3.0, torch.randn(600, generator=g) * 0.001, torch.randn(400, generator=g) * 0.001,
              torch.randn(600, generator=g) * 0.001, torch.randn(I, generator=g) * 0.001]
    data, vae, lo, hi = vp.build_shard(tabs, I, rank, world, B, vae_params=params)
    disc = dis.Discriminator(I, I, 100, 150, 250, 300, seed=4242)
    e = vp.CatalogShardedEngine(vae, disc, data.max_B, data.max_P, I, lo, rank, world, seed=seed, max_active=data.max_active)
    # fold-in rows: the training rows of the first n_eval users without every fifth interaction (held out)
    ip = np.asarray(tabs["indptr"], dtype=np.int64); idx = np.asarray(tabs["indices"], dtype=np.int64)
    n_eval = min(n_eval, len(ip) - 1)
    held = np.zeros(len(idx), dtype=bool); held[4::5] = True
    row = np.repeat(np.arange(len(ip) - 1), np.diff(ip))
    m = row < n_eval
    trp = np.concatenate([[0], np.cumsum(np.bincount(row[m & ~held], minlength=n_eval))]); tep = np.concatenate([[0], np.cumsum(np.bincount(row[m & held], minlength=n_eval))])
    tri, tei = idx[m & ~held], idx[m & held]
    words0 = e.words.clone()
    rec = e.recommend(trp, tri, k=100, keep=1.0)
    torch.cuda.synchronize()
    words_unchanged = bool(torch.equal(e.words, words0))
    met = e.evaluate(trp, tri, tep, tei, k=100, recall_ks=(20, 50), keep=1.0)
    niche = np.sort(np.random.RandomState(99).choice(I, int(0.3 * I), replace=False))
    nic = e.recommend(trp, tri, k=100, keep=1.0, allow=niche)
    niche_ok = bool(np.isin(nic["items"], niche).all() and np.array_equal(nic["lse"].view(np.uint32), rec["lse"].view(np.uint32)))
    for r in range(n_eval):
        inset = np.isin(rec["items"][r], niche)
        pre = rec["items"][r][inset]
        niche_ok &= bool(np.array_equal(nic["items"][r][:len(pre)], pre)
                         and np.array_equal(nic["probs"][r][:len(pre)].view(np.uint32), rec["probs"][r][inset].view(np.uint32)))
    out = dict(world=world, n_items=I, n_users=n_eval, words_unchanged=words_unchanged,
               items_equal_evaluate_topk=bool(np.array_equal(rec["items"], met["topk"])), niche_only_ok=niche_ok)
    if rank == 0:
        vae1 = gen.MultiVAE([200, 600, I], lam=0.0, random_seed=1); vae1.set_params(params); vae1.reset_optimizer()
        disc1 = dis.Discriminator(I, I, 100, 150, 250, 300, seed=4242)
        data1 = eng.TrainData(batch_size=B, **tabs)
        e1 = eng.GanEngine(vae1, disc1, data1.max_B, data1.max_P, seed=seed, use_graphs=False, max_active=data1.max_active)
        rec1 = e1.recommend(trp, tri, k=100, keep=1.0)
        # probabilities position by position (summation order differs between the engines, so near-equal items may swap places)
        diff = np.abs(rec["probs"] - rec1["probs"]).max(1) / rec1["probs"][:, 0]
        out.update(max_prob_diff_rel=float(diff.max()), items_equal_single_gpu_fraction=float((rec["items"] == rec1["items"]).mean()),
                   max_lse_diff=float(np.abs(rec["lse"] - rec1["lse"]).max()))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    return out


def main():
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    res = run_check(2400, 96, rank, world)
    if rank == 0:
        print(json.dumps(res, indent=1))
        for a in sys.argv[1:]:
            if a.endswith(".json"):
                json.dump(res, open(a, "w"), indent=1)
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        sys.stdout.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
