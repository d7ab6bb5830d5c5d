"""Throughput of top-k recommendation on one GPU, written as JSON (default profiles/r3_recommend_bench.json):
    python tools/recommend_bench.py [out.json]

- end to end at the ML-20M shape (I = 20,108; 10,000 synthetic held-out users, synthetic.make_eval_split; k = 100):
  GanEngine.recommend against GanEngine.evaluate in users/s, both at the engine's keep_vae (same forward), alternated in one process
  after a warm-up of each; host upload and read-back inside the time.
- kernel only: ltg_topk_recommend against ltg_topk_metrics on the same fp32 score matrices and seen lists, [3,334 x 20,108]
  (staged path; one evaluation batch of the ML-20M shape) and [1,000 x 125,000] (streaming path; one of 8 shards of the 1 M-item
  catalog), each without and with an allow mask of a 50 % niche set; CUDA events around 20 launches, median of 5 alternated rounds.
  Both matrices are larger than L2, so every launch reads its rows from HBM.
The GPU's name and power limit are read in the same run."""
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
PKG = "long-tail-gan_b200"


def gpu_info():
    info = dict(name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                           text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip()
    except Exception as e:   # noqa: BLE001
        info["power_limit_and_max_sm_clock"] = "unavailable (%s)" % e
    return info


def end_to_end(rounds=5):
    syn = importlib.import_module(PKG + ".synthetic")
    gen = importlib.import_module(PKG + ".generator"); dis = importlib.import_module(PKG + ".discriminator")
    eng = importlib.import_module(PKG + ".engine")
    _, I, deg = syn.CONFIGS["ml20m"]
    n = 10000
    tr_p, tr_i, te_p, te_i = syn.make_eval_split(n, I, deg)
    vae = gen.MultiVAE([200, 600, I], lam=0.0, random_seed=98765); vae.init_weights(98765)
    disc = dis.Discriminator(I, I, 100, 150, 250, 300, seed=4242)
    e = eng.GanEngine(vae, disc, 500, 1, seed=2026, use_graphs=False, max_active=1)

    def t_rec():
        t0 = time.perf_counter(); e.recommend(tr_p, tr_i, k=100, keep=None); return time.perf_counter() - t0

    def t_eval():
        t0 = time.perf_counter(); e.evaluate(tr_p, tr_i, te_p, te_i, k=100); torch.cuda.synchronize(); return time.perf_counter() - t0
    t_rec(); t_eval()
    rec, ev = [], []
    for _ in range(rounds):
        rec.append(t_rec()); ev.append(t_eval())
    med = lambda x: sorted(x)[len(x) // 2]  # noqa: E731
    return dict(n_items=I, users=n, k=100, batch=int(e._eval_ws.rows), recommend_users_per_sec=n / med(rec), evaluate_users_per_sec=n / med(ev),
                recommend_ms=[x * 1e3 for x in rec], evaluate_ms=[x * 1e3 for x in ev], ratio_time_recommend_over_evaluate=med(rec) / med(ev))


def kernel_only(rows, n_items, deg, rounds=5, launches=20):
    """deg: mean seen items per row (the fold-in part of the configuration's mean interactions per user)."""
    ops = importlib.import_module(PKG + ".ops"); eng = importlib.import_module(PKG + ".engine")
    rng = np.random.RandomState(n_items)
    g = torch.Generator(device="cuda").manual_seed(n_items)
    scores = torch.randn(rows, n_items, generator=g, device="cuda") * 2.0
    nnz = rng.poisson(deg, rows).clip(1, n_items // 2)
    seen_ptr = np.concatenate([[0], np.cumsum(nnz)]).astype(np.int32)
    seen_items = np.concatenate([np.sort(rng.choice(n_items, c, replace=False)) for c in nnz]).astype(np.int32)
    held_ptr = np.arange(rows + 1, dtype=np.int32) * 4
    held_items = np.sort(rng.randint(0, n_items, (rows, 4)), axis=1).reshape(-1).astype(np.int32)
    dev = lambda a: torch.as_tensor(a).cuda()  # noqa: E731
    sp, si, hp, hi = dev(seen_ptr), dev(seen_items), dev(held_ptr), dev(held_items)
    niche = np.sort(rng.choice(n_items, n_items // 2, replace=False))
    bits = dev(eng.allow_bits(niche, n_items).view(np.int32))
    dcg = torch.zeros(rows, dtype=torch.float64, device="cuda"); hits = torch.zeros(rows, 2, dtype=torch.int32, device="cuda")
    idx = torch.zeros(rows, 100, dtype=torch.int32, device="cuda"); lg = torch.zeros(rows, 100, device="cuda")
    pr = torch.zeros(rows, 100, device="cuda"); lse = torch.zeros(rows, device="cuda")
    runs = {
        "topk_metrics": lambda: ops.topk_metrics(scores, rows, n_items, sp, si, hp, hi, 100, (20, 50), None, dcg, hits),
        "topk_recommend": lambda: ops.topk_recommend(scores, rows, n_items, sp, si, None, 100, idx, lg, pr, lse),
        "topk_recommend_niche50": lambda: ops.topk_recommend(scores, rows, n_items, sp, si, bits, 100, idx, lg, pr, lse),
    }
    for fn in runs.values():
        fn(); fn()
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    for _ in range(rounds):
        for name, fn in runs.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(launches):
                fn()
            b.record(); b.synchronize()
            times[name].append(a.elapsed_time(b) * 1e3 / launches)
    med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
    nbytes = rows * n_items * 4
    out = dict(rows=rows, n_items=n_items, mean_seen=float(nnz.mean()), k=100, path="staged" if n_items <= 49152 else "streaming",
               us=med, us_all_rounds=times, score_gbs={k: nbytes / (v * 1e-6) / 1e9 for k, v in med.items()},
               ratio_recommend_over_metrics=med["topk_recommend"] / med["topk_metrics"],
               ratio_recommend_niche50_over_metrics=med["topk_recommend_niche50"] / med["topk_metrics"])
    del scores
    torch.cuda.empty_cache()
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_recommend_bench.json")
    importlib.import_module(PKG)._lib.build()
    importlib.import_module(PKG + ".ops").init()
    res = dict(gpu=gpu_info(), end_to_end_ml20m=end_to_end(),
               kernel_staged=kernel_only(3334, 20108, 0.8 * 73.0), kernel_streaming=kernel_only(1000, 125000, 0.8 * 50.0))
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    json.dump(res, open(out_path, "w"), indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
