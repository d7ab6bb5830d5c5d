"""Cost of long-tail evaluation on one GPU, written as JSON (default profiles/r3_longtail_bench.json):
    python tools/longtail_bench.py [out.json]

- kernel only: ltg_topk_longtail against ltg_topk_metrics on the same fp32 score matrices, seen lists and held-out lists, k = 100,
  recall cut-offs (20, 50), a niche set of a third of the catalog and popularity counts: [3,334 x 20,108] (staged path; one evaluation
  batch of the ML-20M shape) and [1,000 x 125,000] (streaming path; one of 8 shards of the 1 M-item catalog). CUDA events around 20
  launches, the two entry points alternated for 7 rounds; the median and the spread (max - min over rounds) of each are reported, so
  the difference can be read against the run-to-run spread of the same call. Both matrices are larger than L2, so every launch reads
  its rows from HBM.
- end to end at the ML-20M shape (I = 20,108; 10,000 synthetic held-out users, synthetic.make_eval_split; k = 100):
  GanEngine.evaluate with and without niche / item_pop, alternated in one process after a warm-up of each; host upload and read-back
  inside the time.
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


def _stats(times):
    s = sorted(times)
    return dict(median=s[len(s) // 2], min=s[0], max=s[-1], spread=s[-1] - s[0], all=times)


def kernel_only(rows, n_items, deg, rounds=7, launches=20):
    """deg: mean seen items per row (the fold-in part of the configuration's mean interactions per user)."""
    ops = importlib.import_module(PKG + ".ops"); eng = importlib.import_module(PKG + ".engine")
    rng = np.random.RandomState(n_items)
    g = torch.Generator(device="cuda").manual_seed(n_items)
    scores = torch.randn(rows, n_items, generator=g, device="cuda") * 2.0
    nnz = rng.poisson(deg, rows).clip(1, n_items // 2)
    seen_ptr = np.concatenate([[0], np.cumsum(nnz)]).astype(np.int32)
    seen_items = np.concatenate([np.sort(rng.choice(n_items, c, replace=False)) for c in nnz]).astype(np.int32)
    n_held = rng.poisson(deg / 4, rows).clip(0, n_items // 4)
    held_ptr = np.concatenate([[0], np.cumsum(n_held)]).astype(np.int32)
    held_items = np.concatenate([np.sort(rng.choice(n_items, c, replace=False)) for c in n_held] + [np.zeros(0, np.int64)]).astype(np.int32)
    dev = lambda a: torch.as_tensor(a).cuda()  # noqa: E731
    sp, si, hp, hi = dev(seen_ptr), dev(seen_items), dev(held_ptr), dev(held_items if len(held_items) else np.zeros(1, np.int32))
    bits = dev(eng.allow_bits(np.sort(rng.choice(n_items, n_items // 3, replace=False)), n_items).view(np.int32))
    pop = dev(rng.zipf(1.5, n_items).clip(0, 2 ** 20).astype(np.int32))
    i32 = lambda *s: torch.zeros(*s, dtype=torch.int32, device="cuda")  # noqa: E731
    dcg, hits = torch.zeros(rows, dtype=torch.float64, device="cuda"), i32(rows, 2)
    dcg_n, hits_n, n_top = torch.zeros(rows, dtype=torch.float64, device="cuda"), i32(rows, 2), i32(rows)
    pop_sum, rec_count = torch.zeros(rows, dtype=torch.int64, device="cuda"), i32(n_items)
    runs = {
        "topk_metrics": lambda: ops.topk_metrics(scores, rows, n_items, sp, si, hp, hi, 100, (20, 50), None, dcg, hits),
        "topk_longtail": lambda: ops.topk_longtail(scores, rows, n_items, sp, si, hp, hi, 100, (20, 50), None, dcg, hits, bits, pop, dcg_n,
                                                   hits_n, n_top, pop_sum, rec_count),
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
    st = {k: _stats(v) for k, v in times.items()}
    out = dict(rows=rows, n_items=n_items, mean_seen=float(nnz.mean()), mean_held=float(n_held.mean()), k=100,
               path="staged" if n_items <= 49152 else "streaming", us=st,
               overhead_longtail_over_metrics=st["topk_longtail"]["median"] / st["topk_metrics"]["median"] - 1.0)
    del scores
    torch.cuda.empty_cache()
    return out


def end_to_end(rounds=7):
    syn = importlib.import_module(PKG + ".synthetic")
    gen = importlib.import_module(PKG + ".generator"); dis = importlib.import_module(PKG + ".discriminator")
    eng = importlib.import_module(PKG + ".engine")
    _, I, deg = syn.CONFIGS["ml20m"]
    n = 10000
    tr_p, tr_i, te_p, te_i = syn.make_eval_split(n, I, deg)
    rng = np.random.RandomState(5)
    niche = np.sort(rng.choice(I, I // 3, replace=False))
    pop = np.bincount(syn.make_interactions(20000, I, deg, 99)[1].astype(np.int64), minlength=I)
    vae = gen.MultiVAE([200, 600, I], lam=0.0, random_seed=98765); vae.init_weights(98765)
    disc = dis.Discriminator(I, I, 100, 150, 250, 300, seed=4242)
    e = eng.GanEngine(vae, disc, 500, 1, seed=2026, use_graphs=False, max_active=1)

    def timed(**kw):
        t0 = time.perf_counter(); e.evaluate(tr_p, tr_i, te_p, te_i, k=100, **kw); torch.cuda.synchronize(); return time.perf_counter() - t0
    timed(); timed(niche=niche, item_pop=pop)
    plain, lt = [], []
    for _ in range(rounds):
        plain.append(timed()); lt.append(timed(niche=niche, item_pop=pop))
    sp, sl = _stats([x * 1e3 for x in plain]), _stats([x * 1e3 for x in lt])
    return dict(n_items=I, users=n, k=100, batch=int(e._eval_ws.rows), evaluate_ms=sp, evaluate_longtail_ms=sl,
                slowdown_longtail_over_plain=sl["median"] / sp["median"] - 1.0)


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "r3_longtail_bench.json")
    importlib.import_module(PKG)._lib.build()
    importlib.import_module(PKG + ".ops").init()
    res = dict(gpu=gpu_info(), kernel_staged=kernel_only(3334, 20108, 0.8 * 73.0), kernel_streaming=kernel_only(1000, 125000, 0.8 * 50.0),
               end_to_end_ml20m=end_to_end())
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    json.dump(res, open(out_path, "w"), indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
