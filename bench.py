#!/usr/bin/env python
"""Headline benchmark: GAN-step users/sec of the Long-Tail-GAN hot path at the ML-20M-shaped configuration
(136,677 users x 20,108 items, VAE 600-200, batch 500 per GPU), BASELINE.json `configs[1]`.

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched under torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                     (the reference's CPU data flow on the host cores)

One "step" = one GAN step over one batch of B users per GPU: phase A (generator inference + niche sampling + pair
construction, train.py:192-269) + one discriminator update (train.py:300) + one generator update (train.py:326).
`value` is users/sec with the inputs resident in HBM; `e2e` is the same step with the batch's inputs copied from pinned
host memory and the losses read back inside the timed region. Prints ONE JSON line on rank 0.
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

CONFIG = "ml20m"
BATCH = 500
# BASELINE.json `configs`: the headline (what the driver runs with no --config) is configs[1]; the others are run with --config and
# their lines are kept under profiles/. batch = users per GPU per step (weak scaling).
BENCH_CONFIGS = {
    "ml20m": dict(batch=500, label="ML-20M-shaped synthetic"),
    # batch is free for the throughput configs (SURVEY 8d): 8192 users per GPU puts the G step on the tensor side of its roofline
    "netflix": dict(batch=8192, label="Netflix-shaped synthetic"),
    # "GAN sampling + discriminator at full batch, 8 B200": one eighth of the 571,355 users per GPU and step
    "msd": dict(batch=71420, label="MSD-shaped synthetic (full batch / 8 per GPU)"),
    # the bundled dataset (tests/golden/askubuntu_sample.npz = the reference loaders' outputs on Dataset/Askubuntu_Sample), config.ini batch
    "askubuntu": dict(batch=100, label="bundled Askubuntu sample (real data)"),
    # configs[4]: 1 M items x 5 M users, catalog-sharded (vocab-parallel) decoder/softmax/top-k: every rank holds I / N items and all
    # ranks process the same 500 users per step (strong scaling over the catalog); N = 1 holds the whole catalog on one GPU
    "x1m": dict(batch=500, label="1M-item synthetic catalog, catalog-sharded"),
}
X1M_ITEMS, X1M_USERS, X1M_DEG = 1000000, 5000000, 50.0
GOLD = os.path.join(ROOT, "tests", "golden", "askubuntu_sample.npz")
N_BENCH_BATCHES = 8   # distinct user batches cycled through by the timed steps (per GPU)
CPU_BATCH_CAP = 1000  # users per step of the CPU baseline sample (dense fp32 [B, I] tensors)
DUMP_ROWS = 4096      # --dump-outputs: item rows sampled from each [I, 600] matrix (2 x 9.8 MB; all of them are 2 x 48 MB at ML-20M)
H0, H1, H2, H3 = 100, 150, 250, 300   # config.ini h0..h3_size
LR, LAM = 1e-4, 1.0                    # config.ini LEARNING_RATE, GANLAMBDA


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=48)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=os.environ.get("LTG_BENCH_CONFIG", "ml20m"), choices=sorted(BENCH_CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="users per GPU per step (default: the config's)")
    ap.add_argument("--no-dp-check", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=6, help="steps of the bounded CPU-baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (losses, updated parameters)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.config == "x1m"):
        ap.error("--dump-outputs writes the GAN step of --impl b200; --impl reference and --config x1m are not covered")
    return args


def measured_peaks(key="hbm_gbs"):
    """HBM GB/s or dense bf16 TFLOP/s (burst figure: the kernels are timed alone, back to back) from the driver-written file."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        if key in d:
            return float(d[key]), "measured (MEASURED_PEAKS.json %s)" % key
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1390.0}[key], "fallback (B200_PROFILING.md)"


class ClockSampler(object):
    """SM clock / throttle reasons sampled WHILE the timed regions run: an NVML polling thread (5 ms period -- the default timed
    region is only tens of milliseconds long, too short for `nvidia-smi -lms`), with nvidia-smi as the fallback."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None
        self.thread = None
        self.rows = []
        self._stop = False
        self.max_mhz = None

    def _poll(self, nv, h):
        reasons = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                   "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                   "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                   "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        while not self._stop:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                self.rows.append((float(mhz), pw, [k for k, b in reasons.items() if mask & b]))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = int(visible.split(",")[self.index]) if visible and all(x.strip().isdigit() for x in visible.split(",")) else self.index
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=2)
            if self.rows:
                sm = sorted(r[0] for r in self.rows)
                out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=self.max_mhz, samples=len(sm), power_w_max=max(r[1] for r in self.rows),
                           reasons=sorted({k for r in self.rows for k in r[2]}), source="NVML, 5 ms period over the timed regions")
            return out
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
        except Exception:
            pass
        try:
            rows = [r.strip().split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = sorted(float(r[0]) for r in rows)
            if sm:
                out["sm_mhz"] = sm[len(sm) // 2]
                out["sm_max_mhz"] = float(rows[0][1])
                out["samples"] = len(sm)
                out["power_w_max"] = max(float(r[2]) for r in rows)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for j, nm in enumerate(names):
                    if any(r[3 + j].strip().lower().startswith("active") for r in rows):
                        out["reasons"].append(nm)
                out["source"] = "nvidia-smi -lms 100"
            os.unlink(self.path)
        except Exception:
            pass
        return out


def step_roofline(n_items, batch, nnz_user, cand_user, pairs_real, pairs_gen, t_a, t_d, t_g, hbm_gbs, tc_tflops, world=1, t_step=None):
    """Whole-step roofline of SURVEY 8d: algorithmic FLOPs and HBM bytes of phase A, the D update and the G update (the formulas of
    that section, written out below), t_roof = max(FLOPs / tensor peak, bytes / HBM peak) per phase, fraction = t_roof / t_measured.
    Times in ms, returns per-phase dicts and the step total. Pure arithmetic (also exercised by the CPU tests).
    world > 1 (data parallel, per-GPU view): the optimizer is row-sharded, so the dense-Adam bytes of the two [I,600] matrices are
    divided by the number of ranks. t_step: the measured time of the whole step when its phases overlap (engine.run_step); the step
    fraction is then roof / t_step, and the per-phase fractions remain those of the phases timed one by one."""
    I, B = float(n_items), float(batch)
    c = 2.0 * (600 * 400 + 200 * 600)              # the two middle layers, flops per user
    d = 2.0 * 600 * I                               # decoder, flops per user
    p_u = 0.5 * (pairs_real + pairs_gen) / B        # pairs of each kind per user
    p_vae = 1201.0 * I + 361600.0
    fl = dict(A=B * (2.0 * nnz_user * 600 + c + d),
              D=B * p_u * 1923600.0,
              G=B * (3.0 * (c + d) + 4.0 * nnz_user * 600 + p_u * 320600.0))
    by = dict(A=2.0 * 600 * I + B * nnz_user * 1204.0 + 8.0 * B * cand_user,
              D=1600.0 * (pairs_real + pairs_gen) + 26.0 * 161001.0,
              G=26.0 * (1200.0 * I / world + I + 361600.0) + 4.0 * 600 * I + 8.0 * 600 * I + 4.0 * B * I + B * nnz_user * 1204.0 + B * 1800 * 4.0)
    meas = dict(A=t_a, D=t_d, G=t_g)
    out, roof_total = {}, 0.0
    for ph in ("A", "D", "G"):
        t_tc = fl[ph] / (tc_tflops * 1e12) * 1e3
        t_hbm = by[ph] / (hbm_gbs * 1e9) * 1e3
        t_roof = max(t_tc, t_hbm)
        roof_total += t_roof
        out[ph] = dict(flops=fl[ph], bytes=by[ph], t_tensor_ms=t_tc, t_hbm_ms=t_hbm, bound="tensor" if t_tc > t_hbm else "hbm",
                       t_roof_ms=t_roof, t_measured_ms=meas[ph], frac=t_roof / meas[ph] if meas[ph] > 0 else None)
    t_sum = t_a + t_d + t_g
    t_meas = t_sum if t_step is None else t_step
    out["step"] = dict(t_roof_ms=roof_total, t_measured_ms=t_meas, frac=roof_total / t_meas if t_meas > 0 else None,
                       t_sum_of_phases_ms=t_sum, frac_sum_of_phases=roof_total / t_sum if t_sum > 0 else None,
                       note="SURVEY 8d algorithmic model (dense-Adam bytes dominate G); t_measured = the whole step (ms_per_step: one "
                            "captured graph per batch, the G forward overlapping the D update); phases also timed one by one")
    return out


EVAL_USERS = {"ml20m": 10000, "netflix": 40000, "msd": 50000}   # SURVEY 8d: held-out users per configuration


def eval_throughput(engine, tabs, n_users=2000):
    """SURVEY 8d asks for evaluation users/s beside the training metric: fold-in forward (dropout on, F4) + exact top-100
    NDCG@100 / Recall@20,50 (engine.evaluate = train.py:333-348 / test.py:138-173). Synthetic configurations: SURVEY 8d's number
    of held-out users (10 k / 40 k / 50 k) with an 80/20 fold-in / held-out split (synthetic.make_eval_split); the bundled real
    dataset: its first n_users training users, every fifth item held out. Host CSR upload and metric read-back are inside the time."""
    import numpy as np
    import torch
    if CONFIG in EVAL_USERS:
        syn = importlib.import_module("long-tail-gan_b200.synthetic")
        _, I, deg = syn.CONFIGS[CONFIG]
        n = EVAL_USERS[CONFIG]
        args = syn.make_eval_split(n, I, deg)
        split = "80/20 random split of %d synthetic held-out users" % n
    else:
        indptr = np.asarray(tabs["indptr"], dtype=np.int64)
        indices = np.asarray(tabs["indices"], dtype=np.int32)
        n = int(min(n_users, len(indptr) - 1))
        tr, te, trp, tep = [], [], [0], [0]
        for u in range(n):
            it = indices[indptr[u]: indptr[u + 1]]
            held = np.zeros(len(it), dtype=bool)
            held[4::5] = True
            tr.append(it[~held]); te.append(it[held])
            trp.append(trp[-1] + len(tr[-1])); tep.append(tep[-1] + len(te[-1]))
        args = (np.asarray(trp, dtype=np.int64), np.concatenate(tr), np.asarray(tep, dtype=np.int64), np.concatenate(te))
        split = "every fifth item of the first %d training users held out" % n
    engine.evaluate(*args)   # warm-up (allocates the evaluation workspaces)
    torch.cuda.synchronize()
    dts = []
    for _ in range(3):
        t0 = time.perf_counter()
        res = engine.evaluate(*args)
        dts.append(time.perf_counter() - t0)
    dt = sorted(dts)[1]
    nd = res["ndcg@100"]
    return dict(users_per_sec=n / dt, users=n, ms=dt * 1e3, users_with_heldout=len(nd), ndcg_at_100_random_init=float(np.mean(nd)) if nd else None,
                split=split, batch=int(engine._eval_ws.rows), repeats_ms=[x * 1e3 for x in dts],
                what="fold-in forward + exact top-100 NDCG@100 / Recall@20,50 per user; host CSR upload and metric read-back included; "
                     "median of 3 calls")


def step_outputs(engine, batch, world):
    """What a caller of the timed GAN step holds after its last step: the losses and the updated generator and discriminator
    parameters in the reference's order, as host arrays. Of the two [I, 600] item matrices (W_q0 rows, W_p1 columns) the same
    DUMP_ROWS items, drawn with a fixed seed, are kept. Under data parallelism a collective: every rank calls it."""
    import numpy as np
    import torch
    engine.gather_master()
    out = {"loss_" + k: np.float64(v) for k, v in engine.last_losses(batch, reduce=world > 1).items()}
    items = np.sort(np.random.RandomState(0).choice(engine.I, min(DUMP_ROWS, engine.I), replace=False))
    sel = torch.from_numpy(items).to(engine.device)
    for name, p in zip(("W_q0", "W_q1", "W_p0", "W_p1", "b_q0", "b_q1", "b_p0", "b_p1"), engine.vae.params):
        p = p[sel] if name == "W_q0" else p[:, sel] if name == "W_p1" else p
        out["gen_" + name] = p.detach().float().cpu().numpy()
    for name, p in zip(("w1", "b1", "w2", "b2", "w3", "b3", "w4", "b4"), engine.disc.d_params):
        out["disc_" + name] = p.detach().float().cpu().numpy()
    return out


def save_outputs(out_dir, arrays):
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def cpu_baseline(tabs, n_steps, n_items):
    """The reference's CPU data flow (oracle/cpu_step.py) on a bounded sample of the same workload."""
    import torch
    from oracle.cpu_step import CpuGanStep
    step = CpuGanStep(n_items, H0, H1, H2, H3, LR, LAM)
    N = len(tabs["indptr"]) - 1
    cb = min(BATCH, CPU_BATCH_CAP)   # the dense fp32 [B, I] restatement is bounded to CPU_BATCH_CAP users per step
    step.step(tabs, 0, min(cb, N))  # warm-up (thread pools, allocator)
    t0 = time.perf_counter()
    users = 0
    parts = {"t_a": 0.0, "t_d": 0.0, "t_g": 0.0}
    for i in range(n_steps):
        b0 = ((i + 1) * cb) % max(cb, N - cb + 1)
        r = step.step(tabs, b0, min(N, b0 + cb))
        users += min(N, b0 + cb) - b0
        for k in parts:
            parts[k] += r[k]
    dt = time.perf_counter() - t0
    return dict(value=users / dt, unit="users/s", cores=torch.get_num_threads(), kind="port",
                sample="%d GAN steps (A+D+G) of %d users at the %s shape, dense fp32 PyTorch-CPU restatement of the TF graph + the "
                       "reference's host sampling loop; %.2f s/step (A %.2f, D %.2f, G %.2f)"
                       % (n_steps, cb, CONFIG, dt / n_steps, parts["t_a"] / n_steps, parts["t_d"] / n_steps, parts["t_g"] / n_steps),
                host_cpu_count=os.cpu_count())


def config_shape():
    """(n_users, n_items) of the selected configuration."""
    if CONFIG == "askubuntu":
        return 10001, 1000
    if CONFIG == "x1m":
        return X1M_USERS, X1M_ITEMS
    syn = importlib.import_module("long-tail-gan_b200.synthetic")
    N, I, deg = syn.CONFIGS[CONFIG]
    return N, I


def config_tables(n_users):
    """Side tables of the first n_users users of the selected configuration."""
    if CONFIG == "askubuntu":
        import numpy as np
        dp = importlib.import_module("long-tail-gan_b200.data_processing")
        tabs = dp.tables_from_golden(np.load(GOLD))
        return tabs
    syn = importlib.import_module("long-tail-gan_b200.synthetic")
    if CONFIG == "x1m":
        indptr, indices = syn.make_interactions(n_users, X1M_ITEMS, X1M_DEG, seed=7)
        return syn.make_side_tables(indptr, indices, X1M_ITEMS, seed=7)
    return syn.make_config(CONFIG, n_users=n_users)


def select_config(args):
    global CONFIG, BATCH
    CONFIG = args.config
    BATCH = args.batch if args.batch > 0 else BENCH_CONFIGS[CONFIG]["batch"]


def workload_config(world):
    N, I = config_shape()
    return dict(workload="%s: %d users x %d items, VAE 600-200, batch %d per GPU, GAN step = A + D + G" % (BENCH_CONFIGS[CONFIG]["label"], N, I, BATCH),
                users=N, items=I, batch_per_gpu=BATCH, global_batch=BATCH * world, parallelism="dp%d" % world,
                disc="h0..h3 = %d/%d/%d/%d" % (H0, H1, H2, H3), ganlambda=LAM,
                l2_policy="per-step working set (weights + Adam state, ~0.8 GB touched) exceeds the 126 MB L2; timed steps cycle over "
                          "%d distinct user batches; no explicit flush" % N_BENCH_BATCHES)


def run_reference(args, rank, world):
    """`--impl reference`: rank 0 times the reference's CPU path (port; TensorFlow is not installable here)."""
    if rank != 0:
        return
    import torch
    # torch.distributed.run exports OMP_NUM_THREADS=1 to its workers; the reference arm is a CPU job that owns the whole host
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    N, I = config_shape()
    n_steps = max(1, min(args.steps, 8))
    cpu_batch = min(BATCH, CPU_BATCH_CAP)
    tabs = config_tables(cpu_batch * (n_steps + 2))
    cb = cpu_baseline(tabs, n_steps, I)
    line = dict(impl="reference", metric="gan_step_users_per_sec", value=cb["value"], unit="users/s", n_gpus=world, steps=n_steps,
                warmup=1, ms_per_step=1e3 * min(BATCH, CPU_BATCH_CAP) / cb["value"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="fp32",
                data="real (bundled sample)" if CONFIG == "askubuntu" else "synthetic", config=workload_config(world), cpu_baseline=cb,
                e2e=dict(value=cb["value"], unit="users/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
    print(json.dumps(line))


def run_x1m(args, rank, world, local_rank):
    """BASELINE configs[4]: the catalog-sharded engine (vocab_parallel.py). Same timing contract; `value` = users per second of the
    whole job (every rank works on the same users, each on its item shard: strong scaling over the catalog)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pkg = importlib.import_module("long-tail-gan_b200")
    pkg._lib.build()
    syn = importlib.import_module("long-tail-gan_b200.synthetic")
    dis = importlib.import_module("long-tail-gan_b200.discriminator")
    eng = importlib.import_module("long-tail-gan_b200.engine")
    vp = importlib.import_module("long-tail-gan_b200.vocab_parallel")
    ops = importlib.import_module("long-tail-gan_b200.ops")
    ops.init()
    I, nb = X1M_ITEMS, 4
    indptr, indices = syn.make_interactions(BATCH * nb, I, X1M_DEG, seed=7)
    tabs = syn.make_side_tables(indptr, indices, I, seed=7)
    data, vae, lo, hi = vp.build_shard(tabs, I, rank, world, BATCH)
    disc = dis.Discriminator(I, I, H0, H1, H2, H3, seed=4242)
    engine = vp.CatalogShardedEngine(vae, disc, data.max_B, data.max_P, I, lo, rank, world, seed=2026, lr=LR, lam=LAM, max_active=data.max_active,
                                     use_graphs=not args.no_graphs)
    eng.pin_host_inputs(data)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step(i):
        engine.run_step(data, i % nb)

    for i in range(max(args.warmup, 3)):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    k0 = engine.kernels_launched
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    launches = engine.kernels_launched - k0
    # end to end: the batch's index arrays come from pinned host memory, the loss scalars go back, every step
    host_scal = torch.zeros(2, ops.NSCAL, dtype=torch.float32).pin_memory()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h2d = 0
    f0.record()
    for i in range(args.steps):
        h2d += eng.upload_batch(data.batches[i % nb])
        step(i)
        host_scal.copy_(engine.scal_all[:2], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        assert np.isfinite(host_scal[0, ops.S_NLL_SUM].item())
    f1.record()
    barrier()
    t = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_e2e = float(t.item())
    clocks = sampler.stop() if rank == 0 else None

    def timed(fn, n):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(i)
        b.record()
        barrier()
        tt = torch.tensor([a.elapsed_time(b) / n], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())
    for i in range(nb):   # the timed steps ran one graph per batch; capture the per-phase graphs before timing them
        engine.run_phase_a(data, i); engine.run_d_step(data, i); engine.run_g_step(data, i)
    t_a = timed(lambda i: engine.run_phase_a(data, i % nb), 8)
    t_d = timed(lambda i: engine.run_d_step(data, i % nb), 8)
    t_g = timed(lambda i: engine.run_g_step(data, i % nb), 8)
    step(0)
    L = engine.last_losses(BATCH)
    # ranking evaluation over the sharded catalog: local top-100 per shard + merge
    tr_p, tr_i, te_p, te_i = syn.make_eval_split(1000, I, X1M_DEG)
    engine.evaluate(tr_p, tr_i, te_p, te_i)
    barrier()
    t0 = time.perf_counter()
    m = engine.evaluate(tr_p, tr_i, te_p, te_i)
    barrier()
    t_eval = time.perf_counter() - t0
    if rank == 0:
        hb, _ = measured_peaks("hbm_gbs")
        tc, _ = measured_peaks("bf16_tflops_sustained")
        users = BATCH * args.steps
        n_u = BATCH * nb
        ip = np.asarray(tabs["indptr"], dtype=np.int64); cp = np.asarray(tabs["cand_ptr"], dtype=np.int64)
        roof = step_roofline(hi - lo, BATCH, float(ip[n_u] - ip[0]) / n_u / world, float(cp[n_u] - cp[0]) / n_u,
                             float(np.mean([b["Pr"] for b in data.batches])) / world, float(np.mean([b["K"] for b in data.batches])) / world,
                             t_a, t_d, t_g, hb, tc, world=1, t_step=ms / args.steps)
        cfg = dict(workload="%s: %d users x %d items over %d GPU(s) (%d items per shard), VAE 600-200, batch %d (the same users on every rank), "
                            "GAN step = A + D + G" % (BENCH_CONFIGS[CONFIG]["label"], X1M_USERS, I, world, hi - lo, BATCH),
                   users=X1M_USERS, items=I, items_per_gpu=hi - lo, batch_per_gpu=BATCH, global_batch=BATCH, parallelism="vp%d" % world,
                   disc="h0..h3 = %d/%d/%d/%d" % (H0, H1, H2, H3), ganlambda=LAM,
                   exchange=("inside the step's CUDA graph: " if not args.no_graphs else "") + "torch.distributed (NCCL) all-reduce of [B,600] activations x2, all-gather of per-row softmax statistics [B,4], "
                            "all-reduce of the candidate logits and of the 161 k discriminator gradients; no weight or weight-gradient traffic",
                   l2_policy="per-step working set (shard weights + Adam state, %.1f GB) exceeds the 126 MB L2; %d distinct batches" %
                             (30.0 * 1200 * (hi - lo) / 1e9, nb))
        line = dict(metric="gan_step_users_per_sec", value=users / (ms * 1e-3), unit="users/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=ms / args.steps, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="bf16", data="synthetic",
                    gpu_launches=launches, config=cfg, clocks=clocks,
                    e2e=dict(value=users / (ms_e2e * 1e-3), unit="users/s", h2d_bytes_per_step=h2d // args.steps, d2h_bytes_per_step=2 * ops.NSCAL * 4,
                             ms_per_step=ms_e2e / args.steps),
                    phases_ms=dict(A=t_a, D=t_d, G=t_g), step_roofline=roof, graphs=not args.no_graphs,
                    roofline=dict(bound=roof["G"]["bound"], kernel="G update of the catalog shard (per GPU; SURVEY 8d model on the shard)",
                                  achieved=(roof["G"]["bytes"] / (t_g * 1e-3) / 1e9) if roof["G"]["bound"] == "hbm" else roof["G"]["flops"] / (t_g * 1e-3) / 1e12,
                                  peak=hb if roof["G"]["bound"] == "hbm" else tc, unit="GB/s" if roof["G"]["bound"] == "hbm" else "TFLOP/s",
                                  frac=roof["G"]["frac"], traffic=None),
                    eval=dict(users_per_sec=1000 / t_eval, users=1000, ms=t_eval * 1e3, ndcg_at_100_random_init=float(np.mean(m["ndcg@100"])),
                              what="fold-in forward over the shards + local exact top-100 per shard + all-gather/merge of 100 (score, id) pairs per rank"),
                    losses_last_step={k: float(v) for k, v in L.items()}, timing=dict(timed_steps=args.steps, block_ms=ms))
        if world > 1:
            line["comm"] = dict(world_size=dist.get_world_size(), backend=dist.get_backend())
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.cuda.synchronize(); dist.barrier()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


def main():
    args = parse()
    select_config(args)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if CONFIG == "x1m":
        run_x1m(args, rank, world, local_rank)
        return
    import numpy as np
    import torch
    import torch.distributed as dist
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    else:
        torch.cuda.set_device(0)
    if args.gpus != world and rank == 0 and world == 1 and args.gpus > 1:
        print("bench.py: --gpus %d requested but WORLD_SIZE=1; launch with torch.distributed.run" % args.gpus, file=sys.stderr)

    pkg = importlib.import_module("long-tail-gan_b200")
    pkg._lib.build()
    syn = importlib.import_module("long-tail-gan_b200.synthetic")
    gen = importlib.import_module("long-tail-gan_b200.generator")
    dis = importlib.import_module("long-tail-gan_b200.discriminator")
    eng = importlib.import_module("long-tail-gan_b200.engine")
    ops = importlib.import_module("long-tail-gan_b200.ops")
    ops.init()

    N, I = config_shape()
    nb = max(1, min(N_BENCH_BATCHES, N // (BATCH * world)))
    # every rank owns its own contiguous slice of users (user-sharded data parallel, weak scaling)
    tabs = config_tables(BATCH * nb * world)
    data = eng.TrainData(batch_size=BATCH, first_batch=rank * nb, max_batches=nb, **tabs)
    vae = gen.MultiVAE([200, 600, I], lam=0.0, random_seed=98765)
    vae.init_weights(98765)
    disc = dis.Discriminator(I, I, H0, H1, H2, H3, seed=4242)
    engine = eng.GanEngine(vae, disc, data.max_B, data.max_P, seed=2026, lr=LR, lam=LAM, use_graphs=not args.no_graphs, world_size=world,
                           B_global=BATCH * world, max_active=data.max_active, rank=rank)
    eng.pin_host_inputs(data)
    if world > 1:
        engine.attach_dp_tables(eng.build_dp_shard_tables(data, tabs["indptr"], tabs["indices"], world, rank, nb, engine.R))

    def step(i):
        bi = i % nb
        engine.run_step(data, bi)   # phase A + D update + G update of this batch, one captured graph

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # graph capture for every batch that the timed region touches (not counted as warm-up)
    for i in range(nb):
        step(i)
    barrier()
    for i in range(args.warmup):
        step(i)
    barrier()
    k0 = engine.kernels_launched
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # The timed region is exactly args.steps steps between two barriers, so the state the timed path leaves behind (and
    # --dump-outputs writes) depends on the arguments alone.
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    k0 = engine.kernels_launched
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    launches = engine.kernels_launched - k0
    outputs = step_outputs(engine, BATCH, world) if args.dump_outputs else None   # before the steps below move the weights on

    # ---- end-to-end: the step's inputs come from pinned host memory, the losses go back to the host, every step ----
    # Software-pipelined like a real input pipeline: while step i computes, the inputs of step i+1 travel host->device on a
    # copy stream (into that batch's own device buffers), and the loss scalars of step i are read back asynchronously and
    # consumed by the host one step later. Every step's H2D and D2H traffic is inside the timed region.
    host_scal = [torch.zeros(2, ops.NSCAL, dtype=torch.float32).pin_memory() for _ in range(2)]
    copy_stream = torch.cuda.Stream()
    comp = torch.cuda.current_stream()

    def e2e_block():
        up_done = [torch.cuda.Event() for _ in range(nb)]
        step_done = [torch.cuda.Event() for _ in range(2)]
        h2d = 0
        losses_seen = 0
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        with torch.cuda.stream(copy_stream):
            h2d += eng.upload_batch(data.batches[0])
            up_done[0].record(copy_stream)
        for i in range(args.steps):
            bi = i % nb
            if i + 1 < args.steps:
                nxt = (i + 1) % nb
                copy_stream.wait_event(step_done[(i + 1) % 2]) if i >= 1 else None   # the previous user of those buffers is long done
                with torch.cuda.stream(copy_stream):
                    h2d += eng.upload_batch(data.batches[nxt])
                    up_done[nxt].record(copy_stream)
            comp.wait_event(up_done[bi])
            step(i)
            host_scal[i % 2].copy_(engine.scal_all[:2], non_blocking=True)
            step_done[i % 2].record(comp)
            if i >= 1:
                step_done[(i - 1) % 2].synchronize()          # the host consumes the losses of the previous step
                losses_seen += int(np.isfinite(host_scal[(i - 1) % 2][0, ops.S_NLL_SUM].item()))
        step_done[(args.steps - 1) % 2].synchronize()
        losses_seen += int(np.isfinite(host_scal[(args.steps - 1) % 2][0, ops.S_NLL_SUM].item()))
        f1.record()
        barrier()
        assert losses_seen == args.steps, "every step's loss must have been read back"
        t = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), h2d

    ms_e2e, h2d = e2e_block()
    clocks = sampler.stop() if rank == 0 else None

    # ---- per-phase split and the dominant kernel (fused Adam over the [I,600] decoder weight), CUDA events, same stream ----
    def timed(fn, n):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    n_ph = max(8, min(args.steps, 32))
    for i in range(nb):   # the timed steps ran one graph per batch; capture the per-phase graphs before timing them
        engine.run_phase_a(data, i); engine.run_d_step(data, i); engine.run_g_step(data, i)
    barrier()
    t_a = timed(lambda i: engine.run_phase_a(data, i % nb), n_ph)
    t_d = timed(lambda i: engine.run_d_step(data, i % nb), n_ph)
    t_g = timed(lambda i: engine.run_g_step(data, i % nb), n_ph)
    n_par = I * 600
    t_adam = timed(lambda i: ops.adam(vae.WdT, vae.WdT_m, vae.WdT_v, engine.dWdT, vae.WdT_b, scal=engine.scal), 50)
    bt0 = data.batches[0]
    t_enc_adam = timed(lambda i: ops.enc_adam(vae.W_q0, vae.W_q0_m, vae.W_q0_v, vae.W_q0_b, I, bt0["slot_of_item"], engine.G_enc,
                                              scal=engine.scal), 50)

    # the fused discriminator forward: its two launches per step (D: real + generated pairs with the head's backward; G: generated
    # pairs, forward only) on the pair tables of batch 0
    dsc = engine.disc
    t_df_d = t_df_g = 0.0
    if engine.fused_disc:
        st_d = ops.STREAM_DISC_DROPOUT
        gw4 = engine.arena_gp[0][dsc._off["w4"][0]: dsc._off["w4"][0] + dsc._off["w4"][1]]
        gb4 = engine.arena_gp[0][dsc._off["b4"][0]: dsc._off["b4"][0] + dsc._off["b4"][1]]
        t_df_d = timed(lambda i: ops.disc_fwd_fused(engine.Xp, engine.Xn, bt0["P"], dsc, bt0["label"], engine.keep_d, engine.seed, st_d,
                                                    engine.words, engine.Hd, engine.y, engine.scal, engine.dz3, gw4, gb4), 30)
        t_df_g = timed(lambda i: ops.disc_fwd_fused(engine.Xp, engine.Xn, bt0["K"], dsc, bt0["label"][bt0["Pr"]:], engine.keep_d, engine.seed,
                                                    st_d, engine.words, engine.Hd, engine.y, engine.scal), 30)

    # max over ranks (device time)
    times = torch.tensor([ms, ms_e2e, t_a, t_d, t_g, t_adam, t_enc_adam, t_df_d, t_df_g], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms, ms_e2e, t_a, t_d, t_g, t_adam, t_enc_adam, t_df_d, t_df_g = [float(x) for x in times.cpu()]

    dp_res = None
    if world > 1 and not args.no_dp_check:
        # driver-visible correctness of the data-parallel step: same global batch on N ranks and on one GPU (dp_check.py)
        dpc = importlib.import_module("long-tail-gan_b200.dp_check")
        bq = min(BATCH, 512)
        try:
            dp_res = dpc.run_check(config_tables(bq * world), I, bq, rank, world, steps=2, lr=1e-3, use_graphs=not args.no_graphs)
        except Exception as e:  # noqa: BLE001
            dp_res = dict(ok=False, error=repr(e)[:300])
    if rank == 0:
        peak, peak_src = measured_peaks()
        users = BATCH * world * args.steps
        adam_bytes = 30.0 * n_par          # p,m,v read+write (24) + fp32 gradient read (4) + bf16 shadow write (2)
        enc_bytes = 26.0 * n_par           # same without a dense gradient read: the compact gradient rows are L2-resident
        traffic = None
        ncu_tab = []
        try:  # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture of one step
            ncu_tab = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_step_table_v0.json")))   # (v0 holds the Adam sweeps too)
            for rec in ncu_tab:
                if "adam_kernel" in rec["kernel"] and "enc_adam" not in rec["kernel"] and rec.get("dram_MB", 0) > 100:
                    traffic = rec["dram_MB"] * 1e6
        except Exception:
            traffic = None
        adam_roof = dict(bound="hbm", kernel="adam_kernel (fused TF-Adam + bf16 shadow over W_dec^T [I,600])",
                         achieved=adam_bytes / (t_adam * 1e-3) / 1e9, peak=peak, unit="GB/s", frac=adam_bytes / (t_adam * 1e-3) / 1e9 / peak,
                         traffic=traffic, traffic_source="profiles/r2_ncu_step_table_v0.json (ncu --set full; writes still resident in L2 at kernel end are not counted)",
                         peak_source=peak_src, algorithmic_bytes_per_launch=adam_bytes, ms_per_launch=t_adam, us_per_step=t_adam * 1e3,
                         how="CUDA events around 50 back-to-back launches on the launching stream after the timed region; each launch "
                             "touches 362 MB (> L2)")
        enc_roof = dict(bound="hbm", kernel="enc_adam_kernel (TF-Adam over W_q0 [I,600], gradient rows fetched through slot_of_item)",
                        achieved=enc_bytes / (t_enc_adam * 1e-3) / 1e9, peak=peak, unit="GB/s", frac=enc_bytes / (t_enc_adam * 1e-3) / 1e9 / peak,
                        algorithmic_bytes_per_launch=enc_bytes, ms_per_launch=t_enc_adam, us_per_step=t_enc_adam * 1e3)
        roof = adam_roof
        roof["others"] = [enc_roof]
        if engine.fused_disc and (t_df_d + t_df_g) > t_adam:
            # By kernel name the fused discriminator forward (two launches per step) now takes the largest share of the step
            # (profiles/r1_launches_summary_v6.txt), so it is the kernel the roofline line is about. It is GEMM-shaped work (three
            # chained tcgen05 MMAs per 128 pairs), so it is rated against the tensor roof -- knowing that with K = 128 / 128 / 408 the
            # MMAs need ~3% of its time and the tanh + counter-hash dropout epilogue (ncu: 21 instructions per activation, IPC 1.5)
            # is what binds. The two HBM-bound Adam sweeps (the floor of a dense-Adam step, SURVEY F7) follow in `others`.
            tpeak, tsrc = measured_peaks("bf16_tflops")
            fl_pair = 2.0 * ((H0 + 1) * H1 + (H0 + 1) * H2 + (H1 + H2 + 1) * H3) + 2.0 * H3
            n_d, n_g = int(bt0["P"]), int(bt0["K"])
            flops = 0.5 * fl_pair * (n_d + n_g)                      # per launch, averaged over the step's two launches
            t_avg = 0.5 * (t_df_d + t_df_g)
            by_pair = 2 * 128 * 2 + dsc.k3 * 2                       # gathered rows in, hidden activation out
            bytes_avg = 0.5 * (n_d * (by_pair + dsc.ld3 * 2) + n_g * by_pair)
            tr = None
            try:
                df = [rec["dram_MB"] * 1e6 for rec in json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_step_table_v2.json")))
                      if "disc_fused_kernel" in rec["kernel"]]
                tr = sum(df) / len(df) if df else None
            except Exception:
                tr = None
            roof = dict(bound="tensor", kernel="disc_fused_kernel (discriminator forward: 3 chained tcgen05 MMAs + tanh/dropout epilogues + head per 128 pairs)",
                        achieved=flops / (t_avg * 1e-3) / 1e12, peak=tpeak, unit="TFLOP/s", frac=flops / (t_avg * 1e-3) / 1e12 / tpeak,
                        traffic=tr, traffic_source="profiles/r2_ncu_step_table_v2.json (ncu --set full of one step, mean of the D and the G launch)",
                        peak_source=tsrc, algorithmic_flops_per_launch=flops, algorithmic_bytes_per_launch=bytes_avg,
                        ms_per_launch=t_avg, us_per_step=(t_df_d + t_df_g) * 1e3,
                        launches=dict(D=dict(pairs=n_d, ms=t_df_d), G=dict(pairs=n_g, ms=t_df_g)),
                        hbm_view=dict(achieved=bytes_avg / (t_avg * 1e-3) / 1e9, peak=peak, unit="GB/s", frac=bytes_avg / (t_avg * 1e-3) / 1e9 / peak),
                        binding_limit="its serial phases and the epilogue instruction stream (tanh + counter-hash dropout, 16 epilogue warps at IPC 1.3; "
                                      "43% of stall samples are one role waiting for another), not the tensor pipe or HBM: "
                                      "profiles/r2_ncu_step_table_v2.txt, profiles/r2_disc_fused_trace.txt",
                        how="CUDA events around 30 back-to-back launches of each of the step's two configurations on the launching stream",
                        others=[adam_roof, enc_roof])
            adam_roof.pop("others", None)
        line = dict(metric="gan_step_users_per_sec", value=users / (ms * 1e-3), unit="users/s", n_gpus=world, steps=args.steps,
                    warmup=args.warmup, ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
                    dtype="bf16", data="real (bundled sample)" if CONFIG == "askubuntu" else "synthetic", config=workload_config(world),
                    e2e=dict(value=users / (ms_e2e * 1e-3), unit="users/s", h2d_bytes_per_step=h2d // args.steps,
                             d2h_bytes_per_step=2 * ops.NSCAL * 4, ms_per_step=ms_e2e / args.steps),
                    gpu_launches=launches, clocks=clocks, roofline=roof,
                    phases_ms=dict(A=t_a, D=t_d, G=t_g, epoch_weighted_users_per_sec=BATCH * world / ((t_a + 10 * t_d + 10 * t_g) * 1e-3)),
                    pairs_per_step=dict(real=int(np.mean([b["Pr"] for b in data.batches])), generated_slots=int(np.mean([b["K"] for b in data.batches]))),
                    graphs=not args.no_graphs, timing=dict(timed_steps=args.steps, block_ms=ms, e2e_block_ms=ms_e2e))
        if world > 1:
            line["dp_check"] = dp_res
            line["comm"] = dict(world_size=dist.get_world_size(), backend=dist.get_backend(), nccl_version=".".join(str(x) for x in torch.cuda.nccl.version()))
            line["config"]["exchange"] = ("our kernels over NVLink peer memory (%s), flag barriers; no NCCL collective in the step"
                                          % ("NVLS multicast stores + in-switch reduction" if engine.peer["dWdT_mc"] else "unicast peer loads/stores")
                                          if engine.peer is not None else "NCCL collectives captured in the step graphs")
        try:   # whole-step roofline (north_star: fraction of roofline for the full GAN step), per GPU
            hb, _ = measured_peaks("hbm_gbs")
            tc, _ = measured_peaks("bf16_tflops_sustained")   # phases are timed inside a long step: the sustained figure applies
            n_u = BATCH * nb
            ip = np.asarray(tabs["indptr"], dtype=np.int64); cp = np.asarray(tabs["cand_ptr"], dtype=np.int64)
            line["step_roofline"] = step_roofline(I, BATCH, float(ip[n_u] - ip[0]) / n_u, float(cp[n_u] - cp[0]) / n_u,
                                                  float(np.mean([b["Pr"] for b in data.batches])), float(np.mean([b["K"] for b in data.batches])),
                                                  t_a, t_d, t_g, hb, tc, world=world, t_step=ms / args.steps)
        except Exception as e:  # noqa: BLE001
            line["step_roofline"] = dict(error=repr(e)[:200])
        if world == 1:
            try:   # reported beside the training metric; never allowed to take the bench line down
                line["eval"] = eval_throughput(engine, tabs)
            except Exception as e:  # noqa: BLE001
                line["eval"] = dict(error=repr(e)[:200])
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(tabs, args.cpu_steps, I)
        if outputs is not None:
            save_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        # NCCL collectives live inside captured CUDA graphs; tearing the process group down under them can block, and
        # there is nothing left to flush: synchronise, meet at a barrier and leave.
        torch.cuda.synchronize()
        dist.barrier()
        sys.stdout.flush(); sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()
