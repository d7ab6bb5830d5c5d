"""The GAN step of Long-Tail-GAN on one B200: phase A (generator inference + niche sampling + pair construction),
D update, G update and ranking evaluation, as sequences of CUDA kernels launched through the C ABI.

This replaces the body of the reference's epoch loop (Codes/train.py:192-348) and test loop (Codes/test.py:138-171):
every `sess.run` site becomes one method below, the host NumPy loops (train.py:212-251) become ltg_sample_pairs, and
the dense fp32/fp64 feeds (X, generated_tags mask) become CSR / index lists that stay on the device.

Device-resident step state (`words`, `scal`) makes every method CUDA-graph capturable: nothing the kernels need comes
from the host after the launch arguments are fixed (RNG step, Adam bias correction and KL anneal are advanced on the
device by ltg_step_advance). `GanEngine.run_*` therefore capture one graph per (phase, batch) on first use and replay it.
"""
import numpy as np
import torch

from . import ops
from .generator import H, L


def _pad(n, q):
    return (n + q - 1) // q * q


def allow_mask(allow, n_items):
    """`allow` as an iterable of item ids or a boolean mask of length n_items -> boolean mask [n_items]."""
    a = allow if isinstance(allow, np.ndarray) else np.asarray(list(allow))
    if a.dtype == bool:
        if a.shape != (n_items,):
            raise ValueError("a boolean allow mask must have shape (%d,), got %s" % (n_items, a.shape))
        return a
    ids = a.astype(np.int64).reshape(-1)
    if ids.size and (ids.min() < 0 or ids.max() >= n_items):
        raise ValueError("allowed item ids must lie in [0, %d)" % n_items)
    m = np.zeros(n_items, dtype=bool)
    m[ids] = True
    return m


def allow_bits(allow, n_items, lo=0, hi=None):
    """The allow bitmap of ltg_topk_recommend for items [lo, hi) of an n_items catalog (a catalog shard; default the whole catalog):
    uint32 words, bit j % 32 of word j // 32 set when item lo + j is allowed. A shard packs from the global set, since its bounds need
    not be multiples of 32."""
    hi = n_items if hi is None else hi
    m = allow_mask(allow, n_items)[lo:hi]
    m = np.concatenate([m, np.zeros(-len(m) % 32, dtype=bool)])
    return np.packbits(m, bitorder="little").view("<u4").astype(np.uint32)


class TrainData(object):
    """Everything phase A/D/G need about the training users, resident on the device, plus per-batch index structures.

    Host inputs (NumPy, int32 CSR-style):
      indptr/indices           training interactions (data_processing.load_train_data)
      pop_ptr/pop_items        the user's popular items (train_GAN_popular.csv order), `train.py:91`
      n_niche[u]               number of niche items of the user (= number of draws, train.py:227)
      cand_ptr/cand_items      sorted candidate set USER_TAGS_TO_SAMPLE (data_processing.py:170-224)
      real_ptr/real_niche/real_pop   precomputed real pairs (data_processing.py:227-271)
      eligible[u]              user has both popular and niche items (train.py:213)
      item_valid[i]            item is in ITEM_FEATURE_DICT (data_processing.py:40-70)
    """

    def __init__(self, n_items, indptr, indices, pop_ptr, pop_items, n_niche, cand_ptr, cand_items, real_ptr, real_niche, real_pop,
                 eligible, item_valid, batch_size, device="cuda", uid_start=0, first_batch=0, max_batches=None):
        self.n_items = int(n_items)
        self.N = len(indptr) - 1
        self.batch_size = int(batch_size)
        self.device = torch.device(device)
        self.uid_start = int(uid_start)
        i32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(self.device)  # noqa: E731
        self.h_indptr = np.asarray(indptr, dtype=np.int64)
        self.h_indices = np.asarray(indices, dtype=np.int32)
        self.indptr = i32(indptr); self.indices = i32(indices)
        self.pop_ptr = i32(pop_ptr); self.pop_items = i32(pop_items if len(pop_items) else np.zeros(1))
        self.cand_ptr = i32(cand_ptr); self.cand_items = i32(cand_items if len(cand_items) else np.zeros(1))
        self.item_valid = torch.as_tensor(np.ascontiguousarray(item_valid, dtype=np.uint8)).to(self.device)
        self.coef = torch.zeros(max(1, len(indices)), dtype=torch.float32, device=self.device)
        eligible = np.asarray(eligible, dtype=bool)
        n_draw = np.where(eligible, np.asarray(n_niche, dtype=np.int64), 0)
        cand_len = np.diff(np.asarray(cand_ptr, dtype=np.int64))
        n_draw = np.minimum(n_draw, cand_len)
        real_ptr = np.asarray(real_ptr, dtype=np.int64)
        self.batches = []
        starts = list(range(0, self.N, self.batch_size))[first_batch:]
        if max_batches is not None:
            starts = starts[:max_batches]
        self._host = dict(cand_ptr=np.asarray(cand_ptr, dtype=np.int32), cand_items=np.asarray(cand_items, dtype=np.int32),
                          pop_ptr=np.asarray(pop_ptr, dtype=np.int32), pop_items=np.asarray(pop_items, dtype=np.int32),
                          indptr=np.asarray(indptr, dtype=np.int32))
        for b0 in starts:
            b1 = min(self.N, b0 + self.batch_size)
            self.batches.append(self._make_batch(b0, b1, n_draw, real_ptr, real_niche, real_pop, cand_len))
        self.max_B = max(bt["B"] for bt in self.batches)
        self.max_P = max(bt["P"] for bt in self.batches)
        self.max_K = max(bt["K"] for bt in self.batches)
        self.max_active = max(bt["n_active"] for bt in self.batches)

    def _make_batch(self, b0, b1, n_draw, real_ptr, real_niche, real_pop, cand_len):
        B = b1 - b0
        dev = self.device
        e0, e1 = int(self.h_indptr[b0]), int(self.h_indptr[b1])
        idx = self.h_indices[e0:e1].astype(np.int64)
        rows = np.repeat(np.arange(B, dtype=np.int64), np.diff(self.h_indptr[b0:b1 + 1]))
        order = np.lexsort((rows, idx))  # item-major, then batch row
        # active items of the batch: compact CSC (act_ptr over the active items) + slot_of_item[I] (-1 = not in the batch)
        active, counts = np.unique(idx, return_counts=True)
        act_ptr = np.concatenate([[0], np.cumsum(counts)])
        slot_of_item = np.full(self.n_items, -1, dtype=np.int64)
        slot_of_item[active] = np.arange(len(active))
        samp_ptr = np.concatenate([[0], np.cumsum(n_draw[b0:b1])])
        K = int(samp_ptr[-1])
        r0, r1 = int(real_ptr[b0]), int(real_ptr[b1])
        Pr = r1 - r0
        P = Pr + K
        pair_pop = np.zeros(max(P, 1), dtype=np.int32); pair_niche = np.zeros(max(P, 1), dtype=np.int32)
        label = np.full(max(P, 1), -1, dtype=np.int32)
        pair_pop[:Pr] = real_pop[r0:r1]; pair_niche[:Pr] = real_niche[r0:r1]; label[:Pr] = 0
        t = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(dev)  # noqa: E731
        enc_work = ops.enc_work_list(self.h_indptr[b0:b1 + 1]) if B > 0 else np.zeros(1, dtype=np.int32)
        self._last_host = dict(act_ptr=act_ptr, slot_of_item=slot_of_item, csc_row=rows[order], csc_pos=order + e0, samp_ptr=samp_ptr,
                               enc_work=enc_work, pair_pop=pair_pop[:max(Pr, 1)],
                               pair_niche=pair_niche[:max(Pr, 1)], label=label[:max(Pr, 1)])
        return dict(b0=b0, B=B, uid0=self.uid_start + b0, nnz=e1 - e0, Pr=Pr, K=K, P=P, e0=e0, e1=e1,
                    host_src={k: np.ascontiguousarray(v, dtype=np.int32) for k, v in self._last_host.items()},
                    act_ptr=t(act_ptr), slot_of_item=t(slot_of_item), n_active=int(len(active)),
                    csc_row=t(rows[order] if len(order) else np.zeros(1)), csc_pos=t(order + e0 if len(order) else np.zeros(1)),
                    samp_ptr=t(samp_ptr),
                    pair_pop=t(pair_pop), pair_niche=t(pair_niche), label=t(label),
                    cnt=torch.zeros(1, dtype=torch.int32, device=dev),
                    max_cand=int(cand_len[b0:b1].max()) if B > 0 else 0,
                    samp_order=t(np.argsort(-cand_len[b0:b1], kind="stable")),
                    enc_work=t(enc_work) if B > 0 else None,
                    max_nnz=int(np.diff(self.h_indptr[b0:b1 + 1]).max()) if B > 0 else 0)


def build_dp_shard_tables(data, tabs_indptr, tabs_indices, world, rank, nb_per_rank, R):
    """Data parallel: for every local batch index bi, the interactions of the GLOBAL batch (batch rank_q*nb + bi of every rank q,
    concatenated in rank order) whose item lies in this rank's shard [rank*R, rank*R + R): entry arrays for
    ltg_enc_coef_scatter, per-row uid / 1/sqrt(nnz), and the shard-local slot map for ltg_enc_adam."""
    dev = data.device
    I = data.n_items
    B = data.batch_size
    row0 = rank * R
    nr = max(0, min(I, row0 + R) - row0)
    indptr = np.asarray(tabs_indptr, dtype=np.int64)
    indices = np.asarray(tabs_indices, dtype=np.int64)
    t32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(dev)  # noqa: E731
    out = []
    for bi in range(len(data.batches)):
        rows, items, uids, rnorm = [], [], [], []
        for q in range(world):
            u0 = (q * nb_per_rank + bi) * B
            u1 = min(len(indptr) - 1, u0 + B)
            deg = np.diff(indptr[u0:u1 + 1])
            e0, e1 = indptr[u0], indptr[u1]
            rows.append(np.repeat(np.arange(q * B, q * B + (u1 - u0)), deg))
            items.append(indices[e0:e1])
            uu = np.zeros(B, dtype=np.int64); uu[: u1 - u0] = data.uid_start + np.arange(u0, u1)
            rn = np.zeros(B, dtype=np.float32); rn[: u1 - u0] = 1.0 / np.sqrt(np.maximum(deg, 1e-12)).astype(np.float32)
            uids.append(uu); rnorm.append(rn)
        rows = np.concatenate(rows); items = np.concatenate(items)
        sel = (items >= row0) & (items < row0 + nr)
        rows, items = rows[sel], items[sel]
        active = np.unique(items)
        slot_local = np.full(max(nr, 1), -1, dtype=np.int64)
        slot_local[active - row0] = np.arange(len(active))
        out.append(dict(e_row=t32(rows if len(rows) else np.zeros(1)), e_item=t32(items if len(items) else np.zeros(1)),
                        e_slot=t32(slot_local[items - row0] if len(items) else np.zeros(1)), n_entries=int(len(rows)),
                        row_uid=torch.as_tensor(np.concatenate(uids)).to(dev), row_rnorm=torch.as_tensor(np.concatenate(rnorm)).to(dev),
                        slot_local=t32(slot_local), n_active=int(len(active))))
    return out


def pin_host_inputs(data):
    """Pinned host mirrors of everything one step consumes, per batch (used by the end-to-end path: the step's inputs are
    copied host->device inside the timed region). Returns total bytes per batch in bt["h2d_bytes"]."""
    h = data._host
    for bt in data.batches:
        b0, B = bt["b0"], bt["B"]
        c0, c1 = int(h["cand_ptr"][b0]), int(h["cand_ptr"][b0 + B])
        p0, p1 = int(h["pop_ptr"][b0]), int(h["pop_ptr"][b0 + B])
        pairs = []

        def add(dst, src):
            src = torch.as_tensor(np.ascontiguousarray(src, dtype=np.int32))
            if src.numel() == 0:
                return
            pairs.append((dst, src.pin_memory()))

        add(data.indptr[b0: b0 + B + 1], h["indptr"][b0: b0 + B + 1])
        add(data.indices[bt["e0"]: bt["e1"]], data.h_indices[bt["e0"]: bt["e1"]])
        add(data.cand_ptr[b0: b0 + B + 1], h["cand_ptr"][b0: b0 + B + 1])
        add(data.cand_items[c0:c1], h["cand_items"][c0:c1])
        add(data.pop_ptr[b0: b0 + B + 1], h["pop_ptr"][b0: b0 + B + 1])
        add(data.pop_items[p0:p1], h["pop_items"][p0:p1])
        hs = bt["host_src"]
        Pr = bt["Pr"]
        for k in ("act_ptr", "slot_of_item", "csc_row", "csc_pos", "samp_ptr", "enc_work"):
            if bt[k] is not None:
                add(bt[k], hs[k])
        if Pr > 0:
            for k in ("pair_pop", "pair_niche", "label"):
                add(bt[k][:Pr], hs[k][:Pr])
        bt["h2d"] = pairs
        bt["h2d_bytes"] = int(sum(src.numel() * 4 for _, src in pairs))


def upload_batch(bt):
    """Asynchronous host->device copy of one batch's inputs from pinned memory (current stream)."""
    for dst, src in bt["h2d"]:
        dst.copy_(src, non_blocking=True)
    return bt["h2d_bytes"]


class _EvalWorkspace(object):
    """Activation buffers of GanEngine.evaluate (attribute names as in the engine: h1, mulv, z, zmu, h2, ...)."""


class GanEngine(object):
    """Owns the workspaces and runs phase A / D / G / evaluation for one (vae, discriminator) pair."""

    def __init__(self, vae, disc, max_B, max_P=1, seed=0, lr=1e-4, lam=1.0, keep_vae=0.75, keep_d=0.7, total_anneal_steps=20000,
                 anneal_cap=0.2, B_global=None, use_graphs=True, world_size=1, max_active=None, rank=0):
        ops.init()
        self.world_size = int(world_size)
        self.rank = int(rank)
        self.kernels_launched = 0
        self._kcount = {}
        self.vae, self.disc = vae, disc
        self.I = vae.n_items
        self.ld = _pad(self.I, 8)
        self.nblk = ops.dec_logits_nblk_max(self.I)  # softmax partials per row: at most (128-column tile) x (chunk phase); a launch
        # writes ops.dec_logits_nblk(B, I) of them (tile width chosen per shape) and the row passes are told that count
        self.seed, self.lr, self.lam = int(seed), float(lr), float(lam)
        self.keep_vae, self.keep_d = float(keep_vae), float(keep_d)
        self.total_anneal_steps, self.anneal_cap = float(total_anneal_steps), float(anneal_cap)
        self.B_global = B_global
        self.use_graphs = use_graphs
        self.device = vae.device
        self.max_B, self.max_P = int(max_B), int(max(1, max_P))
        self.max_active = int(self.I if max_active is None else max(1, max_active))
        # words[0] rng step, [1] Adam t, [2] G-update count; [4], [5], [6]: the rng step of the current phase A / D update / G update
        # (snapshots written by ltg_step_advance: each phase's kernels read their own word, so the G forward may run beside the D update)
        self.words = torch.zeros(8, dtype=torch.int32, device=self.device)
        self.w_a, self.w_d, self.w_g = self.words[4:5], self.words[5:6], self.words[6:7]
        # per-step scalars: row 0 for the G update, row 1 for the D update (same reason), row 2 scratch for phase A (its forward
        # accumulates a KL sum nobody reads: train.py:200 fetches generator_out only)
        self.scal_all = torch.zeros(3, ops.NSCAL, dtype=torch.float32, device=self.device)
        self.scal, self.scal_d, self.scal_a = self.scal_all[0], self.scal_all[1], self.scal_all[2]
        self._graphs = {}
        # Side streams: independent branches of a step (captured as parallel branches of the CUDA graph). Kernel nodes inherit the
        # priority of the stream they were captured on: the critical chain (capture stream) is highest, the G forward that runs beside
        # the D update next, then the small weight-gradient GEMMs, then the HBM-bound sweeps (decoder weight gradient + Adam, early
        # encoder Adam), whose short-lived CTAs fill whatever the chain leaves free (LTG_GRAPH_PRIORITY=0: everything default priority)
        import os
        prio = os.environ.get("LTG_GRAPH_PRIORITY", "1") != "0"
        mk = lambda p: torch.cuda.Stream(device=self.device, priority=(p if prio else 0))  # noqa: E731
        self.s1 = mk(-1)   # decoder weight gradient + Adam sweep / discriminator forward of the G update
        self.s2 = mk(-2)   # small weight-gradient GEMMs
        self.s3 = mk(-3)   # run_step: the G update's VAE forward beside the D update
        self.s4 = mk(0)    # Adam over the encoder rows that get no gradient from this batch
        self.s5 = mk(-1)   # decoder Adam, chunk by chunk behind the weight-gradient GEMM of branch s1
        self.s6 = mk(0)    # clearing Xc behind its consumer
        self.s7 = mk(-2)   # run_step: the real pairs' half of the D forward beside phase A
        self.split_d = int(os.environ.get("LTG_SPLIT_D", "0"))
        # split-K of the discriminator's weight-gradient GEMMs (their partials are summed by the Adam kernel; at most d_splits_max = 32)
        self.d_sp3 = max(1, min(32, int(os.environ.get("LTG_D_SP3", "12"))))
        self.d_sp = max(1, min(32, int(os.environ.get("LTG_D_SP", "16"))))
        self.small_adam_early = os.environ.get("LTG_SMALL_ADAM_EARLY", "1") != "0"
        self.dec_chunks = int(os.environ.get("LTG_DEC_CHUNKS", "1"))
        self._cap_stream = mk(-5) if prio else None
        self.overlap = True
        # The dense TF-Adam sweep over W_q0 (F7) moves every row, but rows of items absent from the batch (two thirds at batch 500)
        # have a zero gradient: their update depends on nothing the step computes, so it is issued at the START of the G update and
        # runs while the latency-bound forward chain leaves HBM idle; only the active rows wait for the backward pass.
        self.early_adam = os.environ.get("LTG_EARLY_ADAM", "1") != "0"
        self.overlap_dg = os.environ.get("LTG_OVERLAP_DG", "1") != "0"   # run_step: G forward beside the D update
        self.adam_after_mid = os.environ.get("LTG_ADAM_AFTER_MID", "0") != "0"
        # Decoder wgrad GEMM with the Adam step as its epilogue (EpiAdam, ltg_wgrad_adam): correct (tests) and 96 MB/step less HBM
        # traffic, but measured SLOWER than wgrad GEMM (38 us) + streaming Adam (58 us): 112 us, 2.9 TB/s -- the 16 epilogue warps
        # walk load -> update -> store chunk by chunk and cannot keep enough HBM requests in flight. Kept off until the epilogue is
        # restructured (TMA-staged p/m/v tiles).
        self.fused_wgrad_adam = False
        self.fused_disc = ops.disc_fused_supported(self.disc)   # one tcgen05 kernel for the discriminator forward (disc_fused.cu)
        # ... and optionally the backward down to dz12 in the same tile (fourth MMA on the resident dz3 tile). Measured at the bench shape:
        # 98 us for forward + dz12 fused vs 65 + 36 us as two kernels, step 0.519 vs 0.513 ms -- the tile is bound by its epilogue warps
        # (tools/disc_trace.py: 30 of 40 us per tile are tanh/dropout/head/dact epilogues at IPC ~1.2), not by the GEMM it absorbs: off.
        self.fused_dz12 = os.environ.get("LTG_FUSED_DZ12", "0") != "0"
        self.reuse_gather = os.environ.get("LTG_REUSE_GATHER", "1") != "0"   # run_step: one embedding gather for the D and the G update
        self.is_dae = bool(getattr(vae, "is_dae", False))   # MultiDAE (MultiVAE.py:11-92): tanh middle, no KL, unfused GEMM chain
        if self.is_dae:
            assert self.world_size == 1, "MultiDAE runs on the single-GPU engine"
        self.fused_mid = not self.is_dae   # fused 600->400->200->600 middle instead of two GEMMs + element-wise launches ...
        # ... on tcgen05 (mid_tc.cu: one CTA per 128 rows x column third) for large batches, where streaming the weights once per 128
        # rows pays; at batch 500 the 12 CTAs of that kernel are a serial L2-latency chain (38 us vs 16 us measured) and the mma.sync
        # kernels (mid_kernels.cu, 160 CTAs) win. LTG_MID_TC=0/1 forces either.
        mt = os.environ.get("LTG_MID_TC", "")
        self.mid_tc = (self.max_B >= 4096) if mt == "" else (mt != "0")
        self._alloc()
        self.eps_inject = None  # optional [B, L] fp32 tensor used instead of the Philox normal (parity tests)

    def _alloc(self):
        dev, B, P, I, ld = self.device, self.max_B, self.max_P, self.I, self.ld
        bf = dict(dtype=torch.bfloat16, device=dev)
        f32 = dict(dtype=torch.float32, device=dev)
        d = self.disc
        # VAE activations
        self.h1 = torch.zeros(B, H, **bf)
        self.enc_ws = torch.zeros(B, H, **f32)          # split-row accumulator of the encoder gather (self-cleaning)
        self.enc_cnt = torch.zeros(B, dtype=torch.int32, device=dev)
        self.mulv = torch.zeros(B, 2 * L, **f32)
        self.z = torch.zeros(B, L, **bf)
        self.zmu = torch.zeros(B, L, **f32)
        self.h2 = torch.zeros(B, 608, **bf)
        self.h2[:, H] = 1.0  # ones column: wgrad's column 600 becomes the decoder-bias gradient
        self.logits = torch.zeros(B, ld, **bf)
        self.dl = torch.zeros(B, ld, **bf)
        self.partial = torch.zeros(self.nblk, B, 2, **f32)
        self.lse = torch.zeros(B, **f32); self.xw = torch.zeros(B, **f32); self.su = torch.zeros(B, **f32)
        self.dWdT = None  # set below (a view of the padded all-gather/reduce-scatter buffer under data parallelism)
        self.dh2pre = torch.zeros(B, H, **bf)
        self.dmulv = torch.zeros(B, 2 * L, **bf)
        self.dh1pre = torch.zeros(B, H, **f32)
        self.G_enc = torch.zeros(self.max_active, H, **f32)   # compact encoder gradient: one row per active item of the batch
        self.ld_xc = _pad(self.max_active, 8)
        self.Xc = torch.zeros(B, self.ld_xc, **bf)            # dense dropout/normalisation coefficients over the active items
        self.dh1pre_b = torch.zeros(B, H, **bf)
        if self.world_size > 1:
            # Sharded optimizer (data parallel): the two [I,600] matrices are row-sharded over the ranks. Gradients are
            # reduce-scattered, every rank runs Adam on its R rows only (Adam HBM traffic / N) and the bf16 shadows are
            # all-gathered (2 B/param on the wire instead of 4). Buffers are padded to I_pad = R * world rows.
            N = self.world_size
            self.R = (I + N - 1) // N
            self.I_pad = self.R * N
            self.row0 = self.rank * self.R
            self.nrows = max(0, min(I, self.row0 + self.R) - self.row0)
            self.dWdT_full = torch.zeros(self.I_pad, H, **f32)
            self.dWq0_full = torch.zeros(self.I_pad, H, **f32)
            self.dW_q0 = self.dWq0_full[:I]
            self.g_dec_shard = torch.zeros(self.R, H, **f32)
            self.g_enc_shard = torch.zeros(self.R, H, **f32)
            self.WdT_b_full = torch.zeros(self.I_pad, H, **bf); self.WdT_b_shard = torch.zeros(self.R, H, **bf)
            self.Wq0_b_full = torch.zeros(self.I_pad, H, **bf); self.Wq0_b_shard = torch.zeros(self.R, H, **bf)
            self.WdT_b_full[:I].copy_(self.vae.WdT_b); self.Wq0_b_full[:I].copy_(self.vae.W_q0_b)
            self.vae.WdT_b = self.WdT_b_full[:I]      # the compute path reads the all-gathered shadows
            self.vae.W_q0_b = self.Wq0_b_full[:I]
            r0, nr = self.row0, self.nrows
            self.WdT_b_shard[:nr].copy_(self.WdT_b_full[r0:r0 + nr]); self.Wq0_b_shard[:nr].copy_(self.Wq0_b_full[r0:r0 + nr])
            # encoder gradient by activation exchange (see _g_backward): all-gathered dh1pre + locally rebuilt coefficients
            self.dp_tables = None                      # set by attach_dp_tables()
            self.dh1_glob = torch.zeros(N * B, H, **bf)
            self.ld_xcg = _pad(max(1, min(self.R, self.max_active * N)), 8)
            self.Xc_glob = torch.zeros(N * B, self.ld_xcg, **bf)
            self.G_shard = torch.zeros(max(1, min(self.R, self.max_active * N)), H, **f32)
            self.peer = None
            self._setup_peer()
        else:
            self.dW_q0 = None
            self.peer = None
        self.dWdT = self.dWdT_full[:I] if self.world_size > 1 else torch.zeros(I, H, **f32)
        # split-K partials of the decoder dgrad (summed by the tanh-backward kernel that consumes them: no atomics, no memset)
        self.dgrad_splits = ops.actual_splits(I, ops.pick_splits(B, H, I, 128))
        self.dh2_part = torch.zeros(self.dgrad_splits, B, H, **f32)
        self.dz = torch.zeros(B, L, **f32)
        self.dzpre = torch.zeros(B, L, **bf)     # MultiDAE: gradient at the pre-activation of the 200-wide layer
        self.dh1 = torch.zeros(B, H, **f32)
        # split-K partials of the three discriminator weight-gradient GEMMs (summed by the Adam kernel)
        self.d_splits_max = 32
        self.arena_gp = torch.zeros(self.d_splits_max, d.arena_n, **f32)
        # discriminator
        self.Xp = torch.zeros(P, 128, **bf); self.Xn = torch.zeros(P, 128, **bf)
        self.Hd = torch.zeros(P, d.k3, **bf)
        self.Hd[:, d.one3] = 1.0   # ones column: row `one3` of W3 is the fc1 bias
        self.Y3 = torch.zeros(P, d.ld3, **bf)
        self.y = torch.zeros(P, **f32)
        self.dz3 = torch.zeros(P, d.ld3, **bf)
        self.dz12 = torch.zeros(P, d.k3, **bf)

    # ------------------------------------------------------------------------------------------------------------
    # building blocks
    # ------------------------------------------------------------------------------------------------------------
    def _fork(self, side):
        """Start a parallel branch on `side` that depends on everything issued so far on the current stream."""
        if not self.overlap:
            return torch.cuda.stream(torch.cuda.current_stream())
        side.wait_stream(torch.cuda.current_stream())
        return torch.cuda.stream(side)

    def _join(self, side):
        if self.overlap:
            torch.cuda.current_stream().wait_stream(side)

    def _vae_forward(self, data, bt, is_training, keep, stash=True, indptr=None, indices=None, coef=None, uid0=None, B=None, max_nnz=None,
                     before_decoder=None):
        """MultiVAE.forward_pass (MultiVAE.py:175-186) up to the logits and their softmax statistics. before_decoder: optional callable
        issued between the middle and the decoder GEMM (run_step forks a side branch there)."""
        v = self.vae
        wstep = self.w_g if is_training else self.w_a
        scal = self.scal if is_training else self.scal_a
        own_rows = indptr is None and B is None      # the batch's own CSR rows: its precomputed chunk list applies
        B = bt["B"] if B is None else B
        indptr = data.indptr[bt["b0"]: bt["b0"] + B + 1] if indptr is None else indptr
        indices = data.indices if indices is None else indices
        coef = data.coef if coef is None else coef
        uid0 = bt["uid0"] if uid0 is None else uid0
        work = bt.get("enc_work") if own_rows else None
        # Xc (dense coefficient matrix, G step only) is all-zero here: the G backward clears it again right after its consumer
        ops.enc_gather_fwd(indptr, indices, None, B, self.I, uid0, v.W_q0_b, v.view("b_q0"), keep, self.seed, 0, wstep, self.h1, coef,
                           bt["max_nnz"] if max_nnz is None else max_nnz, self.enc_ws, self.enc_cnt,
                           bt["slot_of_item"] if is_training else None, self.Xc if is_training else None, work=work)
        if self.fused_mid:
            ops.vae_mid_fwd(self.h1, v.view("W_q1", "b"), v.view("b_q1"), v.view("W_p0", "b"), v.view("b_p0"),
                            self.eps_inject if is_training else None, B, uid0, 1.0 if is_training else 0.0, self.seed, 0, wstep,
                            self.mulv, self.z, self.zmu, self.h2, scal, tc=self.mid_tc)
        else:
            self._middle_unfused(B, uid0, 1.0 if is_training else 0.0, wstep, scal, self.eps_inject if is_training else None)
        if before_decoder is not None:
            before_decoder()
        # (phase A samples with Gumbel-top-k straight from the logits: the softmax statistics are computed by the G forward only)
        ops.dec_logits_fwd(self.h2, v.WdT_b, v.view("b_p1"), B, self.I, self.logits if stash else None,
                           self.partial if (is_training or not stash) else None)
        return indptr, indices

    def _middle_unfused(self, B, uid0, is_training, wstep, scal, eps=None, ws=None):
        """h1 -> z -> h2 as GEMMs with fused epilogues. MultiVAE (MultiVAE.py:157-181): mu|logvar GEMM, latent head (KL,
        reparameterisation), tanh GEMM. MultiDAE (MultiVAE.py:62-68): two tanh GEMMs. `ws`: the activation buffers (default: the
        training workspaces of this engine; evaluation passes its own, larger ones)."""
        v = self.vae
        ws = self if ws is None else ws
        if self.is_dae:
            ops.gemm(ws.h1, v.view("W_q1", "b"), B, L, H, b_mn=True, bn=64, out_bf16=ws.z, bias=v.view("b_q1"), act=1)
        else:
            ops.gemm(ws.h1, v.view("W_q1", "b"), B, 2 * L, H, b_mn=True, bn=64, out_f32=ws.mulv, bias=v.view("b_q1"))
            ops.latent_fwd(ws.mulv, eps, B, uid0, is_training, self.seed, 0, wstep, ws.z, ws.zmu, scal)
        ops.gemm(ws.z, v.view("W_p0", "b"), B, H, L, b_mn=True, bn=64, out_bf16=ws.h2, bias=v.view("b_p0"), act=1)

    def _eval_workspace(self, rows):
        """Activation buffers of the ranking evaluation, allocated on first use and kept: evaluation is a pure forward, so its batch is
        not tied to the training batch -- a few thousand users per launch instead of 500 (fewer launches per user, full waves in the
        GEMM and one top-k CTA per row over many more rows than SMs)."""
        ws = getattr(self, "_eval_ws", None)
        if ws is not None and ws.rows >= rows:
            return ws
        dev = self.device
        bf = dict(dtype=torch.bfloat16, device=dev); f32 = dict(dtype=torch.float32, device=dev)
        ws = _EvalWorkspace()
        ws.rows = int(rows)
        ws.h1 = torch.zeros(rows, H, **bf)
        ws.enc_ws = torch.zeros(rows, H, **f32)
        ws.enc_cnt = torch.zeros(rows, dtype=torch.int32, device=dev)
        ws.mulv = torch.zeros(rows, 2 * L, **f32)
        ws.z = torch.zeros(rows, L, **bf)
        ws.zmu = torch.zeros(rows, L, **f32)
        ws.h2 = torch.zeros(rows, 608, **bf)
        ws.h2[:, H] = 1.0
        ws.scores = torch.zeros(rows, self.ld, **f32)
        self._eval_ws = ws
        return ws

    def _disc_forward(self, pop, niche, label, P, backward, g_w4=None, g_b4=None, gathered_row0=None):
        """discriminator.py:16-55 on P pairs (real and generated share the weights, so they run as one batch).
        gathered_row0: the embedding rows of these pairs already sit in Xp / Xn from that row on (run_step: the D update gathered the
        generated pairs behind the real ones, the G update reads the same rows instead of gathering them again)."""
        d = self.disc
        seed, kd = self.seed, self.keep_d
        st = ops.STREAM_DISC_DROPOUT
        words, scal = (self.w_d, self.scal_d) if backward else (self.w_g, self.scal)   # D update / G update
        if gathered_row0 is None:
            Xp, Xn = self.Xp, self.Xn
            ops.disc_gather(d.E_b, pop, niche, P, Xp, Xn)
        else:
            Xp, Xn = self.Xp[gathered_row0:], self.Xn[gathered_row0:]
        if self.fused_disc:
            ops.disc_fwd_fused(Xp, Xn, P, d, label, kd, seed, st, words, self.Hd, self.y, scal,
                               self.dz3 if backward else None, g_w4 if backward else None, g_b4 if backward else None,
                               self.dz12 if (backward and self.fused_dz12) else None)
            return
        k1 = d.h0 + 1  # embedding columns + the ones column (bias row of W1 / W2)
        ops.gemm(Xp, d.view("W1", "b"), P, d.h1, k1, lda=128, b_mn=True, bn=ops.pick_bn(P, d.h1), out_bf16=self.Hd, ld_bf16=d.k3,
                 act=1, keep=kd, seed=seed, rng_stream=st, rng_step_dev=words, rng_ld=d.ld1)
        ops.gemm(Xn, d.view("W2", "b"), P, d.h2, k1, lda=128, b_mn=True, bn=ops.pick_bn(P, d.h2), out_bf16=self.Hd[:, d.off2:],
                 ld_bf16=d.k3, act=1, keep=kd, seed=seed, rng_stream=st + 1, rng_step_dev=words, rng_ld=d.ld2)
        ops.gemm(self.Hd, d.view("W3", "b"), P, d.h3, d.k3, b_mn=True, bn=ops.pick_bn(P, d.h3), out_bf16=self.Y3, act=1, keep=kd, seed=seed,
                 rng_stream=st + 2, rng_step_dev=words, rng_ld=d.ld3)
        if backward:
            ops.disc_head(self.Y3, P, d.h3, d.view("w4"), d.view("b4"), label, kd, self.y, scal, self.dz3, g_w4, g_b4)
        else:
            ops.disc_head(self.Y3, P, d.h3, d.view("w4"), d.view("b4"), label, kd, self.y, scal)

    # ------------------------------------------------------------------------------------------------------------
    # phase A: train.py:192-269
    # ------------------------------------------------------------------------------------------------------------
    def phase_a(self, data, bi, advance=True, before_decoder=None, before_sampler=None):
        bt = data.batches[bi]
        B = bt["B"]
        if advance:
            ops.step_advance(self.words, self.scal_a, 0, self.lr, anneal_cap=self.anneal_cap, total_anneal_steps=self.total_anneal_steps,
                             zero=bt["cnt"], snap=self.w_a)   # the sampler's per-user counters are cleared by the same launch
        # train.py:200: sess.run(generator_out) with default placeholders: dropout 0.75 (F4), is_training 0
        self._vae_forward(data, bt, False, self.keep_vae, before_decoder=before_decoder)
        if before_sampler is not None:
            before_sampler()
        if bt["K"] > 0:
            Pr = bt["Pr"]
            ops.sample_pairs(self.logits, B, self.I, bt["uid0"], data.cand_ptr[bt["b0"]: bt["b0"] + B + 1], data.cand_items, bt["samp_ptr"],
                             data.pop_ptr[bt["b0"]: bt["b0"] + B + 1], data.pop_items, data.item_valid, self.seed, 0, self.w_a,
                             bt["pair_niche"][Pr:], bt["pair_pop"][Pr:], bt["label"][Pr:], bt["cnt"], bt["max_cand"], bt["samp_order"])

    # ------------------------------------------------------------------------------------------------------------
    # D update: train.py:300
    # ------------------------------------------------------------------------------------------------------------
    def d_step(self, data, bi):
        self._d_fwd_bwd(data, bi)
        self._d_update()

    def _d_advance(self):
        # (the w4 / b4 gradient slots of partial 0, accumulated by the head with atomics, are cleared by the same launch)
        d = self.disc
        ops.step_advance(self.words, self.scal_d, 1, self.lr, anneal_cap=self.anneal_cap, total_anneal_steps=self.total_anneal_steps,
                         zero=self.arena_gp[0][d._off["w4"][0]:], snap=self.w_d)

    def _d_real_forward(self, data, bi):
        """The REAL pairs of the D update (rows [0, Pr) of the batch's pair list): precomputed tables (train.py:223-224), independent of
        phase A, so run_step issues them on a side branch beside it; _d_fwd_bwd(real_done=True) then runs the generated pairs only.
        Same buffers, same rows, same dropout counters (rng_row0) as the one launch over all P pairs."""
        bt = data.batches[bi]
        d = self.disc
        Pr = bt["Pr"]
        gW = lambda name: self.arena_gp[0][d._off[name][0]: d._off[name][0] + d._off[name][1]]  # noqa: E731
        ops.disc_gather(d.E_b, bt["pair_pop"], bt["pair_niche"], Pr, self.Xp, self.Xn)
        ops.disc_fwd_fused(self.Xp, self.Xn, Pr, d, bt["label"], self.keep_d, self.seed, ops.STREAM_DISC_DROPOUT, self.w_d, self.Hd, self.y,
                           self.scal_d, self.dz3, gW("w4"), gW("b4"), None, rng_row0=0)

    def _d_fwd_bwd(self, data, bi, advance=True, real_done=False):
        bt = data.batches[bi]
        d = self.disc
        P = bt["P"]
        if advance:
            self._d_advance()
        # autodiff of discriminator.py:25-55; every bias gradient is the ones-row of its weight-gradient GEMM.
        # Single GPU: the split-K partials of the three weight-gradient GEMMs go to arena_gp[s] and the Adam kernel sums them.
        # Data parallel: atomic accumulation into arena_g (which is what gets all-reduced).
        k1 = d.h0 + 1
        part = True   # data parallel sums the partials into arena_g before the all-reduce (see _d_step_dp)
        bn3 = ops.pick_bn(d.k3, d.h3, True)
        # fixed split counts (empty splits store zeros): dW3 has 8 output tiles -> 12 splits fill the machine; dW1/dW2 have one tile
        sp3 = self.d_sp3 if part else ops.pick_splits(d.k3, d.h3, P, bn3)
        sp = self.d_sp if part else ops.pick_splits(k1, d.h2, P, 256)
        self._d_parts = max(sp, sp3) if part else 1
        if part:
            gW = lambda name: self.arena_gp[0][d._off[name][0]: d._off[name][0] + d._off[name][1]]  # noqa: E731
            kw = dict(split_stride=d.arena_n)
        else:
            d.arena_g.zero_()
            gW = lambda name: d.view(name, "g")  # noqa: E731
            kw = dict(atomic=True)
        if real_done:
            Pr = bt["Pr"]
            ops.disc_gather(d.E_b, bt["pair_pop"][Pr:], bt["pair_niche"][Pr:], P - Pr, self.Xp[Pr:], self.Xn[Pr:])
            ops.disc_fwd_fused(self.Xp[Pr:], self.Xn[Pr:], P - Pr, d, bt["label"][Pr:], self.keep_d, self.seed, ops.STREAM_DISC_DROPOUT, self.w_d,
                               self.Hd[Pr:], self.y[Pr:], self.scal_d, self.dz3[Pr:], gW("w4"), gW("b4"), None, rng_row0=Pr)
            self._join(self.s7)   # the real pairs' half (branch s7, issued beside phase A)
        else:
            self._disc_forward(bt["pair_pop"], bt["pair_niche"], bt["label"], P, True, g_w4=gW("w4"), g_b4=gW("b4"))
        with self._fork(self.s1):
            ops.gemm(self.Hd, self.dz3, d.k3, d.h3, P, a_mn=True, b_mn=True, splits=sp3, bn=bn3, out_f32=gW("W3"), ld_f32=d.ld3, **kw)  # dW3 (+db3)
        if not (self.fused_disc and self.fused_dz12):   # (the fused kernel has already produced dz12 as its fourth MMA)
            ops.gemm(self.dz3, d.view("W3", "b"), P, d.k3, d.h3, bn=ops.pick_bn(P, d.k3), out_bf16=self.dz12, dact_src=self.Hd,
                     dact_keep=self.keep_d)                                                        # dz12 = (dz3 W3^T) * dact(Hd)
        with self._fork(self.s2):
            ops.gemm(self.Xp, self.dz12, k1, d.h1, P, a_mn=True, b_mn=True, splits=sp, bn=ops.pick_bn(k1, d.h1, True), out_f32=gW("W1"),
                     ld_f32=d.ld1, **kw)                                                           # dW1 (+db1) = Xp^T dz1
        ops.gemm(self.Xn, self.dz12[:, d.off2:], k1, d.h2, P, a_mn=True, b_mn=True, ldb=d.k3, splits=sp, bn=ops.pick_bn(k1, d.h2, True),
                 out_f32=gW("W2"), ld_f32=d.ld2, **kw)                                             # dW2 (+db2) = Xn^T dz2
        self._join(self.s2)
        self._join(self.s1)

    def _d_update(self):
        d = self.disc
        if self.world_size == 1:
            ops.adam(d.arena, d.arena_m, d.arena_v, self.arena_gp, d.arena_b, scal=self.scal_d, n_partials=self._d_parts,
                     partial_stride=d.arena_n)
        else:
            ops.adam(d.arena, d.arena_m, d.arena_v, d.arena_g, d.arena_b, scal=self.scal_d)

    # ------------------------------------------------------------------------------------------------------------
    # G update: train.py:326
    # ------------------------------------------------------------------------------------------------------------
    def g_step(self, data, bi, update=True):
        """Single-GPU G update. The data-parallel variant (run_g_step with world_size > 1) runs the same three parts with
        the two exchange steps in between."""
        self._fuse_update = bool(update) and self.world_size == 1
        self._g_forward(data, bi)
        self._g_backward(data, bi)
        self._fuse_update = False
        if update and self.world_size > 1:
            self._g_update(data, bi)

    def _g_advance(self):
        ops.step_advance(self.words, self.scal, 2, self.lr, anneal_cap=self.anneal_cap, total_anneal_steps=self.total_anneal_steps,
                         zero=self.vae.small_g, snap=self.w_g)   # bias gradients are accumulated atomically: cleared by the same launch

    def _g_early(self, data, bi):
        """Part of the G update that depends on nothing but the step counters: TF-Adam over the encoder rows without a gradient."""
        self._early_done = False
        if not (self.early_adam and self.world_size == 1 and getattr(self, "_fuse_update", False)):
            return
        v = self.vae
        with self._fork(self.s4):
            ops.enc_adam(v.W_q0, v.W_q0_m, v.W_q0_v, v.W_q0_b, self.I, data.batches[bi]["slot_of_item"], self.G_enc, scal=self.scal, rows=1)
        self._early_done = True

    def _g_disc_forward(self, data, bi, reuse_gather=False):
        # y_generated with fresh dropout masks (keep_prob 0.7 is fed in the G step too, train.py:326)
        bt = data.batches[bi]
        Pr, K = bt["Pr"], bt["K"]
        if K > 0:
            self._disc_forward(bt["pair_pop"][Pr:], bt["pair_niche"][Pr:], bt["label"][Pr:], K, False,
                               gathered_row0=Pr if (reuse_gather and self.reuse_gather) else None)

    def _g_forward(self, data, bi):
        bt = data.batches[bi]
        self._g_advance()
        self._g_early(data, bi)
        if bt["K"] > 0:
            # independent of the generator forward, so it runs as a parallel branch
            with self._fork(self.s1):
                self._g_disc_forward(data, bi)
        self._vae_forward(data, bt, True, self.keep_vae)
        if bt["K"] > 0:
            self._join(self.s1)
        # the softmax statistics are fused into the backward's per-user kernel (ltg_dec_row_bwd)

    def _g_backward(self, data, bi):
        bt = data.batches[bi]
        v = self.vae
        B, Pr, K = bt["B"], bt["Pr"], bt["K"]
        Bg = (B if self.B_global is None else self.B_global)
        indptr = data.indptr[bt["b0"]: bt["b0"] + B + 1]
        indices = data.indices
        lam = self.lam if (K > 0 or self.world_size > 1) else 0.0
        samp = (bt["samp_ptr"], bt["pair_niche"][Pr:], bt["label"][Pr:]) if K > 0 else (None, None, None)
        ops.dec_row_bwd(self.partial, ops.dec_logits_nblk(B, self.I), self.logits, B, self.I, Bg, lam, indptr, indices, None, samp[0], samp[1], samp[2],
                        self.lse, self.scal, self.dl)
        # decoder backward: dh2 = dl W_p1^T (split-K over the catalog), dW_p1^T = dl^T [h2 | 1].
        # Branch s1: decoder weight gradient (+ its Adam sweep when the update is fused into this graph, single GPU) -- HBM-bound,
        # runs under the latency-bound chain of small GEMMs of the encoder-side backward on the main stream.
        fuse_update = self.world_size == 1 and getattr(self, "_fuse_update", False)
        dp_comm = self.world_size > 1 and getattr(self, "_dp_comm", False)
        fused_wa = fuse_update and self.fused_wgrad_adam
        # single GPU: the decoder weight gradient and its Adam sweep are cut into row chunks of the catalog and pipelined -- Adam on
        # chunk c (branch s5) runs beside the weight-gradient GEMM of chunk c+1 (branch s1), and reads a gradient chunk that is still
        # in L2 (8 MB per chunk instead of a 48 MB round trip through HBM)
        chunked = fuse_update and not fused_wa and self.dec_chunks > 1
        self._dec_ev = []
        if not fused_wa:
            with self._fork(self.s1):
                if chunked:
                    for r0, nr in self._dec_chunk_rows():
                        ops.gemm(self.dl[:, r0:], self.h2, nr, H + 1, B, a_mn=True, b_mn=True, bn=128, out_f32=self.dWdT[r0:r0 + nr], ld_f32=H,
                                 aux_col=H, aux_out=v.view("b_p1", "g")[r0:])
                        ev = torch.cuda.Event(); ev.record()
                        self._dec_ev.append(ev)
                else:
                    ops.gemm(self.dl, self.h2, self.I, H + 1, B, a_mn=True, b_mn=True, bn=128, out_f32=self.dWdT, ld_f32=H, aux_col=H,
                             aux_out=v.view("b_p1", "g"))
                if dp_comm and self.peer is None:
                    import torch.distributed as dist
                    dist.reduce_scatter_tensor(self.g_dec_shard, self.dWdT_full)
                if dp_comm and self.peer is not None:
                    self._ev_wgrad = torch.cuda.Event()
                    self._ev_wgrad.record()
        ops.gemm(self.dl, v.WdT_b, B, H, self.I, b_mn=True, splits=self.dgrad_splits, bn=128, out_f32=self.dh2_part, ld_f32=H,
                 split_stride=self.max_B * H)
        if fused_wa:
            # single GPU: the decoder weight-gradient GEMM applies Adam in its epilogue (the [I,600] fp32 gradient never reaches
            # HBM). It rewrites the bf16 weights the dgrad GEMM above reads, hence the fork AFTER dgrad; it then runs beside the
            # encoder-side backward chain of the main stream.
            with self._fork(self.s1):
                ops.wgrad_adam(self.dl, self.h2, self.I, H + 1, B, v.WdT, v.WdT_m, v.WdT_v, v.WdT_b, H, aux_col=H, aux_out=v.view("b_p1", "g"),
                               scal=self.scal)
        if dp_comm and self.peer is not None:
            # peer-memory path: once every rank has finished its weight-gradient GEMM and its dgrad GEMM (which reads the bf16
            # weights), ONE kernel sums this rank's rows of all ranks' gradient buffers, runs Adam on them and stores the bf16
            # result into every rank's weight shadow: reduce-scatter + update + all-gather without a collective launch
            if self.overlap:
                self.s1.wait_stream(torch.cuda.current_stream())
            with (torch.cuda.stream(self.s1) if self.overlap else torch.cuda.stream(torch.cuda.current_stream())):
                self._pbar(1)
                if self.nrows > 0:
                    r0, nr = self.row0, self.nrows
                    ops.adam_peer(v.WdT[r0:r0 + nr], v.WdT_m[r0:r0 + nr], v.WdT_v[r0:r0 + nr], self.peer["dWdT"], self.peer["WdT_b"], r0 * H,
                                  self.world_size, scal=self.scal, grads_mc=self.peer["dWdT_mc"], shadows_mc=self.peer["WdT_b_mc"])
        if dp_comm and self.peer is None and self.nrows > 0:
            # Adam on this rank's decoder rows: after the reduce-scatter (same branch) and after dgrad (it reads the bf16 weights;
            # the shard Adam only writes the shard staging buffer, the full shadow is replaced by the all-gather at the end)
            if self.overlap:
                self.s1.wait_stream(torch.cuda.current_stream())
            with (torch.cuda.stream(self.s1) if self.overlap else torch.cuda.stream(torch.cuda.current_stream())):
                r0, nr = self.row0, self.nrows
                ops.adam(v.WdT[r0:r0 + nr], v.WdT_m[r0:r0 + nr], v.WdT_v[r0:r0 + nr], self.g_dec_shard, self.WdT_b_shard, scal=self.scal)
        if dp_comm and self.peer is None:
            # every rank (also one whose shard is empty) joins the all-gather; issued here so it overlaps the encoder-side backward
            if self.overlap:
                self.s1.wait_stream(torch.cuda.current_stream())
            with (torch.cuda.stream(self.s1) if self.overlap else torch.cuda.stream(torch.cuda.current_stream())):
                import torch.distributed as dist
                dist.all_gather_into_tensor(self.WdT_b_full, self.WdT_b_shard)
        if fuse_update and not fused_wa:
            # the Adam sweep rewrites the bf16 decoder weights the dgrad GEMM above reads: order it after dgrad
            if self.overlap:
                self.s1.wait_stream(torch.cuda.current_stream())
            if chunked:
                side = self.s5 if self.overlap else torch.cuda.current_stream()
                if self.overlap:
                    self.s5.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    for (r0, nr), ev in zip(self._dec_chunk_rows(), self._dec_ev):
                        if self.overlap:
                            side.wait_event(ev)
                        ops.adam(v.WdT[r0:r0 + nr], v.WdT_m[r0:r0 + nr], v.WdT_v[r0:r0 + nr], self.dWdT[r0:r0 + nr], v.WdT_b[r0:r0 + nr], scal=self.scal)
            elif self.adam_after_mid and self.overlap and self.fused_mid:
                self._dec_adam_pending = True   # issued below, behind the latency-bound middle of the backward chain
            else:
                with (torch.cuda.stream(self.s1) if self.overlap else torch.cuda.stream(torch.cuda.current_stream())):
                    ops.adam(v.WdT, v.WdT_m, v.WdT_v, self.dWdT, v.WdT_b, scal=self.scal)
        if self.fused_mid:
            # split-K sum + tanh' with full-machine parallelism, then two fused kernels (dz + latent backward; dh1 + tanh' + db_q0);
            # the two weight-gradient GEMMs (contractions over the batch) run on side branches
            ops.tanh_bwd(self.dh2_part, self.h2, B, H, dx_bf16=self.dh2pre, dbias=v.view("b_p0", "g"), n_partials=self.dgrad_splits,
                         partial_stride=self.max_B * H, ld_dy=H)
            with self._fork(self.s2):
                ops.gemm(self.z, self.dh2pre, L, H, B, a_mn=True, b_mn=True, bn=64, out_f32=v.view("W_p0", "g"))
            ops.vae_mid_bwd(self.dh2pre, v.view("W_p0", "b"), v.view("W_q1", "b"), self.mulv, self.zmu, self.h1, B, Bg, -1.0, self.scal,
                            self.dmulv, self.dh1pre, self.dh1pre_b, v.view("b_q1", "g"), v.view("b_q0", "g"), tc=self.mid_tc)
            if getattr(self, "_dec_adam_pending", False):
                # The decoder Adam sweep saturates HBM for ~60 us; the two middle kernels above are L2-latency chains that ran 2.5x
                # slower beside it (34 + 34 us instead of 15 + 12, timeline of round 2). It starts once they are done and then shares
                # HBM with the other bandwidth-bound tail of the step (encoder weight gradient + Adam over the active rows).
                self._dec_adam_pending = False
                self.s1.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(self.s1):
                    ops.adam(v.WdT, v.WdT_m, v.WdT_v, self.dWdT, v.WdT_b, scal=self.scal)
            self._join(self.s2)
            with self._fork(self.s2):
                ops.gemm(self.h1, self.dmulv, H, 2 * L, B, a_mn=True, b_mn=True, bn=64, out_f32=v.view("W_q1", "g"))
                if dp_comm and self.peer is not None:
                    # every small gradient of this rank is final here (the last one, db_p1, comes from the decoder weight-gradient
                    # GEMM on branch s1): exchange + update of the small arena run on this branch, beside the encoder chain
                    torch.cuda.current_stream().wait_event(self._ev_wgrad)
                    self._small_exchange(2)
                    self._small_done = True
        else:
            ops.tanh_bwd(self.dh2_part, self.h2, B, H, dx_bf16=self.dh2pre, dbias=v.view("b_p0", "g"), n_partials=self.dgrad_splits,
                         partial_stride=self.max_B * H, ld_dy=H)
            with self._fork(self.s2):
                ops.gemm(self.z, self.dh2pre, L, H, B, a_mn=True, b_mn=True, bn=64, out_f32=v.view("W_p0", "g"))
            ops.gemm(self.dh2pre, v.view("W_p0", "b"), B, L, H, bn=64, out_f32=self.dz)
            if self.is_dae:   # through z = tanh(.) (MultiVAE.py:66-67); column sums -> db_1
                ops.tanh_bwd(self.dz, self.z, B, L, dx_bf16=self.dzpre, dbias=v.view("b_q1", "g"))
                dmid, q1 = self.dzpre, L
            else:
                ops.latent_bwd(self.dz, self.mulv, self.zmu, B, Bg, -1.0, self.scal, self.dmulv, v.view("b_q1", "g"))
                dmid, q1 = self.dmulv, 2 * L
            self._join(self.s2)
            with self._fork(self.s2):
                ops.gemm(self.h1, dmid, H, q1, B, a_mn=True, b_mn=True, bn=64, out_f32=v.view("W_q1", "g"))
            ops.gemm(dmid, v.view("W_q1", "b"), B, H, q1, bn=64, out_f32=self.dh1)
            ops.tanh_bwd(self.dh1, self.h1, B, H, dx_bf16=self.dh1pre_b, dx_f32=self.dh1pre, dbias=v.view("b_q0", "g"))
        # encoder weight gradient over the batch's active items as a tensor-core GEMM: G = Xc^T dh1pre   [n_active, 600]
        if not (self.world_size > 1 and getattr(self, "_dp_comm", False) and self.dp_tables is not None):
            ops.gemm(self.Xc, self.dh1pre_b, bt["n_active"], H, B, a_mn=True, b_mn=True, bn=ops.pick_bn(bt["n_active"], H), out_f32=self.G_enc)
        with self._fork(self.s6):
            # self-cleaning, off the critical path (own branch: nothing of this step waits for it): the next G forward scatters into an
            # all-zero matrix
            ops.enc_xc_clear(indptr, indices, B, bt["nnz"], bt["slot_of_item"], self.Xc)
        act_exchange = dp_comm and self.dp_tables is not None
        if self.world_size > 1 and not act_exchange:
            ops.enc_wgrad_expand(self.dW_q0, self.I, bt["slot_of_item"], self.G_enc)
        if act_exchange:
            # encoder gradient of THIS rank's item shard over the GLOBAL batch: only dh1pre (bf16 [B,600] per rank) is exchanged
            import torch.distributed as dist
            tb = self.dp_tables[bi]
            ops.enc_coef_scatter(tb["e_row"], tb["e_item"], tb["e_slot"], tb["row_uid"], tb["row_rnorm"], tb["n_entries"], self.I,
                                 self.keep_vae, self.seed, 0, self.w_g, self.Xc_glob)
            if self.peer is not None:
                nb_ = self.dh1pre_b.numel() * 2
                ops.peer_push(self.dh1pre_b, nb_, self.peer["dh1"], self.rank * nb_, self.world_size, dst_mc=self.peer["dh1_mc"])
                self._pbar(0)
            else:
                dist.all_gather_into_tensor(self.dh1_glob, self.dh1pre_b)   # rows beyond B meet all-zero Xc rows
            if tb["n_active"] > 0:
                ops.gemm(self.Xc_glob, self.dh1_glob, tb["n_active"], H, self.world_size * self.max_B, a_mn=True, b_mn=True,
                         bn=ops.pick_bn(tb["n_active"], H), out_f32=self.G_shard)
            with self._fork(self.s2):   # self-cleaning, off the critical path: the next step scatters into an all-zero matrix
                ops.enc_coef_clear(tb["e_row"], tb["e_slot"], tb["n_entries"], self.Xc_glob)
            if self.nrows > 0:
                r0, nr = self.row0, self.nrows
                if self.peer is not None:   # Adam on the shard rows, bf16 rows stored straight into every rank's encoder shadow
                    ops.enc_adam_peer(v.W_q0[r0:r0 + nr], v.W_q0_m[r0:r0 + nr], v.W_q0_v[r0:r0 + nr], self.peer["Wq0_b"], r0 * H, nr,
                                      tb["slot_local"], self.G_shard, self.world_size, scal=self.scal, shadows_mc=self.peer["Wq0_b_mc"])
                else:
                    ops.enc_adam(v.W_q0[r0:r0 + nr], v.W_q0_m[r0:r0 + nr], v.W_q0_v[r0:r0 + nr], self.Wq0_b_shard, nr, tb["slot_local"],
                                 self.G_shard, scal=self.scal)
        elif dp_comm:
            import torch.distributed as dist
            dist.reduce_scatter_tensor(self.g_enc_shard, self.dWq0_full)
            if self.nrows > 0:
                r0, nr = self.row0, self.nrows
                ops.adam(v.W_q0[r0:r0 + nr], v.W_q0_m[r0:r0 + nr], v.W_q0_v[r0:r0 + nr], self.g_enc_shard, self.Wq0_b_shard, scal=self.scal)
        small_done = False
        if fuse_update and self.overlap and self.small_adam_early:
            # Every small gradient is final once the W_q1 weight-gradient GEMM (branch s2) and the decoder weight-gradient GEMM (branch s1:
            # its aux column is db_p1) are: the small arena's Adam runs on s2 beside the encoder sweep below instead of behind it
            self.s2.wait_stream(self.s1)
            with torch.cuda.stream(self.s2):
                ops.adam(v.small, v.small_m, v.small_v, v.small_g, v.small_b, scal=self.scal)
            small_done = True
        if fuse_update:
            ops.enc_adam(v.W_q0, v.W_q0_m, v.W_q0_v, v.W_q0_b, self.I, bt["slot_of_item"], self.G_enc, scal=self.scal,
                         rows=2 if getattr(self, "_early_done", False) else 0)
            if getattr(self, "_early_done", False):
                self._join(self.s4)
                self._early_done = False
        self._join(self.s2)
        self._join(self.s1)
        if chunked:
            self._join(self.s5)
        if fuse_update and not small_done:
            ops.adam(v.small, v.small_m, v.small_v, v.small_g, v.small_b, scal=self.scal)
        self._join(self.s6)

    def _dec_chunk_rows(self):
        """Row chunks [(r0, n_rows)] of the decoder matrix for the pipelined weight gradient + Adam (multiples of 128 rows)."""
        per = max(128, (-(-self.I // self.dec_chunks) + 127) // 128 * 128)
        return [(r0, min(per, self.I - r0)) for r0 in range(0, self.I, per)]

    def _g_update(self, data, bi):
        bt = data.batches[bi]
        v = self.vae
        if self.world_size > 1:
            r0, nr = self.row0, self.nrows
            if nr > 0:   # this rank's row shard of the two big matrices; gradients arrive reduce-scattered
                ops.adam(v.W_q0[r0:r0 + nr], v.W_q0_m[r0:r0 + nr], v.W_q0_v[r0:r0 + nr], self.g_enc_shard, self.Wq0_b_shard, scal=self.scal)
                ops.adam(v.WdT[r0:r0 + nr], v.WdT_m[r0:r0 + nr], v.WdT_v[r0:r0 + nr], self.g_dec_shard, self.WdT_b_shard, scal=self.scal)
        else:
            ops.enc_adam(v.W_q0, v.W_q0_m, v.W_q0_v, v.W_q0_b, self.I, bt["slot_of_item"], self.G_enc, scal=self.scal)
            ops.adam(v.WdT, v.WdT_m, v.WdT_v, self.dWdT, v.WdT_b, scal=self.scal)
        ops.adam(v.small, v.small_m, v.small_v, v.small_g, v.small_b, scal=self.scal)

    # ------------------------------------------------------------------------------------------------------------
    # graph capture / replay
    # ------------------------------------------------------------------------------------------------------------
    def _run(self, key, fn):
        if not self.use_graphs:
            k0 = ops.kernel_launches
            fn()
            self.kernels_launched += ops.kernel_launches - k0
            return
        g = self._graphs.get(key)
        if g is None:
            k0 = ops.kernel_launches
            fn()  # eager warm-up (also opts kernels into their shared-memory sizes outside of capture)
            self._kcount[key] = ops.kernel_launches - k0
            self.kernels_launched += self._kcount[key]
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with (torch.cuda.graph(g, stream=self._cap_stream) if self._cap_stream is not None else torch.cuda.graph(g)):
                fn()  # capture only: the eager call above already performed this step
            self._graphs[key] = g
            return
        g.replay()
        self.kernels_launched += self._kcount[key]

    def run_phase_a(self, data, bi):
        self._run(("a", id(data), bi), lambda: self.phase_a(data, bi))

    def run_d_step(self, data, bi):
        if self.world_size == 1:
            self._run(("d", id(data), bi), lambda: self.d_step(data, bi))
            return
        self._run(("ddp", id(data), bi), lambda: self._d_step_dp(data, bi))

    def _d_step_dp(self, data, bi):
        self._d_fwd_bwd(data, bi)
        self._d_update_dp()

    def _d_update_dp(self):
        import torch.distributed as dist
        d = self.disc
        # split-K partials -> the one gradient arena the exchange reads (arena_n is padded to a multiple of 4)
        ops.sum_partials(self.arena_gp, self._d_parts, d.arena_n, d.arena_g.numel(), d.arena_g)
        if self.peer is not None:
            d = self.disc
            self._pbar(0)
            ops.peer_reduce(self.peer["arena_g"], 0, d.arena_g.numel(), self.world_size, self.arena_gsum, bufs_mc=self.peer["arena_g_mc"])
            ops.adam(d.arena, d.arena_m, d.arena_v, self.arena_gsum, d.arena_b, scal=self.scal_d)
            return
        dist.all_reduce(self.disc.arena_g)                       # 161 k discriminator gradients: one small bucket
        self._d_update()

    def run_step(self, data, bi):
        """Phase A, the D update and the G update of one batch as ONE captured graph (the per-phase run_* methods are what the
        reference's epoch schedule needs -- all of phase A first, then sub-epochs of D and G; a per-batch step is what the
        benchmark times, and one graph launch instead of three removes two launch gaps)."""
        if self.world_size == 1:
            self._run(("adg", id(data), bi), lambda: self._step_fused(data, bi))
        else:
            self._run(("adgdp", id(data), bi), lambda: self._step_fused(data, bi))

    def _step_fused(self, data, bi):
        """A -> D -> G of one batch with the dependencies the data flow has, not the ones the call order suggests: the G update's VAE
        forward (train.py:326, generator side) needs the weights phase A used and nothing from the D update, so it runs on a side
        branch beside it; only y_generated (discriminator forward with the UPDATED weights) and everything behind it wait for D."""
        dp = self.world_size > 1
        if not (self.overlap and self.overlap_dg):
            self.phase_a(data, bi)
            if dp:
                self._d_step_dp(data, bi); self._g_step_dp(data, bi)
            else:
                self.d_step(data, bi); self.g_step(data, bi)
            return
        bt = data.batches[bi]
        # the three advances of the step in one launch: the counters move in the reference's order (phase A, D's Adam step, G's)
        # before any of the step's kernels start
        d = self.disc
        ops.step_advance3(self.words, self.scal_a, self.scal_d, self.scal, self.lr, bt["cnt"], self.arena_gp[0][d._off["w4"][0]:],
                          self.vae.small_g, self.w_a, self.w_d, self.w_g, anneal_cap=self.anneal_cap,
                          total_anneal_steps=self.total_anneal_steps)
        # LTG_SPLIT_D = 1 / 2 / 3: the real pairs' half of the D forward starts beside phase A (after the advance / before the decoder
        # GEMM / before the sampler) on branch s7; only the generated pairs' half waits for the sampler
        split = self.split_d if (self.split_d and not dp and self.fused_disc and not self.fused_dz12 and bt["Pr"] > 0 and bt["K"] > 0) else 0

        def real_half():
            with self._fork(self.s7):
                self._d_real_forward(data, bi)
        if split == 1:
            real_half()
        self.phase_a(data, bi, advance=False, before_decoder=real_half if split == 2 else None, before_sampler=real_half if split == 3 else None)
        self._fuse_update = not dp
        self._g_early(data, bi)
        with self._fork(self.s3):
            self._vae_forward(data, bt, True, self.keep_vae)
        self._d_fwd_bwd(data, bi, advance=False, real_done=split > 0)
        if dp:
            self._d_update_dp()    # (its gradient exchange involves the peers; the G forward on branch s3 is rank-local)
        else:
            self._d_update()
        # (the D update above gathered the embedding rows of all P pairs of THIS batch, the generated ones from row Pr on, and nothing
        # has overwritten them: the frozen embedding, F5, makes the second gather of train.py:326 a copy of the first)
        self._g_disc_forward(data, bi, reuse_gather=True)
        self._join(self.s3)
        if dp:
            self._g_rest_dp(data, bi)
        else:
            self._g_backward(data, bi)
        self._fuse_update = False

    def run_g_step(self, data, bi):
        if self.world_size == 1:
            self._run(("g", id(data), bi), lambda: self.g_step(data, bi))
            return
        # data parallel: the whole step, collectives included, is ONE captured graph (NCCL ops are capturable), so there is no
        # host round trip between the forward, the exchange step and the update
        self._run(("gdp", id(data), bi), lambda: self._g_step_dp(data, bi))

    def _g_step_dp(self, data, bi):
        """G update under user-sharded data parallelism with a row-sharded optimizer (SURVEY 8e).
        Peer-memory path (default on one NVLink node, see _setup_peer): in-place all-reduce of (sum y, cnt) in one small kernel ->
        backward; on branch s1: barrier -> ltg_adam_peer (gradient rows pulled from every rank, bf16 rows stored to every rank);
        on the main stream: push of dh1pre -> barrier -> shard gradient GEMM over the global batch -> ltg_enc_adam_peer; on branch
        s2: barrier -> pull-sum of the small gradients -> Adam on the replicated small arena; one barrier closes the step.
        NCCL path (LTG_DP_PEER=0 / no peer mapping), collectives in issue order, identical on every rank: all-reduce(sum y, cnt) ->
        reduce-scatter(dW_dec) -> all-gather(bf16 W_dec) -> all-gather(dh1pre) or reduce-scatter(dW_enc) -> all-reduce(small grads)
        -> all-gather(bf16 W_enc)."""
        self._g_forward(data, bi)
        self._g_rest_dp(data, bi)

    def _g_rest_dp(self, data, bi):
        import torch.distributed as dist
        v = self.vae
        # F3: the adversarial term multiplies GLOBAL sums; Ybar = sum y / cnt must be global before the backward pass starts
        if self.peer is not None:
            pr = self.peer
            N = self.world_size
            ops.peer_allreduce_small(pr["scal"], ops.S_SUM_Y, 2, pr["pads"], self.rank, N, 0, self.peer_epochs)
            self._dp_comm = True
            self._small_done = False
            self._g_backward(data, bi)
            self._dp_comm = False
            r0, nr = self.row0, self.nrows
            if nr > 0 and self.dp_tables is None:   # (with the activation exchange, enc_adam_peer has already stored them)
                ops.peer_push(self.Wq0_b_shard, nr * H * 2, pr["Wq0_b"], r0 * H * 2, N, dst_mc=pr["Wq0_b_mc"])
            if not self._small_done:
                self._small_exchange(0)
            self._pbar(0)   # end of step: all pushes have landed, nobody still reads this step's gradient buffers
            return
        dist.all_reduce(self.scal[ops.S_SUM_Y: ops.S_CNT + 1])
        self._dp_comm = True
        self._g_backward(data, bi)
        self._dp_comm = False
        r0, nr = self.row0, self.nrows
        dist.all_reduce(v.small_g)
        ops.adam(v.small, v.small_m, v.small_v, v.small_g, v.small_b, scal=self.scal)
        dist.all_gather_into_tensor(self.Wq0_b_full, self.Wq0_b_shard)

    def _setup_peer(self):
        """Data parallel on one NVLink node: map every exchanged buffer into all ranks (torch symmetric memory = CUDA VMM handles
        exchanged through the process group) so the exchange steps run inside our own kernels (peer_kernels.cu) instead of NCCL
        collectives. LTG_DP_PEER=0, a non-NCCL process group or a failed rendezvous keep the NCCL-collective path."""
        import os
        import torch.distributed as dist
        if os.environ.get("LTG_DP_PEER", "1") == "0" or not dist.is_initialized() or dist.get_backend() != "nccl" or self.world_size > 8:
            return
        try:
            import torch.distributed._symmetric_memory as symm
            handles = []
            mc = {}
            # NVLS multicast stores / in-switch reduction (multimem.*): measured on B200 x8 5.11 M vs 4.87 M users/s with unicast
            # peer accesses, but slower at 2 ranks (1.38 M vs 1.48 M), where a unicast access already moves every byte once
            mc_env = os.environ.get("LTG_DP_MULTICAST", "")
            use_mc = (self.world_size >= 4) if mc_env == "" else (mc_env != "0")

            def sym(like):
                t = symm.empty(*like.shape, dtype=like.dtype, device=self.device)
                t.copy_(like)
                h = symm.rendezvous(t, dist.group.WORLD)
                handles.append(h)
                mc[len(handles) - 1] = int(h.multicast_ptr) if use_mc else 0
                return t, ops.peer_table(h.buffer_ptrs)

            peer = {}
            self.dWdT_full, peer["dWdT"] = sym(self.dWdT_full); peer["dWdT_mc"] = mc[0]
            self.WdT_b_full, peer["WdT_b"] = sym(self.WdT_b_full); peer["WdT_b_mc"] = mc[1]
            self.Wq0_b_full, peer["Wq0_b"] = sym(self.Wq0_b_full); peer["Wq0_b_mc"] = mc[2]
            self.dh1_glob, peer["dh1"] = sym(self.dh1_glob); peer["dh1_mc"] = mc[3]
            self.scal_all, peer["scal"] = sym(self.scal_all)
            self.scal, self.scal_d, self.scal_a = self.scal_all[0], self.scal_all[1], self.scal_all[2]
            self.disc.arena_g, peer["arena_g"] = sym(self.disc.arena_g); peer["arena_g_mc"] = mc[5]
            self.vae.small_g, peer["small_g"] = sym(self.vae.small_g); peer["small_g_mc"] = mc[6]
            pads = torch.zeros(ops.PEER_SLOTS * 8, dtype=torch.int32, device=self.device)
            self._peer_pads, peer["pads"] = sym(pads)
            failure = None
        except Exception as e:  # noqa: BLE001  -- no peer mapping on this system: NCCL collectives do the same exchange
            failure = e
        # every rank must take the same path: the peer kernels spin on flags that only the peer path writes. A rank that failed says so
        # itself (not only rank 0), and one failure anywhere sends all ranks to the NCCL collectives.
        import sys
        all_ok = torch.tensor([0 if failure is not None else 1], dtype=torch.int32, device=self.device)
        dist.all_reduce(all_ok, op=dist.ReduceOp.MIN)
        if failure is not None:
            print("long-tail-gan_b200 [rank %d]: peer-memory exchange unavailable (%s); using NCCL collectives" % (self.rank, failure),
                  file=sys.stderr)
        if int(all_ok.item()) == 0:
            if failure is None and self.rank == 0:
                print("long-tail-gan_b200: another rank has no peer mapping; all ranks use NCCL collectives", file=sys.stderr)
            return
        I = self.I
        self.vae.WdT_b = self.WdT_b_full[:I]
        self.vae.W_q0_b = self.Wq0_b_full[:I]
        self.peer_epochs = torch.zeros(ops.PEER_SLOTS, dtype=torch.int32, device=self.device)
        self.arena_gsum = torch.zeros_like(self.disc.arena_g)
        self.small_gsum = torch.zeros_like(self.vae.small_g)
        self._peer_handles = handles
        torch.cuda.synchronize()
        dist.barrier()
        self.peer = peer

    def _small_exchange(self, slot):
        """barrier (every rank's small gradients are final) -> sum of all ranks' small gradients -> Adam on the replicated small arena"""
        v = self.vae
        self._pbar(slot)
        ops.peer_reduce(self.peer["small_g"], 0, v.small_g.numel(), self.world_size, self.small_gsum, bufs_mc=self.peer["small_g_mc"])
        ops.adam(v.small, v.small_m, v.small_v, self.small_gsum, v.small_b, scal=self.scal)

    def _pbar(self, slot=0):
        ops.peer_barrier(self.peer["pads"], self.rank, self.world_size, slot, self.peer_epochs)

    def attach_dp_tables(self, tables):
        """tables = build_dp_shard_tables(...): switches the encoder-gradient exchange from a 48 MB reduce-scatter of dW_q0 to a
        0.6 MB-per-rank all-gather of dh1pre (the dropout coefficients of the other ranks' users are recomputed locally)."""
        self.dp_tables = tables

    def gather_master(self):
        """Data parallel only: all-gather the fp32 master rows of the two sharded matrices (checkpointing / checks)."""
        if self.world_size == 1:
            return
        import torch.distributed as dist
        for t in (self.vae.W_q0, self.vae.WdT, self.vae.W_q0_m, self.vae.WdT_m, self.vae.W_q0_v, self.vae.WdT_v):
            full = torch.zeros(self.I_pad, H, dtype=torch.float32, device=self.device)
            shard = torch.zeros(self.R, H, dtype=torch.float32, device=self.device)
            shard[: self.nrows].copy_(t[self.row0: self.row0 + self.nrows])
            dist.all_gather_into_tensor(full, shard)
            t.copy_(full[: self.I])

    # ------------------------------------------------------------------------------------------------------------
    # losses of the last step (host reads; train.py:303,329 print them once per sub-epoch)
    # ------------------------------------------------------------------------------------------------------------
    def last_losses(self, B, B_global=None, reduce=False):
        """reduce (data parallel): sums the per-rank NLL / KL / sum p / d_loss over the ranks (sum y and cnt already are global) and
        normalises by the global batch -- a collective, every rank must call it."""
        sa_t = self.scal_all.detach().clone()
        if reduce and self.world_size > 1:
            import torch.distributed as dist
            loc = torch.stack([sa_t[0, ops.S_NLL_SUM], sa_t[0, ops.S_KL_SUM], sa_t[0, ops.S_SUM_P], sa_t[1, ops.S_D_LOSS]])
            dist.all_reduce(loc)
            sa_t[0, ops.S_NLL_SUM], sa_t[0, ops.S_KL_SUM], sa_t[0, ops.S_SUM_P], sa_t[1, ops.S_D_LOSS] = loc[0], loc[1], loc[2], loc[3]
            if B_global is None:
                B_global = self.B_global
        sa = sa_t.cpu().numpy().astype(np.float64)
        s = sa[0]
        Bg = B if B_global is None else B_global
        neg_ll = s[ops.S_NLL_SUM] / Bg
        kl = s[ops.S_KL_SUM] / Bg
        anneal = s[ops.S_ANNEAL]
        vae_loss = neg_ll + anneal * kl
        cnt = s[ops.S_CNT]
        gan = -(self.lam / cnt) * s[ops.S_SUM_P] * s[ops.S_SUM_Y] if cnt > 0 else 0.0
        return dict(neg_ll=neg_ll, KL=kl, anneal=anneal, vae_loss=vae_loss, gan_loss=gan, g_loss=vae_loss + gan, d_loss=sa[1][ops.S_D_LOSS],
                    cnt=cnt, sum_p=s[ops.S_SUM_P], sum_y=s[ops.S_SUM_Y])

    # ------------------------------------------------------------------------------------------------------------
    # evaluation: train.py:333-348, test.py:138-173 + eval_functions.py
    # ------------------------------------------------------------------------------------------------------------
    def _eval_batch(self, N, batch):
        """Users per evaluation launch. Default: up to 4,096, bounded by 1 GiB of fp32 scores (the reference's batch_size_vad /
        batch_size_test only bound its dense host arrays, train.py:333-337; every user is scored independently, dropout keyed by user id)."""
        cap = max(1, min(4096, (1 << 30) // (4 * self.ld)))
        if batch is None:
            nbat = max(1, -(-N // cap))
            return max(1, -(-N // nbat))          # equal batches (10,000 users -> 3 x 3,334, not 4,096 + 4,096 + 1,808)
        return max(1, min(int(batch), cap))

    def _eval_forward(self, ws, trp, tri, coef, b0, B, uid0, keep, max_nnz, words, scal):
        """One batch of the inference forward (MultiVAE.forward_pass at is_training = 0, MultiVAE.py:175-186): rng-step advance, encoder
        gather of fold-in rows [b0, b0 + B) -> middle -> fp32 decoder GEMM into ws.scores. `words` / `scal` are the step state it advances
        and reads: the engine's own for evaluate, private copies for recommend. Returns the batch's row pointers."""
        v = self.vae
        ops.step_advance(words, scal, 0, self.lr)
        ip = trp[b0: b0 + B + 1]
        ops.enc_gather_fwd(ip, tri, None, B, self.I, uid0, v.W_q0_b, v.view("b_q0"), keep, self.seed, 0, words, ws.h1, coef, max_nnz,
                           ws.enc_ws, ws.enc_cnt)
        self._middle_unfused(B, uid0, 0.0, words, scal, ws=ws)
        ops.gemm(ws.h2, v.WdT_b, B, self.I, H, bn=256, out_f32=ws.scores, bias=v.view("b_p1"))
        return ip

    def evaluate(self, tr_indptr, tr_indices, te_indptr, te_indices, k=100, recall_ks=(20, 50), batch=None, uid_start=0, keep=None):
        """Scores every eval user from its fold-in interactions, masks them, ranks, and returns the per-user lists
        (ndcg@k, recall@rk...) over users with a non-empty held-out set, exactly like eval_functions.py."""
        dev = self.device
        N = len(tr_indptr) - 1
        batch = self._eval_batch(N, batch)
        ws = self._eval_workspace(batch)
        keep = self.keep_vae if keep is None else keep
        scores = ws.scores
        tr_ptr_h = np.ascontiguousarray(tr_indptr, dtype=np.int32)
        tr_idx_h = torch.from_numpy(np.ascontiguousarray(tr_indices if len(tr_indices) else np.zeros(1), dtype=np.int32))
        max_eval_nnz = int(np.diff(tr_ptr_h.astype(np.int64)).max()) if N > 0 else 0
        # Host set-up is a third of the call at 10 k users (profiles/r2_timeline_eval.txt: 0.88 of 2.5 ms before the first kernel), so only
        # what the first batch's forward needs is uploaded before it is launched -- the row pointers and the first batch's fold-in items;
        # the rest of the fold-in items and the held-out CSR follow on a copy stream while the GPU works on batch 0.
        main = torch.cuda.current_stream()
        up = getattr(self, "_eval_up_stream", None)
        if up is None:
            up = self._eval_up_stream = torch.cuda.Stream(device=dev)
        trp = torch.as_tensor(tr_ptr_h).to(dev)
        tri = torch.empty(tr_idx_h.numel(), dtype=torch.int32, device=dev)
        coef = torch.empty(tr_idx_h.numel(), dtype=torch.float32, device=dev)   # written by the gather, not read by evaluation
        first_end = int(tr_ptr_h[min(batch, N)]) if N > 0 else 0
        if len(tr_indices) == 0:
            tri.zero_()
        elif first_end > 0:
            tri[:first_end].copy_(tr_idx_h[:first_end], non_blocking=True)
        ev_alloc = torch.cuda.Event()
        ev_alloc.record(main)             # tri exists and its first rows are on their way: the copy stream may fill in the rest
        state = {}

        def upload_rest():
            up.wait_event(ev_alloc)       # (not wait_stream: batch 0's forward is already queued on main, the copies run beside it)
            with torch.cuda.stream(up):
                if len(tr_indices) > first_end:
                    tri[first_end:].copy_(tr_idx_h[first_end:], non_blocking=True)
                state["tep"] = torch.as_tensor(np.ascontiguousarray(te_indptr, dtype=np.int32)).to(dev, non_blocking=True)
                state["tei"] = torch.as_tensor(np.ascontiguousarray(te_indices if len(te_indices) else np.zeros(1), dtype=np.int32)).to(dev, non_blocking=True)
                state["dcg"] = torch.zeros(N, dtype=torch.float64, device=dev)
                state["hits"] = torch.zeros(N, max(1, len(recall_ks)), dtype=torch.int32, device=dev)
            main.wait_stream(up)

        for b0 in range(0, N, batch):
            B = min(batch, N - b0)
            # fp32 logits: softmax is monotone per row, so ranking the logits equals ranking generator_out (SURVEY section 7)
            ip = self._eval_forward(ws, trp, tri, coef, b0, B, uid_start + b0, keep, max_eval_nnz, self.words, self.scal)
            if b0 == 0:
                upload_rest()
            ops.topk_metrics(scores, B, self.I, ip, tri, state["tep"][b0: b0 + B + 1], state["tei"], k, recall_ks, None, state["dcg"][b0:],
                             state["hits"][b0:])
        if N <= 0:
            upload_rest()
        dcg, hits = state["dcg"], state["hits"][:, :len(recall_ks)]
        torch.cuda.synchronize()
        return metrics_from_counts(dcg.cpu().numpy(), hits.cpu().numpy(), np.diff(np.asarray(te_indptr, dtype=np.int64)), k, recall_ks)

    def recommend(self, tr_indptr, tr_indices, k=100, batch=None, uid_start=0, keep=1.0, exclude_seen=True, allow=None):
        """Top-k recommendation lists for the users whose fold-in interactions are the CSR rows (tr_indptr, tr_indices). Users are scored
        exactly as `evaluate` scores them (same batches, dropout keyed by uid_start + row); keep=1.0 (default) gives deterministic lists,
        keep=None the engine's keep_vae (the reference's inference default). exclude_seen: never list a fold-in item. allow (optional): an
        iterable of item ids or a boolean mask of length I; only those items are listed. Returns NumPy arrays: items int64 [N, k] ordered
        by probability (ties: lower id first; -1 pads a row with fewer than k eligible items), probs float32 [N, k] (the generator's
        softmax over the whole catalog, MultiVAE.py:143: a filter does not renormalise them; 0 for padding), lse float32 [N] (the row's
        log-sum-exp of the logits). The engine's rng step and scalars are left as they were: the forward advances private copies."""
        dev = self.device
        N = len(tr_indptr) - 1
        batch = self._eval_batch(N, batch)
        ws = self._eval_workspace(batch)
        keep = self.keep_vae if keep is None else float(keep)
        tr_ptr_h = np.ascontiguousarray(tr_indptr, dtype=np.int32)
        tr_idx_h = np.ascontiguousarray(tr_indices if len(tr_indices) else np.zeros(1), dtype=np.int32)
        if len(tr_indices) and (tr_idx_h.min() < 0 or tr_idx_h.max() >= self.I):
            raise ValueError("fold-in item ids must lie in [0, %d)" % self.I)
        trp = torch.as_tensor(tr_ptr_h).to(dev)
        tri = torch.as_tensor(tr_idx_h).to(dev)
        coef = torch.empty(tri.numel(), dtype=torch.float32, device=dev)
        max_nnz = int(np.diff(tr_ptr_h.astype(np.int64)).max()) if N > 0 else 0
        bits = None if allow is None else torch.from_numpy(allow_bits(allow, self.I).view(np.int32)).to(dev)
        words, scal = self.words.clone(), self.scal.clone()
        items = torch.empty(N, k, dtype=torch.int32, device=dev)
        logits = torch.empty(N, k, dtype=torch.float32, device=dev)
        probs = torch.empty(N, k, dtype=torch.float32, device=dev)
        lse = torch.empty(N, dtype=torch.float32, device=dev)
        for b0 in range(0, N, batch):
            B = min(batch, N - b0)
            ip = self._eval_forward(ws, trp, tri, coef, b0, B, uid_start + b0, keep, max_nnz, words, scal)
            ops.topk_recommend(ws.scores, B, self.I, ip if exclude_seen else None, tri if exclude_seen else None, bits, k, items[b0:],
                               logits[b0:], probs[b0:], lse[b0:])
        torch.cuda.synchronize()
        return dict(items=items.cpu().numpy().astype(np.int64), probs=probs.cpu().numpy(), lse=lse.cpu().numpy())


class Session(object):
    """Stand-in for the reference's `sess.run(fetches, feed_dict)` on the generator graph (train.py:200,339; test.py:146):
    fetch the lazy handles returned by generator_VAECF -- `item_prob_dist` (softmax over the catalog, MultiVAE.py:143) and
    `neg_ELBO` -- with a dense `input_ph` feed and the reference's placeholder defaults (keep_prob 0.75, is_training 0,
    anneal 1). Compatibility path: it materialises the dense [B, I] probabilities the training path never builds."""

    def __init__(self, engine):
        self.engine = engine

    def run(self, fetches, feed_dict):
        single = not isinstance(fetches, (list, tuple))
        fl = [fetches] if single else list(fetches)
        e = self.engine
        v = e.vae
        X = np.asarray(feed_dict[v.input_ph], dtype=np.float32)
        keep = float(feed_dict.get(v.keep_prob_ph, v.keep_prob_ph.default))
        is_training = float(feed_dict.get(v.is_training_ph, v.is_training_ph.default))
        anneal = float(feed_dict.get(v.anneal_ph, v.anneal_ph.default))
        from scipy import sparse
        csr = sparse.csr_matrix(X)
        csr.sort_indices()
        n = X.shape[0]
        dev = e.device
        ip = torch.as_tensor(csr.indptr.astype(np.int32)).to(dev)
        idx = torch.as_tensor((csr.indices if csr.nnz else np.zeros(1)).astype(np.int32)).to(dev)
        val = torch.as_tensor((csr.data if csr.nnz else np.zeros(1)).astype(np.float32)).to(dev)
        coef = torch.zeros(max(1, csr.nnz), dtype=torch.float32, device=dev)
        probs = np.zeros((n, e.I), dtype=np.float32)
        nll_sum = kl_sum = 0.0
        out_dev = torch.zeros(e.max_B, e.I, dtype=torch.float32, device=dev)
        max_nnz = int(np.diff(csr.indptr).max()) if n else 0
        for b0 in range(0, n, e.max_B):
            B = min(e.max_B, n - b0)
            ops.step_advance(e.words, e.scal, 0, e.lr)
            ipb = ip[b0: b0 + B + 1]
            ops.enc_gather_fwd(ipb, idx, val, B, e.I, b0, v.W_q0_b, v.view("b_q0"), keep, e.seed, 0, e.words, e.h1, coef, max_nnz,
                               e.enc_ws, e.enc_cnt)
            e._middle_unfused(B, b0, is_training, e.words, e.scal)
            ops.dec_logits_fwd(e.h2, v.WdT_b, v.view("b_p1"), B, e.I, e.logits, e.partial)
            ops.dec_row_stats(e.partial, ops.dec_logits_nblk(B, e.I), e.logits, B, ipb, idx, val, None, None, None, e.lse, e.xw, None, e.scal)
            ops.dec_probs(e.logits, e.lse, B, e.I, out_dev)
            torch.cuda.synchronize()
            probs[b0: b0 + B] = out_dev[:B].cpu().numpy()
            sc = e.scal.cpu().numpy()
            nll_sum += float(sc[ops.S_NLL_SUM]); kl_sum += float(sc[ops.S_KL_SUM])
        res = []
        for f in fl:
            name = getattr(f, "name", None)
            if name == "item_prob_dist":
                res.append(probs)
            elif name == "neg_ELBO":
                res.append(np.float32(nll_sum / max(n, 1) + anneal * kl_sum / max(n, 1)))   # MultiVAE.py:110-119
            else:
                raise KeyError("Session.run can fetch the generator's item_prob_dist and neg_ELBO handles, got %r" % (f,))
        return res[0] if single else res


def metrics_from_counts(dcg, hits, n_held, k, recall_ks):
    """Host tail of eval_functions.py: IDCG (29-30), the IDCG!=0 / denom!=0 filters (34-36, 58-60), fp64 like NumPy."""
    tp = 1.0 / np.log2(np.arange(2, k + 2))
    csum = np.concatenate([[0.0], np.cumsum(tp)])
    idcg = csum[np.minimum(n_held, k)]
    keep = n_held > 0
    out = {"ndcg@%d" % k: (dcg[keep] / idcg[keep]).tolist()}
    for j, rk in enumerate(recall_ks):
        denom = np.minimum(rk, n_held)
        out["recall@%d" % rk] = (hits[keep, j].astype(np.float32) / denom[keep]).tolist()
    return out
