"""Catalog-sharded (vocab-parallel) GAN step and ranking evaluation: the second multi-GPU split of SURVEY 8e, the only layout in
which the 1 M-item configuration (BASELINE configs[4]) exists. One process per GPU; rank r owns the item shard
[lo_r, lo_r + I_r): rows of W_enc, columns of W_dec (stored transposed, so rows again), b_dec and their Adam state -- 99.97 % of the
parameters never cross NVLink. Every rank processes the SAME batch of users; what is exchanged per step is activations:

    encoder  (MultiVAE.py:148-155)   partial pre-activation sums [B,600] fp32           all-reduce
    middle   (MultiVAE.py:157-181)   replicated (identical inputs -> identical results on every rank)
    softmax  (MultiVAE.py:108,143)   per-row (lse_r, sum x_r, sum sampled prob_r) [B,3]   all-gather, combined as
                                     lse = LSE_r(lse_r), s_u = sum_r s_ur exp(lse_r - lse)
    sampling (sample.py:40-67)       the candidates' logits [sum C_u] fp32 (each rank fills the ones it owns)   all-reduce
    backward (train.py:164)          dh2 = dl_r W_dec_r  [B,600] fp32                     all-reduce
    discriminator (train.py:300)     pairs split over the ranks (frozen embedding table replicated, F5); 161 k gradients all-reduce
    top-k    (eval_functions.py:17-23,43-45)  local top-k per shard (ltg_topk_metrics) -> all-gather of k (score, global id)
                                     pairs per rank -> merge (score desc, id asc)

The exchanges are torch.distributed (NCCL) collectives on [B,600]-sized tensors; the kernels are the same C-ABI kernels as the
single-GPU path plus ltg_enc_gather_partial / ltg_bias_tanh / ltg_sample_pairs_vals. Results equal the single-GPU engine on the same
batch up to float summation order (tests/test_vocab_parallel_gpu.py, tools/vp_check.py)."""
import numpy as np
import torch
import torch.distributed as dist

from . import ops
from .engine import GanEngine, TrainData, _pad, allow_bits, metrics_from_counts
from .generator import H, L


def shard_bounds(n_items, world):
    """Block shards of the catalog: rank r owns [r*R, min(I, (r+1)*R)), R a multiple of 8 (TMA pitch / vector loads)."""
    R = _pad((n_items + world - 1) // world, 8)
    return [(min(n_items, r * R), min(n_items, (r + 1) * R)) for r in range(world)]


def shard_tables(tabs, lo, hi):
    """Side tables for one rank: the training CSR restricted to items [lo, hi) with shard-local ids; everything that names items
    by their global id (candidates, popular items, real pairs, validity) is kept as is. Adds row_rnorm (over the WHOLE row)."""
    indptr = np.asarray(tabs["indptr"], dtype=np.int64)
    indices = np.asarray(tabs["indices"], dtype=np.int64)
    n = len(indptr) - 1
    deg = np.diff(indptr)
    owner = np.repeat(np.arange(n, dtype=np.int64), deg)
    sel = (indices >= lo) & (indices < hi)
    loc_ptr = np.zeros(n + 1, dtype=np.int64)
    np.add.at(loc_ptr, owner[sel] + 1, 1)
    out = dict(tabs)
    out.update(n_items=int(hi - lo), indptr=np.cumsum(loc_ptr).astype(np.int32), indices=(indices[sel] - lo).astype(np.int32))
    out["row_rnorm"] = (1.0 / np.sqrt(np.maximum(deg, 1e-12))).astype(np.float32)
    out["row_nnz"] = deg.astype(np.float32)
    return out


def combine_softmax_stats(sa):
    """Per-shard softmax statistics -> global ones (MultiVAE.py:108,143 over a catalog split into shards). sa [R, B, >=3] holds, per
    shard r and user, (lse_r = log sum_{i in shard} exp(logit_i), sum_{i in shard} x_i, sum over the user's sampled items in the
    shard of exp(logit_i - lse_r)). Returns (lse [B] = log sum_r exp(lse_r), sum x [B], sum of sampled softmax probabilities [B] =
    sum_r s_r exp(lse_r - lse))."""
    lse = torch.logsumexp(sa[:, :, 0], dim=0)
    w = torch.exp(sa[:, :, 0] - lse[None])
    return lse, sa[:, :, 1].sum(0), (sa[:, :, 2] * w).sum(0)


def merge_topk(vals, gids, k, with_vals=False):
    """Per-shard top-k lists side by side (vals / gids [B, R*k]: scores and GLOBAL item ids) -> the global top-k ids [B, k] ordered by
    (score desc, id asc), the tie rule of ltg_topk_metrics (eval_functions.py:17-23 leaves ties to argpartition). Two stable sorts:
    ascending id first, then descending score. with_vals: return (ids, their scores)."""
    o1 = torch.argsort(gids, dim=1, stable=True)
    vals, gids = torch.gather(vals, 1, o1), torch.gather(gids, 1, o1)
    o2 = torch.argsort(vals, dim=1, descending=True, stable=True)
    if with_vals:
        return torch.gather(gids, 1, o2)[:, :k], torch.gather(vals, 1, o2)[:, :k]
    return torch.gather(gids, 1, o2)[:, :k]


class ShardData(TrainData):
    """TrainData over the shard-local CSR + per-batch catalog-shard structures (row norms, owned candidate positions)."""

    def __init__(self, tabs_shard, lo, hi, batch_size, device="cuda", **kw):
        t = dict(tabs_shard)
        self.row_rnorm_h = t.pop("row_rnorm"); self.row_nnz_h = t.pop("row_nnz")
        super().__init__(batch_size=batch_size, device=device, **t, **kw)
        self.lo, self.hi = int(lo), int(hi)
        dev = self.device
        cand_ptr, cand_items = self._host["cand_ptr"].astype(np.int64), self._host["cand_items"].astype(np.int64)
        self.cand_vals = torch.zeros(max(1, len(cand_items)), dtype=torch.float32, device=dev)
        for bt in self.batches:
            b0, B = bt["b0"], bt["B"]
            bt["row_rnorm"] = torch.as_tensor(self.row_rnorm_h[b0: b0 + B]).to(dev)
            bt["row_nnz"] = torch.as_tensor(self.row_nnz_h[b0: b0 + B]).to(dev)
            c0, c1 = int(cand_ptr[b0]), int(cand_ptr[b0 + B])
            it = cand_items[c0:c1]
            rows = np.repeat(np.arange(B, dtype=np.int64), np.diff(cand_ptr[b0: b0 + B + 1]))
            own = (it >= lo) & (it < hi)
            bt["cand_range"] = (c0, c1)
            bt["cand_own_pos"] = torch.as_tensor(np.nonzero(own)[0] + c0).to(dev)
            bt["cand_own_row"] = torch.as_tensor(rows[own]).to(dev)
            bt["cand_own_lid"] = torch.as_tensor(it[own] - lo).to(dev)


class CatalogShardedEngine(GanEngine):
    """GanEngine whose generator holds ONE item shard. `vae` is a MultiVAE([200, 600, I_r]) over the shard (its small arena -- W_q1, W_p0,
    b_q0, b_q1, b_p0 -- is replicated, b_p1 is the shard's); `disc` is the full discriminator (replicated)."""

    def __init__(self, vae, disc, max_B, max_P, n_items_global, item_lo, rank, world, group=None, **kw):
        kw.setdefault("use_graphs", False)
        # use_graphs=True: phase A / D / G (or the whole step) of a batch are captured as CUDA graphs with their NCCL collectives inside
        # (every rank captures and replays the same sequence); nothing in the step reads a device value back to the host
        super().__init__(vae, disc, max_B, max_P, world_size=1, rank=0, **kw)
        self.vp_rank, self.vp_world, self.group = int(rank), int(world), group
        self.I_global, self.item_lo = int(n_items_global), int(item_lo)
        dev, B = self.device, self.max_B
        f32 = dict(dtype=torch.float32, device=dev)
        self.pre_sum = torch.zeros(B, H, **f32)
        self.dh2sum = torch.zeros(B, H, **f32)
        self.stats = torch.zeros(B, 4, **f32)
        self.stats_all = torch.zeros(self.vp_world, B, 4, **f32)
        self.lse_g = torch.zeros(B, **f32); self.xw_g = torch.zeros(B, **f32); self.su_g = torch.zeros(B, **f32)
        self.overlap = False   # collectives are issued on the current stream between the kernels
        self.early_adam = False

    # ---- collectives ---------------------------------------------------------------------------------------------------
    def _allreduce(self, t):
        if self.vp_world > 1:
            dist.all_reduce(t, group=self.group)
        return t

    # ---- forward over the shard ----------------------------------------------------------------------------------------
    def _vp_forward(self, data, bt, is_training, keep):
        v = self.vae
        B = bt["B"]
        wstep = self.w_g if is_training else self.w_a
        indptr = data.indptr[bt["b0"]: bt["b0"] + B + 1]
        self.pre_sum[:B].zero_()
        ops.enc_gather_partial(indptr, data.indices, B, self.I_global, self.item_lo, bt["uid0"], v.W_q0_b, bt["row_rnorm"], keep, self.seed, 0,
                               wstep, self.pre_sum, data.coef, bt["max_nnz"], bt["slot_of_item"] if is_training else None,
                               self.Xc if is_training else None)
        self._allreduce(self.pre_sum[:B])
        ops.bias_tanh(self.pre_sum, v.view("b_q0"), B, H, self.h1)
        ops.vae_mid_fwd(self.h1, v.view("W_q1", "b"), v.view("b_q1"), v.view("W_p0", "b"), v.view("b_p0"),
                        self.eps_inject if is_training else None, B, bt["uid0"], 1.0 if is_training else 0.0, self.seed, 0, wstep,
                        self.mulv, self.z, self.zmu, self.h2, self.scal, tc=self.mid_tc)
        ops.dec_logits_fwd(self.h2, v.WdT_b, v.view("b_p1"), B, self.I, self.logits, self.partial)
        return indptr

    # ---- phase A: train.py:192-269 --------------------------------------------------------------------------------------
    def phase_a(self, data, bi):
        bt = data.batches[bi]
        B = bt["B"]
        ops.step_advance(self.words, self.scal, 0, self.lr, anneal_cap=self.anneal_cap, total_anneal_steps=self.total_anneal_steps,
                         zero=bt["cnt"], snap=self.w_a)
        self._vp_forward(data, bt, False, self.keep_vae)
        if bt["K"] > 0:
            Pr = bt["Pr"]
            c0, c1 = bt["cand_range"]
            cv = data.cand_vals[c0:c1]
            cv.zero_()
            # every rank fills the logits of the candidates it owns; the sum over the ranks is the full candidate-logit list
            data.cand_vals[bt["cand_own_pos"]] = self.logits[bt["cand_own_row"], bt["cand_own_lid"]].float()
            self._allreduce(cv)
            ops.sample_pairs(None, B, self.I_global, bt["uid0"], data.cand_ptr[bt["b0"]: bt["b0"] + B + 1], data.cand_items, bt["samp_ptr"],
                             data.pop_ptr[bt["b0"]: bt["b0"] + B + 1], data.pop_items, data.item_valid, self.seed, 0, self.w_a,
                             bt["pair_niche"][Pr:], bt["pair_pop"][Pr:], bt["label"][Pr:], bt["cnt"], bt["max_cand"], bt["samp_order"],
                             cand_vals=data.cand_vals)

    # ---- D update: the pair list is split over the ranks ----------------------------------------------------------------
    def _pair_slice(self, n):
        per = (n + self.vp_world - 1) // self.vp_world
        s0 = min(n, self.vp_rank * per)
        return s0, min(n, s0 + per)

    def d_step(self, data, bi):
        bt = data.batches[bi]
        d = self.disc
        s0, s1 = self._pair_slice(bt["P"])
        self._d_advance()

        class _View(object):
            pass
        view = _View()
        view.batches = [dict(bt, pair_pop=bt["pair_pop"][s0:], pair_niche=bt["pair_niche"][s0:], label=bt["label"][s0:], P=s1 - s0)]
        if s1 > s0:
            self._d_fwd_bwd(view, 0, advance=False)
            ops.sum_partials(self.arena_gp, self._d_parts, d.arena_n, d.arena_g.numel(), d.arena_g)
        else:
            d.arena_g.zero_()
        self._allreduce(d.arena_g)
        self._allreduce(self.scal_d[ops.S_SUM_Y: ops.S_D_LOSS + 1])
        ops.adam(d.arena, d.arena_m, d.arena_v, d.arena_g, d.arena_b, scal=self.scal_d)

    # ---- G update ---------------------------------------------------------------------------------------------------------
    def g_step(self, data, bi, update=True):
        bt = data.batches[bi]
        v = self.vae
        B, Pr, K = bt["B"], bt["Pr"], bt["K"]
        Bg = B
        self._g_advance()
        # y_generated on this rank's slice of the generated pairs; sum y / cnt are global before the backward pass (F3)
        if K > 0:
            g0, g1 = self._pair_slice(K)
            if g1 > g0:
                self._disc_forward(bt["pair_pop"][Pr + g0:], bt["pair_niche"][Pr + g0:], bt["label"][Pr + g0:], g1 - g0, False)
        self._allreduce(self.scal[ops.S_SUM_Y: ops.S_CNT + 1])
        indptr = self._vp_forward(data, bt, True, self.keep_vae)
        # sampled items that live in this shard (shard-local ids; the others are marked invalid for this rank)
        if K > 0:
            it = bt["pair_niche"][Pr:] - self.item_lo
            ok = (it >= 0) & (it < self.I) & (bt["label"][Pr:] > 0)
            samp_items = it.clamp(0, self.I - 1).to(torch.int32)
            samp_valid = torch.where(ok, torch.ones_like(it), -torch.ones_like(it)).to(torch.int32)
            samp = (bt["samp_ptr"], samp_items, samp_valid)
        else:
            samp = (None, None, None)
        # local softmax statistics -> global (lse, sum x, sum of sampled probabilities) per user
        self.scal[ops.S_SUM_P].zero_()
        ops.dec_row_stats(self.partial, ops.dec_logits_nblk(B, self.I), self.logits, B, indptr, data.indices, None, samp[0], samp[1], samp[2], self.lse, self.xw,
                          self.su if K > 0 else None, self.scal)
        st = self.stats[:B]
        st[:, 0] = self.lse[:B]; st[:, 1] = self.xw[:B]; st[:, 2] = self.su[:B] if K > 0 else 0.0
        if self.vp_world > 1:
            sa = self.stats_all[:, :B]
            if B != self.max_B:
                sa = torch.empty(self.vp_world, B, 4, dtype=torch.float32, device=self.device)
            dist.all_gather_into_tensor(sa, st.contiguous(), group=self.group)
        else:
            sa = st[None]
        lse, xw_g, su_g = combine_softmax_stats(sa)
        self.lse_g[:B] = lse
        self.xw_g[:B] = xw_g
        self.su_g[:B] = su_g
        # NLL: the local pass used the local lse; -sum_i x (logit - lse) = local + sum x_r (lse - lse_r)
        self.scal[ops.S_NLL_SUM] += (self.xw[:B] * (lse - self.lse[:B])).sum()
        self.scal[ops.S_SUM_P] = self.su_g[:B].sum()
        lam = self.lam
        ops.dec_dlogits(self.logits, self.lse_g, self.xw_g, self.su_g if K > 0 else None, B, self.I, Bg, lam if K > 0 else 0.0, self.scal, indptr,
                        data.indices, None, samp[0], samp[1], samp[2], self.dl)
        # decoder backward on the shard: local weight gradient, partial dh2 summed over the shards
        ops.gemm(self.dl, self.h2, self.I, H + 1, B, a_mn=True, b_mn=True, bn=128, out_f32=self.dWdT, ld_f32=H, aux_col=H,
                 aux_out=v.view("b_p1", "g"))
        ops.gemm(self.dl, v.WdT_b, B, H, self.I, b_mn=True, splits=self.dgrad_splits, bn=128, out_f32=self.dh2_part, ld_f32=H,
                 split_stride=self.max_B * H)
        ops.sum_partials(self.dh2_part, self.dgrad_splits, self.max_B * H, self.max_B * H, self.dh2sum)
        self._allreduce(self.dh2sum[:B])
        ops.tanh_bwd(self.dh2sum, self.h2, B, H, dx_bf16=self.dh2pre, dbias=v.view("b_p0", "g"), n_partials=1, partial_stride=0, ld_dy=H)
        ops.gemm(self.z, self.dh2pre, L, H, B, a_mn=True, b_mn=True, bn=64, out_f32=v.view("W_p0", "g"))
        ops.vae_mid_bwd(self.dh2pre, v.view("W_p0", "b"), v.view("W_q1", "b"), self.mulv, self.zmu, self.h1, B, Bg, -1.0, self.scal,
                        self.dmulv, self.dh1pre, self.dh1pre_b, v.view("b_q1", "g"), v.view("b_q0", "g"), tc=self.mid_tc)
        ops.gemm(self.h1, self.dmulv, H, 2 * L, B, a_mn=True, b_mn=True, bn=64, out_f32=v.view("W_q1", "g"))
        if bt["n_active"] > 0:
            ops.gemm(self.Xc, self.dh1pre_b, bt["n_active"], H, B, a_mn=True, b_mn=True, bn=ops.pick_bn(bt["n_active"], H), out_f32=self.G_enc)
        ops.enc_xc_clear(indptr, data.indices, B, bt["nnz"], bt["slot_of_item"], self.Xc)
        if not update:
            return
        # replicated small parameters: their gradients are computed from all-reduced activations on every rank; averaging them keeps
        # the replicas bit-identical although the bias gradients are accumulated with float atomics (order differs between ranks)
        off_bp1 = v._small_off["b_p1"][0]
        if self.vp_world > 1:
            dist.all_reduce(v.small_g[:off_bp1], group=self.group)
            v.small_g[:off_bp1].mul_(1.0 / self.vp_world)
        ops.adam(v.WdT, v.WdT_m, v.WdT_v, self.dWdT, v.WdT_b, scal=self.scal)
        ops.enc_adam(v.W_q0, v.W_q0_m, v.W_q0_v, v.W_q0_b, self.I, bt["slot_of_item"], self.G_enc, scal=self.scal)
        ops.adam(v.small, v.small_m, v.small_v, v.small_g, v.small_b, scal=self.scal)

    def run_phase_a(self, data, bi):
        self._run(("vpa", id(data), bi), lambda: self.phase_a(data, bi))

    def run_d_step(self, data, bi):
        self._run(("vpd", id(data), bi), lambda: self.d_step(data, bi))

    def run_g_step(self, data, bi):
        self._run(("vpg", id(data), bi), lambda: self.g_step(data, bi))

    def _step(self, data, bi):
        self.phase_a(data, bi); self.d_step(data, bi); self.g_step(data, bi)

    def run_step(self, data, bi):
        self._run(("vpadg", id(data), bi), lambda: self._step(data, bi))

    def last_losses(self, B, B_global=None, reduce=False):
        """NLL is a sum over the shards (all-reduced here: a collective); KL, sum p, sum y, cnt, d_loss are already global/replicated."""
        sa = self.scal_all.detach().clone()
        nll = sa[0, ops.S_NLL_SUM: ops.S_NLL_SUM + 1].clone()
        self._allreduce(nll)
        s = sa.cpu().numpy().astype(np.float64)
        neg_ll = float(nll.item()) / B
        kl = s[0][ops.S_KL_SUM] / B
        anneal = s[0][ops.S_ANNEAL]
        cnt = s[0][ops.S_CNT]
        gan = -(self.lam / cnt) * s[0][ops.S_SUM_P] * s[0][ops.S_SUM_Y] if cnt > 0 else 0.0
        vae_loss = neg_ll + anneal * kl
        return dict(neg_ll=neg_ll, KL=kl, anneal=anneal, vae_loss=vae_loss, gan_loss=gan, g_loss=vae_loss + gan, d_loss=s[1][ops.S_D_LOSS], cnt=cnt,
                    sum_p=s[0][ops.S_SUM_P], sum_y=s[0][ops.S_SUM_Y])

    # ---- evaluation: train.py:333-348, test.py:138-173 -------------------------------------------------------------------
    def _shard_fold_in(self, tr_indptr, tr_indices):
        """GLOBAL fold-in CSR -> this shard's part on the device: (row pointers, shard-local item ids, 1/|x_u| over the whole row,
        coefficient buffer, longest shard row)."""
        dev, lo, I_r = self.device, self.item_lo, self.I
        tr_indptr = np.asarray(tr_indptr, dtype=np.int64); tr_indices = np.asarray(tr_indices, dtype=np.int64)
        N = len(tr_indptr) - 1
        deg = np.diff(tr_indptr)
        owner = np.repeat(np.arange(N, dtype=np.int64), deg)
        sel = (tr_indices >= lo) & (tr_indices < lo + I_r)
        lp = np.zeros(N + 1, dtype=np.int64); np.add.at(lp, owner[sel] + 1, 1); lp = np.cumsum(lp)
        t32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.int32)).to(dev)  # noqa: E731
        trp, tri = t32(lp), t32(tr_indices[sel] - lo if sel.any() else np.zeros(1))
        rnorm = torch.as_tensor((1.0 / np.sqrt(np.maximum(deg, 1e-12))).astype(np.float32)).to(dev)
        coef = torch.zeros(max(1, int(sel.sum())), dtype=torch.float32, device=dev)
        max_nnz = int(np.diff(lp).max()) if N > 0 else 0
        return trp, tri, rnorm, coef, max_nnz

    def _vp_eval_forward(self, fold, b0, B, uid0, keep, words, scal, scores):
        """One batch of the inference forward over the shard (is_training = 0) into scores[:B, :I_r]: rng-step advance (snapshot in
        words[4], the phase-A word), partial encoder gather + all-reduce, middle, fp32 decoder GEMM. `words` / `scal`: the engine's own
        for evaluate, private copies for recommend. Returns the batch's shard-local row pointers."""
        v = self.vae
        trp, tri, rnorm, coef, max_nnz = fold
        w_a = words[4:5]
        ops.step_advance(words, scal, 0, self.lr, snap=w_a)
        ip = trp[b0: b0 + B + 1]
        self.pre_sum[:B].zero_()
        ops.enc_gather_partial(ip, tri, B, self.I_global, self.item_lo, uid0, v.W_q0_b, rnorm[b0: b0 + B], keep, self.seed, 0, w_a,
                               self.pre_sum, coef, max_nnz)
        self._allreduce(self.pre_sum[:B])
        ops.bias_tanh(self.pre_sum, v.view("b_q0"), B, H, self.h1)
        ops.gemm(self.h1, v.view("W_q1", "b"), B, 2 * L, H, b_mn=True, bn=64, out_f32=self.mulv, bias=v.view("b_q1"))
        ops.latent_fwd(self.mulv, None, B, uid0, 0.0, self.seed, 0, w_a, self.z, self.zmu, scal)
        ops.gemm(self.z, v.view("W_p0", "b"), B, H, L, b_mn=True, bn=64, out_bf16=self.h2, bias=v.view("b_p0"), act=1)
        ops.gemm(self.h2, v.WdT_b, B, self.I, H, bn=256, out_f32=scores, bias=v.view("b_p1"))
        return ip

    def _all_gather_cols(self, t):
        """[B, n] on every rank -> [B, R*n], rank r's block at columns [r*n, (r+1)*n)."""
        if self.vp_world == 1:
            return t
        parts = [torch.empty_like(t) for _ in range(self.vp_world)]
        dist.all_gather(parts, t.contiguous(), group=self.group)
        return torch.cat(parts, 1)

    def evaluate(self, tr_indptr, tr_indices, te_indptr, te_indices, k=100, recall_ks=(20, 50), batch=None, uid_start=0, keep=None):
        """tr_/te_ are the GLOBAL fold-in / held-out CSRs (global item ids). Every rank scores its shard, takes the exact local top-k
        (ltg_topk_metrics, seen items masked), the k (score, global id) pairs per rank are all-gathered and merged by
        (score desc, id asc); the metrics follow eval_functions.py:25-36,47-60 on the merged list. Returns the same dict as
        GanEngine.evaluate on every rank."""
        dev = self.device
        lo, I_r = self.item_lo, self.I
        te_indptr = np.asarray(te_indptr, dtype=np.int64); te_indices = np.asarray(te_indices, dtype=np.int64)
        N = len(tr_indptr) - 1
        batch = self.max_B if batch is None else min(batch, self.max_B)
        keep = self.keep_vae if keep is None else keep
        fold = self._shard_fold_in(tr_indptr, tr_indices)
        tri = fold[1]
        scores = torch.zeros(batch, self.ld, dtype=torch.float32, device=dev)
        kk = min(k, I_r)
        idx_loc = torch.zeros(batch, kk, dtype=torch.int32, device=dev)
        dcg_dummy = torch.zeros(batch, dtype=torch.float64, device=dev)
        hits_dummy = torch.zeros(batch, max(1, len(recall_ks)), dtype=torch.int32, device=dev)
        zero_ptr = torch.zeros(batch + 1, dtype=torch.int32, device=dev); one_item = torch.zeros(1, dtype=torch.int32, device=dev)
        top_all = np.zeros((N, k), dtype=np.int64)
        for b0 in range(0, N, batch):
            B = min(batch, N - b0)
            ip = self._vp_eval_forward(fold, b0, B, uid_start + b0, keep, self.words, self.scal, scores)
            ops.topk_metrics(scores, B, I_r, ip, tri, zero_ptr[: B + 1], one_item, kk, recall_ks, idx_loc, dcg_dummy, hits_dummy)
            val_loc = torch.gather(scores[:B, :I_r], 1, idx_loc[:B].long())
            gid_loc = idx_loc[:B].long() + lo
            vals, gids = self._all_gather_cols(val_loc), self._all_gather_cols(gid_loc)
            top_all[b0: b0 + B] = merge_topk(vals, gids, k).cpu().numpy()
        # metrics on the merged lists (eval_functions.py:25-30, 47-52), fp64 like NumPy
        n_held = np.diff(te_indptr)
        tp = 1.0 / np.log2(np.arange(2, k + 2))
        dcg = np.zeros(N, dtype=np.float64)
        hits = np.zeros((N, len(recall_ks)), dtype=np.int32)
        for u in range(N):
            held = te_indices[te_indptr[u]: te_indptr[u + 1]]
            if len(held) == 0:
                continue
            m = np.isin(top_all[u], held)
            dcg[u] = (m * tp).sum()
            for j, rk in enumerate(recall_ks):
                hits[u, j] = int(m[:rk].sum())
        out = metrics_from_counts(dcg, hits, n_held, k, recall_ks)
        out["topk"] = top_all
        return out

    def recommend(self, tr_indptr, tr_indices, k=100, batch=None, uid_start=0, keep=1.0, exclude_seen=True, allow=None):
        """GanEngine.recommend over the sharded catalog, with the same GLOBAL item ids in and out; returns the same dict on every rank.
        Every rank lists its shard's top k eligible items (ltg_topk_recommend: logits and the shard's log-sum-exp, no probabilities), the
        (logit, global id) lists and the per-shard lse are all-gathered, the lists merged by (logit desc, id asc) and the probabilities
        formed as exp(logit - lse) with lse = logsumexp over the shards. The engine's rng step, its phase-A snapshot and its scalars are
        left as they were: the forward advances private copies."""
        dev = self.device
        lo, I_r = self.item_lo, self.I
        N = len(tr_indptr) - 1
        batch = self.max_B if batch is None else min(batch, self.max_B)
        keep = self.keep_vae if keep is None else float(keep)
        if len(tr_indices) and (np.min(tr_indices) < 0 or np.max(tr_indices) >= self.I_global):
            raise ValueError("fold-in item ids must lie in [0, %d)" % self.I_global)
        fold = self._shard_fold_in(tr_indptr, tr_indices)
        tri = fold[1]
        bits = None if allow is None else torch.from_numpy(allow_bits(allow, self.I_global, lo, lo + I_r).view(np.int32)).to(dev)
        words, scal = self.words.clone(), self.scal.clone()
        scores = torch.zeros(batch, self.ld, dtype=torch.float32, device=dev)
        idx_loc = torch.empty(batch, k, dtype=torch.int32, device=dev)
        val_loc = torch.empty(batch, k, dtype=torch.float32, device=dev)
        lse_loc = torch.empty(batch, dtype=torch.float32, device=dev)
        items = np.empty((N, k), dtype=np.int64)
        probs = np.empty((N, k), dtype=np.float32)
        lse = np.empty(N, dtype=np.float32)
        for b0 in range(0, N, batch):
            B = min(batch, N - b0)
            ip = self._vp_eval_forward(fold, b0, B, uid_start + b0, keep, words, scal, scores)
            ops.topk_recommend(scores, B, I_r, ip if exclude_seen else None, tri if exclude_seen else None, bits, k, idx_loc, val_loc, None,
                               lse_loc)
            il = idx_loc[:B].long()
            gid_loc = torch.where(il >= 0, il + lo, self.I_global)   # padding sorts behind every real item of equal logit
            vals, gids = self._all_gather_cols(val_loc[:B]), self._all_gather_cols(gid_loc)
            lse_b = torch.logsumexp(self._all_gather_cols(lse_loc[:B, None]), dim=1)
            top, top_val = merge_topk(vals, gids, k, with_vals=True)
            pad = top >= self.I_global
            items[b0: b0 + B] = torch.where(pad, -1, top).cpu().numpy()
            probs[b0: b0 + B] = torch.where(pad, 0.0, torch.exp(top_val - lse_b[:, None])).cpu().numpy()
            lse[b0: b0 + B] = lse_b.cpu().numpy()
        return dict(items=items, probs=probs, lse=lse)


def build_shard(tabs, n_items, rank, world, batch_size, vae_params=None, disc=None, seed=98765, device="cuda", first_batch=0, max_batches=None):
    """Per-rank data + generator shard. vae_params (optional, GLOBAL [W_q0, W_q1, W_p0, W_p1, b_q0, b_q1, b_p0, b_p1]) is sliced to
    the shard (parity tests); otherwise the shard is initialised directly (Xavier limits of the global fan-in/out)."""
    from .generator import MultiVAE
    lo, hi = shard_bounds(n_items, world)[rank]
    data = ShardData(shard_tables(tabs, lo, hi), lo, hi, batch_size, device=device, first_batch=first_batch, max_batches=max_batches)
    vae = MultiVAE([L, H, hi - lo], lam=0.0, random_seed=seed)
    if vae_params is not None:
        p = [torch.as_tensor(x, dtype=torch.float32) for x in vae_params]
        vae.set_params([p[0][lo:hi], p[1], p[2], p[3][:, lo:hi], p[4], p[5], p[6], p[7][lo:hi]])
        vae.reset_optimizer()
    else:
        g = torch.Generator(device="cpu").manual_seed(int(seed))
        lim_e = float(np.sqrt(6.0 / (n_items + H)))
        small = [(torch.rand(H, 2 * L, generator=g) * 2 - 1) * float(np.sqrt(6.0 / (H + 2 * L))), (torch.rand(L, H, generator=g) * 2 - 1) * float(np.sqrt(6.0 / (L + H))),
                 torch.randn(H, generator=g) * 0.001, torch.randn(2 * L, generator=g) * 0.001, torch.randn(H, generator=g) * 0.001]
        gs = torch.Generator(device="cpu").manual_seed(int(seed) + 1 + rank)   # the shard's own rows
        vae.set_params([(torch.rand(hi - lo, H, generator=gs) * 2 - 1) * lim_e, small[0], small[1], (torch.rand(H, hi - lo, generator=gs) * 2 - 1) * lim_e,
                        small[2], small[3], small[4], torch.randn(hi - lo, generator=gs) * 0.001])
        vae.reset_optimizer()
    return data, vae, lo, hi
