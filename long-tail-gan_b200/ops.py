"""Thin Python wrappers over the C ABI (include/ltgan.h). Tensors are torch CUDA tensors used as plain device
buffers; every wrapper passes raw pointers + sizes and the current CUDA stream, and raises on a non-zero status.
There is no CPU implementation behind these functions."""
import torch

from . import _lib
from ._lib import check, ptr

H = 600
L = 200

S_KL_SUM, S_NLL_SUM, S_SUM_P, S_SUM_Y, S_CNT, S_D_LOSS = 0, 1, 2, 3, 4, 5
S_LR_T, S_ANNEAL, NSCAL = 8, 9, 16

STREAM_ENC_DROPOUT = 1
STREAM_EPS = 2
STREAM_DISC_DROPOUT = 3
STREAM_SAMPLE = 8
STREAM_PARTNER = 9

_initialised = False
# number of CUDA kernels launched through this module (graph capture counts the captured launches once)
kernel_launches = 0


def _count(n=1):
    global kernel_launches
    kernel_launches += n


def lib():
    return _lib.load()


def init():
    """Loads the library and initialises it for the current device. Raises without a B200."""
    global _initialised
    if not _initialised:
        if not torch.cuda.is_available():
            raise RuntimeError("long-tail-gan_b200 needs a CUDA (sm_100a) device; there is no CPU fallback")
        check(lib().ltg_init())
        _initialised = True


def _stream():
    return torch.cuda.current_stream().cuda_stream


def step_advance(words, scal, kind, lr, beta1=0.9, beta2=0.999, anneal_cap=0.2, total_anneal_steps=20000.0, zero=None, snap=None):
    _count(1)
    zw = 0
    if zero is not None:
        assert zero.is_contiguous() and zero.element_size() == 4
        zw = zero.numel()
    check(lib().ltg_step_advance(ptr(words), ptr(scal), kind, lr, beta1, beta2, anneal_cap, total_anneal_steps, ptr(zero), zw, ptr(snap), _stream()))


def step_advance3(words, scal_a, scal_d, scal_g, lr, zero_a, zero_d, zero_g, snap_a, snap_d, snap_g, beta1=0.9, beta2=0.999, anneal_cap=0.2,
                  total_anneal_steps=20000.0):
    """Phase A, D-update and G-update advances of one step in one launch (same state as three step_advance calls, kinds 0, 1, 2)."""
    _count(1)
    for z in (zero_a, zero_d, zero_g):
        assert z is None or (z.is_contiguous() and z.element_size() == 4)
    nw = lambda z: 0 if z is None else z.numel()  # noqa: E731
    check(lib().ltg_step_advance3(ptr(words), ptr(scal_a), ptr(scal_d), ptr(scal_g), lr, beta1, beta2, anneal_cap, total_anneal_steps,
                                  ptr(zero_a), nw(zero_a), ptr(zero_d), nw(zero_d), ptr(zero_g), nw(zero_g), ptr(snap_a), ptr(snap_d),
                                  ptr(snap_g), _stream()))


def pick_bn(M, N, splits_ok=False):
    """Tile width for the tcgen05 GEMM. Large-M problems take the widest tile that wastes the fewest padded columns (fewer
    tiles, A streamed once per n-block); problems with only a handful of 128-row blocks take 64-wide tiles so that the tile
    count, not the tile efficiency, fills the SMs -- unless split-K provides the parallelism (splits_ok)."""
    m_blocks = (M + 127) // 128
    if m_blocks < 37 and not splits_ok:
        return 64
    if N <= 64:
        return 64
    if N <= 128:
        return 128
    if N <= 192:
        return 192
    if N <= 256:
        return 256
    best = None
    for bn in (256, 192, 128):
        padded = (N + bn - 1) // bn * bn
        if best is None or padded < best[0]:
            best = (padded, bn)
    return best[1]


def pick_splits(M, N, K, bn, n_sm=132):
    """Split-K factor that brings the tile count of a skinny (small M*N, long K) GEMM up to about one wave of CTAs
    (132 rather than 148: 4-CTA clusters cannot use the SMs of GPCs whose SM count is not a multiple of 4)."""
    tiles = ((M + 127) // 128) * ((N + bn - 1) // bn)
    kb = (K + 63) // 64
    # at most 32 splits: every split adds one fp32 atomic per output element, all landing on the same addresses
    return max(1, min(kb, n_sm // max(1, tiles), 32))


def actual_splits(K, splits):
    """Number of split-K partials launch_gemm writes: exactly the requested count (trailing splits that receive no k-block
    store zeros), so consumers can sum a fixed number of partial buffers."""
    return max(1, splits)


def gemm(A, B, M, N, K, *, a_mn=False, b_mn=False, lda=None, ldb=None, splits=1, bn=128, out_f32=None, out_bf16=None, bias=None,
         act=0, alpha=1.0, atomic=False, keep=1.0, seed=0, rng_stream=0, rng_step=0, rng_step_dev=None, rng_ld=0, aux_col=-1,
         aux_out=None, ld_f32=None, ld_bf16=None, dact_src=None, dact_keep=1.0, split_stride=0):
    """D[M,N] = alpha*A*B^T on the tcgen05 GEMM. A is [M,K] (or stored [K,M] when a_mn), B is [N,K] (or [K,N] when b_mn)."""
    _count(1)
    lda = A.stride(0) if lda is None else lda
    ldb = B.stride(0) if ldb is None else ldb
    if out_f32 is not None and ld_f32 is None:
        ld_f32 = out_f32.stride(0)
    if out_bf16 is not None and ld_bf16 is None:
        ld_bf16 = out_bf16.stride(0)
    check(lib().ltg_gemm_bf16(ptr(A), lda, int(a_mn), ptr(B), ldb, int(b_mn), M, N, K, splits, bn, ptr(out_f32), ld_f32 or 0,
                              ptr(out_bf16), ld_bf16 or 0, ptr(bias), act, alpha, int(atomic), keep, seed, rng_stream, rng_step,
                              ptr(rng_step_dev), rng_ld, aux_col, ptr(aux_out), ptr(dact_src),
                              dact_src.stride(0) if dact_src is not None else 0, dact_keep, split_stride, _stream()))


def enc_gather_fwd(indptr, indices, values, B, n_items, uid0, W_enc_bf16, b_q0, keep, seed, step, step_dev, h1, coef, max_row_nnz=0,
                   pre_ws=None, counters=None, slot_of_item=None, xc=None, work=None):
    _count(1)
    check(lib().ltg_enc_gather_fwd(ptr(indptr), ptr(indices), ptr(values), B, n_items, uid0, ptr(W_enc_bf16), ptr(b_q0), keep, seed,
                                   step, ptr(step_dev), ptr(h1), h1.stride(0), ptr(coef), max_row_nnz, ptr(pre_ws), ptr(counters),
                                   ptr(slot_of_item), ptr(xc), xc.stride(0) if xc is not None else 0, ptr(work),
                                   work.numel() if work is not None else 0, _stream()))


ENC_CHUNK = 128   # nonzeros per CTA of ltg_enc_gather_fwd (csrc/vae_kernels.cu)


def enc_work_list(indptr):
    """Host-side work list of ltg_enc_gather_fwd for the CSR rows indptr[0..B]: one int32 (chunk << 20 | row) per non-empty
    128-nonzero chunk (rows without interactions keep their chunk 0: they still need bias + tanh), full chunks first."""
    import numpy as np
    deg = np.diff(np.asarray(indptr, dtype=np.int64))
    B = len(deg)
    assert B < (1 << 20)
    nch = np.maximum(1, -(-deg // ENC_CHUNK))
    rows = np.repeat(np.arange(B, dtype=np.int64), nch)
    first = np.concatenate([[0], np.cumsum(nch)[:-1]])
    chunk = np.arange(len(rows), dtype=np.int64) - np.repeat(first, nch)
    size = np.minimum(ENC_CHUNK, deg[rows] - chunk * ENC_CHUNK)
    order = np.argsort(-size, kind="stable")
    return ((chunk[order] << 20) | rows[order]).astype(np.int32)


def enc_gather_partial(indptr, indices, B, n_items_global, item_offset, uid0, W_shard_bf16, row_rnorm, keep, seed, step, step_dev, pre_sum, coef,
                       max_row_nnz=0, slot_of_item=None, xc=None):
    _count(1)
    check(lib().ltg_enc_gather_partial(ptr(indptr), ptr(indices), B, n_items_global, item_offset, uid0, ptr(W_shard_bf16), ptr(row_rnorm), keep,
                                       seed, step, ptr(step_dev), ptr(pre_sum), ptr(coef), max_row_nnz, ptr(slot_of_item), ptr(xc),
                                       xc.stride(0) if xc is not None else 0, _stream()))


def bias_tanh(pre, bias, B, N, out):
    _count(1)
    check(lib().ltg_bias_tanh(ptr(pre), pre.stride(0), ptr(bias), B, N, ptr(out), out.stride(0), _stream()))


def enc_coef_scatter(e_row, e_item, e_slot, row_uid, row_rnorm, n_entries, n_items, keep, seed, step, step_dev, xc):
    _count(1)
    check(lib().ltg_enc_coef_scatter(ptr(e_row), ptr(e_item), ptr(e_slot), ptr(row_uid), ptr(row_rnorm), n_entries, n_items, keep, seed,
                                     step, ptr(step_dev), ptr(xc), xc.stride(0), _stream()))


def latent_fwd(mulv, eps, B, uid0, is_training, seed, step, step_dev, z, zmu, scal):
    _count(1)
    check(lib().ltg_latent_fwd(ptr(mulv), ptr(eps), B, uid0, float(is_training), seed, step, ptr(step_dev), ptr(z), z.stride(0),
                               ptr(zmu), ptr(scal), _stream()))


def latent_bwd(dz, mulv, zmu, B, B_global, anneal, scal, dmulv, db_q1):
    _count(1)
    check(lib().ltg_latent_bwd(ptr(dz), ptr(mulv), ptr(zmu), B, B_global, anneal, ptr(scal), ptr(dmulv), dmulv.stride(0), ptr(db_q1),
                               _stream()))


def vae_mid_fwd(h1, Wq1_b, b_q1, Wp0_b, b_p0, eps, B, uid0, is_training, seed, step, step_dev, mulv, z, zmu, h2, scal, tc=False):
    """tc: the tcgen05 kernel (mid_tc.cu, one launch) instead of the two mma.sync kernels (mid_kernels.cu)."""
    _count(1 if tc else 2)
    fn = lib().ltg_vae_mid_fwd_tc if tc else lib().ltg_vae_mid_fwd
    check(fn(ptr(h1), h1.stride(0), ptr(Wq1_b), ptr(b_q1), ptr(Wp0_b), ptr(b_p0), ptr(eps), B, uid0, float(is_training),
                                seed, step, ptr(step_dev), ptr(mulv), ptr(z), z.stride(0), ptr(zmu), ptr(h2), h2.stride(0), ptr(scal),
                                _stream()))


def vae_mid_bwd(dh2pre, Wp0_b, Wq1_b, mulv, zmu, h1, B, B_global, anneal, scal, dmulv, dh1pre, dh1pre_b, db_q1, db_q0, tc=False):
    _count(1 if tc else 2)
    fn = lib().ltg_vae_mid_bwd_tc if tc else lib().ltg_vae_mid_bwd
    check(fn(ptr(dh2pre), ptr(Wp0_b), ptr(Wq1_b), ptr(mulv), ptr(zmu), ptr(h1), h1.stride(0), B, B_global, anneal,
                                ptr(scal), ptr(dmulv), ptr(dh1pre), ptr(dh1pre_b), ptr(db_q1), ptr(db_q0), _stream()))


def tanh_bwd(dy, y_bf16, B, N, dx_bf16=None, dx_f32=None, dbias=None, n_partials=1, partial_stride=0, ld_dy=None):
    _count(1)
    check(lib().ltg_tanh_bwd(ptr(dy), dy.stride(0) if ld_dy is None else ld_dy, n_partials, partial_stride, ptr(y_bf16), y_bf16.stride(0), B, N,
                             ptr(dx_bf16),
                             dx_bf16.stride(0) if dx_bf16 is not None else 0, ptr(dx_f32),
                             dx_f32.stride(0) if dx_f32 is not None else 0, ptr(dbias), _stream()))


def dec_logits_nblk(B, n_items):
    """Rows of the (max, sumexp) partial buffer ltg_dec_logits_fwd writes for this shape (what the row passes must be told)."""
    return int(lib().ltg_dec_logits_nblk(int(B), int(n_items)))


def dec_logits_nblk_max(n_items):
    return 4 * ((int(n_items) + 127) // 128)


def dec_logits_fwd(h2, WdT_bf16, b_dec, B, n_items, logits, partial):
    _count(1)
    check(lib().ltg_dec_logits_fwd(ptr(h2), h2.stride(0), ptr(WdT_bf16), ptr(b_dec), B, n_items, ptr(logits),
                                   logits.stride(0) if logits is not None else 0, ptr(partial), _stream()))


def dec_row_stats(partial, n_blocks, logits, B, indptr, indices, values, samp_ptr, samp_items, samp_valid, lse, xw, s_u, scal):
    _count(1)
    check(lib().ltg_dec_row_stats(ptr(partial), n_blocks, ptr(logits), logits.stride(0) if logits is not None else 0, B, ptr(indptr),
                                  ptr(indices), ptr(values), ptr(samp_ptr), ptr(samp_items), ptr(samp_valid), ptr(lse), ptr(xw),
                                  ptr(s_u), ptr(scal), _stream()))


def dec_probs(logits, lse, B, n_items, out):
    _count(1)
    check(lib().ltg_dec_probs(ptr(logits), logits.stride(0), ptr(lse), B, n_items, ptr(out), out.stride(0), _stream()))


def dec_dlogits(logits, lse, xw, s_u, B, n_items, B_global, lam, scal, indptr, indices, values, samp_ptr, samp_items, samp_valid, dl):
    _count(2)
    check(lib().ltg_dec_dlogits(ptr(logits), logits.stride(0), ptr(lse), ptr(xw), ptr(s_u), B, n_items, B_global, lam, ptr(scal),
                                ptr(indptr), ptr(indices), ptr(values), ptr(samp_ptr), ptr(samp_items), ptr(samp_valid), ptr(dl),
                                _stream()))


def dec_row_bwd(partial, n_blocks, logits, B, n_items, B_global, lam, indptr, indices, values, samp_ptr, samp_items, samp_valid, lse, scal, dl):
    _count(1)
    check(lib().ltg_dec_row_bwd(ptr(partial), n_blocks, ptr(logits), logits.stride(0), B, n_items, B_global, lam, ptr(indptr), ptr(indices),
                                ptr(values), ptr(samp_ptr), ptr(samp_items), ptr(samp_valid), ptr(lse), ptr(scal), ptr(dl), _stream()))


def adam(p, m, v, g, shadow, lr_t=-1.0, scal=None, beta1=0.9, beta2=0.999, eps=1e-8, n_partials=1, partial_stride=0):
    _count(1)
    check(lib().ltg_adam(ptr(p), ptr(m), ptr(v), ptr(g), n_partials, partial_stride, ptr(shadow), p.numel(), lr_t, ptr(scal), beta1, beta2,
                         eps, _stream()))


# ---- data-parallel exchange over peer memory (peer_kernels.cu). A "table" is a ctypes array of one device pointer per rank.
PEER_SLOTS = 4   # LTG_PEER_SLOTS


def peer_table(ptrs):
    import ctypes
    return (ctypes.c_void_p * len(ptrs))(*[int(p) for p in ptrs])


def peer_barrier(pads, rank, world, slot, epochs):
    _count(1)
    check(lib().ltg_peer_barrier(pads, rank, world, slot, ptr(epochs), _stream()))


def peer_allreduce_small(bufs, offset, count, pads, rank, world, slot, epochs):
    _count(1)
    check(lib().ltg_peer_allreduce_small(bufs, offset, count, pads, rank, world, slot, ptr(epochs), _stream()))


def peer_reduce(bufs, offset, n, world, out, bufs_mc=None):
    _count(1)
    check(lib().ltg_peer_reduce(bufs, bufs_mc or None, offset, n, world, ptr(out), _stream()))


def peer_push(src, nbytes, dst, dst_offset_bytes, world, dst_mc=None):
    _count(1)
    check(lib().ltg_peer_push(ptr(src), nbytes, dst, dst_mc or None, dst_offset_bytes, world, _stream()))


def adam_peer(p, m, v, grads, shadows, offset, world, lr_t=-1.0, scal=None, beta1=0.9, beta2=0.999, eps=1e-8, grads_mc=None, shadows_mc=None):
    _count(1)
    check(lib().ltg_adam_peer(ptr(p), ptr(m), ptr(v), grads, grads_mc or None, shadows, shadows_mc or None, offset, p.numel(), world, lr_t,
                              ptr(scal), beta1, beta2, eps, _stream()))


def wgrad_adam(A, B, M, N, K, p, m, v, shadow, n_cols, aux_col=-1, aux_out=None, lr_t=-1.0, scal=None, beta1=0.9, beta2=0.999, eps=1e-8):
    """dW = A^T B (A stored [K, M], B stored [K, N]) with TF-Adam on p/m/v [M, ld] + bf16 shadow as the GEMM epilogue."""
    _count(1)
    check(lib().ltg_wgrad_adam(ptr(A), A.stride(0), ptr(B), B.stride(0), M, N, K, ptr(p), ptr(m), ptr(v), ptr(shadow), p.stride(0), n_cols,
                               aux_col, ptr(aux_out), lr_t, ptr(scal), beta1, beta2, eps, _stream()))


def enc_adam_peer(p, m, v, shadows, offset, n_items, slot_of_item, G, world, lr_t=-1.0, scal=None, beta1=0.9, beta2=0.999, eps=1e-8,
                  shadows_mc=None):
    _count(1)
    check(lib().ltg_enc_adam_peer(ptr(p), ptr(m), ptr(v), shadows, shadows_mc or None, offset, n_items, ptr(slot_of_item), ptr(G), world, lr_t,
                                  ptr(scal), beta1, beta2, eps, _stream()))


def enc_wgrad_compact(G, n_active, act_ptr, csc_row, csc_pos, coef, dh1pre):
    _count(1)
    check(lib().ltg_enc_wgrad_compact(ptr(G), n_active, ptr(act_ptr), ptr(csc_row), ptr(csc_pos), ptr(coef), ptr(dh1pre),
                                      dh1pre.stride(0), _stream()))


def enc_adam(p, m, v, shadow, n_items, slot_of_item, G, lr_t=-1.0, scal=None, beta1=0.9, beta2=0.999, eps=1e-8, rows=0):
    _count(1)
    check(lib().ltg_enc_adam(ptr(p), ptr(m), ptr(v), ptr(shadow), n_items, ptr(slot_of_item), ptr(G), lr_t, ptr(scal), beta1, beta2,
                             eps, rows, _stream()))


def sum_partials(src, n_partials, stride, n, out):
    _count(1)
    check(lib().ltg_sum_partials(ptr(src), n_partials, stride, n, ptr(out), _stream()))


def enc_coef_clear(e_row, e_slot, n_entries, xc):
    _count(1)
    check(lib().ltg_enc_coef_clear(ptr(e_row), ptr(e_slot), n_entries, ptr(xc), xc.stride(0), _stream()))


def enc_xc_clear(indptr, indices, B, nnz, slot_of_item, xc):
    _count(1)
    check(lib().ltg_enc_xc_clear(ptr(indptr), ptr(indices), B, nnz, ptr(slot_of_item), ptr(xc), xc.stride(0), _stream()))


def enc_wgrad_expand(dW, n_items, slot_of_item, G):
    _count(1)
    check(lib().ltg_enc_wgrad_expand(ptr(dW), n_items, ptr(slot_of_item), ptr(G), _stream()))


def sample_pairs(logits, B, n_items, uid0, cand_ptr, cand_items, samp_ptr, pop_ptr, pop_items, item_valid, seed, step, step_dev,
                 samp_items, samp_partner, samp_valid, cnt, max_cand, user_order=None, cand_vals=None):
    """cand_vals (fp32, aligned with cand_items): the candidates' logits given explicitly (catalog-sharded layout); logits may be None."""
    _count(1)
    check(lib().ltg_sample_pairs_vals(ptr(logits), logits.stride(0) if logits is not None else 0, ptr(cand_vals), B, n_items, uid0, ptr(cand_ptr),
                                      ptr(cand_items), ptr(samp_ptr), ptr(pop_ptr), ptr(pop_items), ptr(item_valid), seed, step, ptr(step_dev),
                                      ptr(samp_items), ptr(samp_partner), ptr(samp_valid), ptr(cnt), max_cand, ptr(user_order), _stream()))


def disc_gather(E_bf16, pop_ids, niche_ids, P, Xp, Xn):
    _count(1)
    check(lib().ltg_disc_gather(ptr(E_bf16), ptr(pop_ids), ptr(niche_ids), P, ptr(Xp), ptr(Xn), _stream()))


def disc_head(Y3, P, h3, w4, b4, label, keep, y_out, scal, dz3=None, dw4=None, db4=None):
    _count(1)
    check(lib().ltg_disc_head(ptr(Y3), Y3.stride(0), P, h3, ptr(w4), ptr(b4), ptr(label), keep, ptr(y_out), ptr(scal), ptr(dz3),
                              ptr(dw4), ptr(db4), _stream()))


def disc_fused_supported(d):
    return bool(lib().ltg_disc_fused_supported(d.h0 + 1, d.ld1, d.ld2, d.ld3, d.off2, d.one3, d.h2, d.k3))


def disc_fwd_fused(Xp, Xn, P, d, label, keep, seed, rng_stream, rng_step_dev, Hd, y, scal, dz3=None, dw4=None, db4=None, dz12=None, rng_row0=0):
    """discriminator.py:16-55 in one launch; `d` is the package's Discriminator (ones-row weight layout). rng_row0: dropout-counter
    row of pair 0 (a launch over a row slice of a larger pair batch)."""
    _count(1)
    check(lib().ltg_disc_fwd_fused(ptr(Xp), ptr(Xn), P, d.h0 + 1, ptr(d.view("W1", "b")), d.ld1, ptr(d.view("W2", "b")), d.ld2, d.h2,
                                   ptr(d.view("W3", "b")), d.ld3, d.k3, d.off2, d.one3, ptr(d.view("w4")), ptr(d.view("b4")), ptr(label),
                                   keep, seed, rng_stream, 0, ptr(rng_step_dev), ptr(Hd), ptr(y), ptr(scal), ptr(dz3), ptr(dw4), ptr(db4),
                                   ptr(dz12), int(rng_row0), _stream()))


def topk_metrics(scores, n_rows, n_items, seen_ptr, seen_items, held_ptr, held_items, k, rks, topk_idx, dcg, hits):
    _count(1)
    import numpy as np
    rk = np.asarray(list(rks), dtype=np.int32)
    is_bf16 = scores.dtype == torch.bfloat16
    check(lib().ltg_topk_metrics(ptr(scores), int(is_bf16), scores.stride(0), n_rows, n_items, ptr(seen_ptr), ptr(seen_items),
                                 ptr(held_ptr), ptr(held_items), k, rk.ctypes.data if len(rk) else None, len(rk), ptr(topk_idx),
                                 ptr(dcg), ptr(hits), _stream()))


def topk_recommend(scores, n_rows, n_items, seen_ptr, seen_items, allow_bits, k, out_idx, out_logit, out_prob, out_lse):
    """Top-k eligible items per row of fp32 logits with their logits, probabilities (out_prob may be None) and the row's log-sum-exp
    over the whole catalog. seen_ptr/seen_items (CSR, may be None) and allow_bits (the uint32 bitmap held in an int32 tensor, may be
    None) choose what is eligible."""
    _count(1)
    assert scores.dtype == torch.float32 and out_idx.dtype == torch.int32
    assert allow_bits is None or (allow_bits.dtype == torch.int32 and allow_bits.numel() >= (n_items + 31) // 32)
    check(lib().ltg_topk_recommend(ptr(scores), scores.stride(0), n_rows, n_items, ptr(seen_ptr), ptr(seen_items), ptr(allow_bits), k,
                                   ptr(out_idx), ptr(out_logit), ptr(out_prob), ptr(out_lse), _stream()))


def cast_bf16(src, dst, rows, cols):
    _count(1)
    check(lib().ltg_cast_bf16(ptr(src), src.stride(0) if src.dim() > 1 else cols, ptr(dst), dst.stride(0) if dst.dim() > 1 else cols,
                              rows, cols, _stream()))
