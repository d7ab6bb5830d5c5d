"""Shared builders for synthetic Long-Tail-GAN inputs used by the tests (small, seeded)."""
import numpy as np


def synth_side_tables(rng, N, I, mean_nnz=18, n_pop=None, invalid=(3, 7)):
    """Random training CSR + the GAN side tables with the structure of the bundled dataset: the first n_pop item ids are
    "popular", the rest "niche"; candidates = own niche items + max(2n, 10-n) other niche items (data_processing.py:182)."""
    n_pop = max(4, I // 10) if n_pop is None else n_pop
    indptr = [0]
    indices = []
    pop_ptr, pop_items = [0], []
    n_niche = []
    cand_ptr, cand_items = [0], []
    real_ptr, real_niche, real_pop = [0], [], []
    eligible = []
    item_valid = np.ones(I, dtype=np.uint8)
    item_valid[list(invalid)] = 0
    niche_all = np.arange(n_pop, I)
    for u in range(N):
        n = int(np.clip(rng.poisson(mean_nnz), 2, I // 2))
        if u % 11 == 5:
            items = np.sort(rng.choice(niche_all, n, replace=False))  # niche only -> not eligible
        elif u % 13 == 7:
            items = np.sort(rng.choice(n_pop, min(n, n_pop), replace=False))  # popular only -> not eligible
        else:
            k_pop = int(np.clip(rng.binomial(n, 0.5), 1, min(n - 1, n_pop)))
            items = np.sort(np.concatenate([rng.choice(n_pop, k_pop, replace=False), rng.choice(niche_all, n - k_pop, replace=False)]))
        indices.append(items)
        indptr.append(indptr[-1] + len(items))
        pops = items[items < n_pop]
        niches = items[items >= n_pop]
        pops = rng.permutation(pops)  # file order, not sorted
        pop_items.append(pops); pop_ptr.append(pop_ptr[-1] + len(pops))
        ok = len(pops) > 0 and len(niches) > 0
        eligible.append(ok)
        n_niche.append(len(niches))
        if ok:
            others = np.setdiff1d(niche_all, niches)
            extra = rng.choice(others, min(len(others), max(2 * len(niches), 10 - len(niches))), replace=False)
            c = np.sort(np.concatenate([niches, extra]))
            rn, rp = [], []
            for g in niches:
                p = int(pops[rng.randint(len(pops))])
                if item_valid[g] and item_valid[p]:
                    rn.append(int(g)); rp.append(p)
        else:
            c, rn, rp = np.zeros(0, dtype=np.int64), [], []
        cand_items.append(c); cand_ptr.append(cand_ptr[-1] + len(c))
        real_niche += rn; real_pop += rp; real_ptr.append(real_ptr[-1] + len(rn))
    cat = lambda xs: np.concatenate(xs).astype(np.int32) if len(xs) else np.zeros(0, dtype=np.int32)  # noqa: E731
    return dict(n_items=I, indptr=np.asarray(indptr, dtype=np.int32), indices=cat(indices), pop_ptr=np.asarray(pop_ptr, dtype=np.int32),
                pop_items=cat(pop_items), n_niche=np.asarray(n_niche, dtype=np.int32), cand_ptr=np.asarray(cand_ptr, dtype=np.int32),
                cand_items=cat(cand_items), real_ptr=np.asarray(real_ptr, dtype=np.int32),
                real_niche=np.asarray(real_niche, dtype=np.int32), real_pop=np.asarray(real_pop, dtype=np.int32),
                eligible=np.asarray(eligible, dtype=bool), item_valid=item_valid)


def dense_rows(indptr, indices, r0, r1, I):
    X = np.zeros((r1 - r0, I), dtype=np.float32)
    for r in range(r0, r1):
        X[r - r0, indices[indptr[r]:indptr[r + 1]]] = 1.0
    return X


# ---- per-element error bounds against float64 references (torch tensors; torch is imported by the callers) -------------------------
TAU = 2.0 ** -14      # GEMM-shaped stages: |got - ref| <= TAU * (|A| |B|) per element, fp32 accumulation of exact bf16 products
U32 = 2.0 ** -24      # unit roundoff of fp32
HALF_BF16 = 2.0 ** -8  # half a bf16 ulp of any value of magnitude <= x is at most 2^-8 x
TINY = 1e-30


def gemm_ref(A, B):
    """float64 product of the exact (bf16 or fp32) operands and the product of their magnitudes (the per-element error scale)."""
    A = A.double(); B = B.double()
    return A @ B, A.abs() @ B.abs()


def drop_last_kblock(ref, A, B):
    """The reference with its last 64-deep k block missing: what a GEMM that skipped that block would compute."""
    K = A.shape[1]
    k0 = (K - 1) // 64 * 64
    return ref - A[:, k0:].double() @ B[k0:].double()


def assert_within(name, got, ref, bound):
    """Every element of `got` within `bound` of the float64 `ref`; prints the worst error-to-bound ratio and returns it."""
    import torch
    got = got.double()
    assert bool(torch.isfinite(got).all()), "%s: non-finite output" % name
    err = (got - ref).abs()
    bound = torch.broadcast_to(bound, err.shape)
    ratio = (err / bound.clamp_min(1e-300)).max().item() if err.numel() else 0.0
    bad = err > bound
    if bool(bad.any()):
        i = tuple(int(x) for x in torch.nonzero(bad)[0])
        raise AssertionError("%s: %d of %d elements out of bound, worst err/bound %.3g; first at %s: got %r ref %r bound %r"
                             % (name, int(bad.sum()), bad.numel(), ratio, i, got[i].item(), ref[i].item(), bound[i].item()))
    print("[bound] %-40s worst err/bound %.3g" % (name, ratio))
    return ratio


def assert_detects(name, got, wrong_ref, bound):
    """Sensitivity of a bound: a reference carrying an error of the kind that matters (a missing k block, a dropped split partial)
    must fail it somewhere."""
    import torch
    err = (got.double() - wrong_ref).abs()
    assert bool((err > torch.broadcast_to(bound, err.shape)).any()), "%s: the bound does not see the injected error" % name
