"""CPU checks of the host tail of long-tail evaluation (engine.longtail_from_counts, engine.longtail_inputs) on hand-built counts with
known answers: Gini at its two extremes, coverage and niche coverage, which users each per-user list keeps, the IDCG cut at k, and
the rejection of bad niche / item_pop arguments."""
import importlib

import numpy as np
import pytest


@pytest.fixture(scope="module")
def eng():
    return importlib.import_module("long-tail-gan_b200.engine")


def _lt(eng, rec_count, niche_mask, n_held=(1,), n_held_niche=(0,), k=100, recall_ks=(20, 50), dcg_niche=None, hits_niche=None,
        n_niche_top=None, pop_sum=None):
    n = len(n_held)
    return eng.longtail_from_counts(np.zeros(n) if dcg_niche is None else np.asarray(dcg_niche, dtype=np.float64),
                                    np.zeros((n, len(recall_ks)), np.int32) if hits_niche is None else np.asarray(hits_niche, np.int32),
                                    np.zeros(n, np.int32) if n_niche_top is None else np.asarray(n_niche_top, np.int32),
                                    np.zeros(n, np.int64) if pop_sum is None else np.asarray(pop_sum, np.int64),
                                    np.asarray(rec_count, np.int32), np.asarray(n_held), np.asarray(n_held_niche), np.asarray(niche_mask, bool),
                                    k, recall_ks)


def test_gini_uniform_is_zero(eng):
    I = 37
    out = _lt(eng, np.full(I, 5), np.ones(I, bool))
    assert out["gini@100"] == 0.0
    assert out["coverage@100"] == 1.0 and out["niche_coverage@100"] == 1.0


def test_gini_single_item_is_maximal(eng):
    for I in (1, 2, 10, 1000):
        c = np.zeros(I, np.int32)
        c[I // 3] = 42
        out = _lt(eng, c, np.ones(I, bool))
        assert out["gini@100"] == pytest.approx((I - 1) / I, abs=1e-15)
        assert out["coverage@100"] == 1.0 / I


def test_gini_known_value_and_no_recommendations(eng):
    # c sorted ascending = (0, 1, 3): sum_j (2j - 4) c_(j) = -2*0 + 0*1 + 2*3 = 6; I * sum c = 12
    out = _lt(eng, [3, 0, 1], np.ones(3, bool))
    assert out["gini@100"] == 0.5
    assert _lt(eng, np.zeros(5), np.ones(5, bool))["gini@100"] == 0.0


def test_coverage_and_niche_coverage(eng):
    I = 10
    niche = np.zeros(I, bool)
    niche[[1, 4, 6, 9]] = True
    c = np.zeros(I, np.int32)
    c[[0, 1, 2, 6]] = [3, 1, 2, 7]      # four items recommended, two of them niche
    out = _lt(eng, c, niche)
    assert out["coverage@100"] == 0.4
    assert out["niche_coverage@100"] == 0.5


def test_user_filters_and_normalisation(eng):
    """Users without held-out niche items leave the niche lists but stay in niche share / avg pop; users without held-out items leave
    every list. kk = min(k, I) normalises share and popularity."""
    I, k = 50, 20
    niche = np.zeros(I, bool)
    niche[:10] = True
    n_held = [3, 0, 4, 2]
    n_held_niche = [2, 0, 0, 1]
    dcg = [1.0 + 1.0 / np.log2(3), 0.0, 0.0, 0.5]
    hits = [[2, 2], [0, 0], [0, 0], [1, 1]]
    top = [5, 7, 0, 20]
    pop = [100, 999, 40, 2 ** 20 * 20]
    out = _lt(eng, np.zeros(I), niche, n_held, n_held_niche, k=k, recall_ks=(5, 10), dcg_niche=dcg, hits_niche=hits, n_niche_top=top,
              pop_sum=pop)
    idcg2 = 1.0 + 1.0 / np.log2(3)
    assert out["niche_ndcg@20"] == [dcg[0] / idcg2, 0.5 / 1.0]
    assert out["niche_recall@5"] == [1.0, 1.0] and out["niche_recall@10"] == [1.0, 1.0]
    assert out["niche_share@20"] == [5 / 20, 0.0, 1.0]
    assert out["avg_pop@20"] == [100 / 20, 40 / 20, float(2 ** 20)]
    # a catalog smaller than k: kk = I
    out = _lt(eng, np.zeros(8), np.ones(8, bool), [1], [1], k=20, recall_ks=(5,), n_niche_top=[8], pop_sum=[16])
    assert out["niche_share@20"] == [1.0] and out["avg_pop@20"] == [2.0]


def test_idcg_cut_at_k_and_recall_denominator(eng):
    k = 3
    idcg3 = 1.0 + 1.0 / np.log2(3) + 0.5
    # 7 held-out niche items, list of 3 all hits: IDCG uses min(7, k) = 3 terms -> NDCG 1; recall@2 = 2 / min(2, 7)
    out = _lt(eng, np.zeros(10), np.ones(10, bool), [7], [7], k=k, recall_ks=(2, 3), dcg_niche=[idcg3], hits_niche=[[2, 3]])
    assert out["niche_ndcg@3"] == [1.0]
    assert out["niche_recall@2"] == [1.0] and out["niche_recall@3"] == [1.0]
    # 1 held-out niche item, hit at rank 2: 1/log2(3) / IDCG(1) = 1/log2(3); recall@3 = 1 / min(3, 1)
    out = _lt(eng, np.zeros(10), np.ones(10, bool), [5], [1], k=k, recall_ks=(3,), dcg_niche=[1.0 / np.log2(3)], hits_niche=[[1]])
    assert out["niche_ndcg@3"] == [1.0 / np.log2(3)] and out["niche_recall@3"] == [1.0]


def test_longtail_inputs_validation(eng):
    I = 20
    pop = np.arange(I)
    mask, p = eng.longtail_inputs([3, 5, 5], pop, I)
    assert mask.sum() == 2 and mask[3] and mask[5] and p.dtype == np.int64
    m = np.zeros(I, bool); m[7] = True
    assert np.array_equal(eng.longtail_inputs(m, pop, I)[0], m)
    bad = [
        dict(niche=[0, I], item_pop=pop),                      # id out of range
        dict(niche=[-1], item_pop=pop),
        dict(niche=[], item_pop=pop),                          # empty niche set
        dict(niche=np.zeros(I, bool), item_pop=pop),
        dict(niche=np.ones(I + 1, bool), item_pop=pop),        # mask of the wrong length
        dict(niche=[1], item_pop=pop[:-1]),                    # popularity of the wrong length
        dict(niche=[1], item_pop=np.r_[pop[:-1], -1]),         # negative count
        dict(niche=[1], item_pop=pop.astype(np.float64)),      # not counts
        dict(niche=[1], item_pop=None),                        # niche without item_pop
        dict(niche=None, item_pop=pop),                        # item_pop without niche
    ]
    for b in bad:
        with pytest.raises(ValueError):
            eng.longtail_inputs(b["niche"], b["item_pop"], I)


def test_summary_order_and_means(eng):
    m = {"niche_ndcg@100": [0.2, 0.4], "niche_recall@20": [0.5], "niche_recall@50": [1.0, 0.0], "niche_share@100": [0.1, 0.3],
         "avg_pop@100": [10.0, 30.0], "coverage@100": 0.25, "niche_coverage@100": 0.125, "gini@100": 0.75}
    s = eng.longtail_summary(m)
    assert list(s) == ["niche_ndcg", "niche_r20", "niche_r50", "niche_share", "avg_pop", "coverage", "niche_coverage", "gini"]
    assert list(s.values()) == pytest.approx([0.3, 0.5, 0.5, 0.2, 20.0, 0.25, 0.125, 0.75])
