"""Host rules of the genome-wide budget: the bracket's cost sum and the genome target (no kernel is launched)."""
import math
import random

import numpy as np


def test_genome_cost_sum_is_correctly_rounded_and_order_free():
    from rocco_b200.pipeline import genome_cost_sum
    rng = random.Random(3)
    lengths = [1, 2, 257, 4096, 4097, 70_001, 300_001, 5_000_003]
    gammas = [0.0, 1.0, 6.86, 0.1, 1e-7, 3.3333333333333335, 0.7, 2.0 / 3.0]
    want = math.fsum(x for n, g in zip(lengths, gammas) for x in [g] * (n - 1))
    assert genome_cost_sum(lengths, gammas) == want
    for _ in range(5):
        order = list(range(len(lengths)))
        rng.shuffle(order)
        assert genome_cost_sum([lengths[k] for k in order], [gammas[k] for k in order]) == want
    # a chromosome split differently over "ranks" is the same multiset of costs
    assert genome_cost_sum(lengths[:3] + lengths[3:], gammas) == want
    # numpy's pairwise sum of the same vector is not order-free in general; this one is exact by construction
    assert genome_cost_sum([1], [5.0]) == 0.0 and genome_cost_sum([], []) == 0.0


def test_genome_target():
    from rocco_b200.pipeline import target_count_for_budget
    lengths = [4096, 70_001, 300_001]
    n = sum(lengths)
    for budget in (0.0, 0.02, 0.3, 0.035, 1.0):
        assert target_count_for_budget(n, budget) == int(np.floor(n * budget))
    # the genome target is NOT the sum of per-chromosome targets
    assert target_count_for_budget(n, 0.3) == 112229 != sum(target_count_for_budget(k, 0.3) for k in lengths)
    assert target_count_for_budget(n, 1.0) == n
