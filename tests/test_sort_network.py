"""CPU check of the in-register sorting network of learning3d_b200/csrc/reg_sort.cuh (reg_sort_desc, with either
compare-exchange, cex_f32 or tpr_cex): the same loop nest restated in Python must be a sorting network (0/1 principle) with Batcher's merge-exchange size.
The GPU suites only see its results; this pins the loop structure itself."""
import itertools
import random


def merge_exchange(n):
    """Compare-exchange list (i, j), i < j, larger element ends at i — the loop nest of reg_sort.cuh."""
    ces = []
    p = n // 2
    while p >= 1:
        for i in range(n - p):
            if (i & p) == 0:
                ces.append((i, i + p))
        q = n // 2
        while q > p:
            d = q - p
            for i in range(n - d):
                if (i & p) == p:
                    ces.append((i, i + d))
            q //= 2
        p //= 2
    return ces


def run(ces, v):
    v = list(v)
    for i, j in ces:
        if v[i] < v[j]:
            v[i], v[j] = v[j], v[i]
    return v


def test_sizes_match_batcher():
    assert len(merge_exchange(8)) == 19
    assert len(merge_exchange(16)) == 63
    assert len(merge_exchange(32)) == 191      # bitonic: 240


def test_zero_one_principle_exhaustive_small():
    for n in (8, 16):
        ces = merge_exchange(n)
        for bits in itertools.product((0, 1), repeat=n):
            out = run(ces, bits)
            assert all(out[i] >= out[i + 1] for i in range(n - 1))


def test_zero_one_principle_sampled_32():
    rng = random.Random(5)
    ces = merge_exchange(32)
    for _ in range(20000):
        ones = rng.randrange(33)
        v = [1] * ones + [0] * (32 - ones)
        rng.shuffle(v)
        out = run(ces, v)
        assert out == sorted(v, reverse=True)
    for _ in range(2000):                       # and distinct keys
        v = rng.sample(range(1000), 32)
        assert run(ces, v) == sorted(v, reverse=True)
