"""Assignment of the cross terms of a sharded quadratic form to ranks (sharded.quadform_pair_assignment): every
unordered pair of shards exactly once, and the same work on every rank up to one half pair."""
from fractions import Fraction

import pytest

from basq_b200 import sharded


@pytest.mark.parametrize("world", range(1, 9))
def test_every_pair_once_and_balanced(world):
    tasks = sharded.quadform_pair_assignment(world)
    assert len(tasks) == world
    cover = {}
    work = []
    for r, mine in enumerate(tasks):
        w = Fraction(0)
        for i, j, half in mine:
            assert 0 <= i < j < world
            assert half in (None, 0, 1)
            if half is not None:
                assert r in (i, j)
            cover.setdefault((i, j), []).append(half)
            w += 1 if half is None else Fraction(1, 2)
        work.append(w)
    pairs = {(i, j) for i in range(world) for j in range(i + 1, world)}
    assert set(cover) == pairs
    for halves in cover.values():
        assert sorted(halves, key=str) in ([None], [0, 1])
    assert max(work) - min(work) <= Fraction(1, 2)
    assert sum(work) == len(pairs)
