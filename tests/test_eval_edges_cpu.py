"""CPU: the edge table of tests/eval_edges.py (n <= 513) through the sharded driver (evaluate._align_ranks_steps) on the
CPU stand-ins of the three kernel backends, under the lockstep simulator, against the oracle. A failure here is in the
host logic (target partition, candidate and top-4 merges, counter reduction at empty shards), not in a kernel."""
from __future__ import annotations

import numpy as np
import pytest
import torch

from oracle import oracle
from snag_b200 import evaluate
from tests import eval_edges as ee
from tests import oracle_backend
from tests.test_fp32_eval_cpu import _operand as _fp32_operand
from tests.test_fp32_eval_cpu import backend as fp32_backend
from tests.test_l1_sharding_cpu import _operands as _l1_operands
from tests.test_l1_sharding_cpu import backend as l1_backend

N_MAX = 513


def _bf16_operand(x):
    n, d = x.shape
    X = torch.zeros((n, evaluate.round_up(d, 64)), dtype=torch.bfloat16)
    X[:, :d] = torch.from_numpy(x).to(torch.bfloat16)
    return X, torch.from_numpy(oracle.norm2(x))


def _run(route, x, y, csls, k, want_top3, world):
    """Every rank's result of the driver on `route`'s stand-in, and the oracle's."""
    n = x.shape[0]
    if route == "bf16":
        x, y = oracle.bf16_round(x), oracle.bf16_round(y)
        (X, xn), (Y, yn) = _bf16_operand(x), _bf16_operand(y)
        be, kw = oracle_backend, {}
    elif route == "fp32":
        (X, xn), (Y, yn) = _fp32_operand(x, 0), _fp32_operand(y, 1)
        be, kw = fp32_backend, {}
    else:
        X, Y, xn, yn, _ = _l1_operands(x, y)
        be, kw = l1_backend, {"two_sweep": False}
    res = evaluate.simulate_sharded(
        lambda r: evaluate._align_ranks_steps(be, X, Y, xn, yn, n, k, csls, want_top3, world, r, **kw), world)
    ref = oracle.align_eval_l1(x, y, csls, k) if route == "l1" else oracle.align_eval(x, y, csls, k)
    return res, ref


def _ids(cases):
    return ["-".join(str(v) for v in c) for c in cases]


_EDGES = [(route,) + c for route in ee.ROUTES for c in ee.edge_cases(route, N_MAX)]


@pytest.mark.parametrize("route,n,d,csls,k,want_top3,path", _EDGES, ids=_ids(_EDGES))
def test_edge_table_through_the_stand_ins(route, n, d, csls, k, want_top3, path):
    x, y = ee.clustered(n, d, 1.0, n + d)
    res, ref = _run(route, x, y, csls, k, want_top3, 1)
    ee.assert_equal_to_oracle(res[0], ref, csls, want_top3)


_SHARDED = [(route,) + c for route in ee.ROUTES for c in ee.sharded_cases(route) if c[0] <= N_MAX]


@pytest.mark.parametrize("route,n,d,world,csls,k", _SHARDED, ids=_ids(_SHARDED))
def test_sharded_edges_through_the_stand_ins(route, n, d, world, csls, k):
    sizes = ee.shard_sizes(n, world)
    assert sum(sizes) == n and min(sizes) <= 1, sizes          # a trailing rank owns one target or none
    x, y = ee.clustered(n, d, 1.0, 7 * n + world)
    res, ref = _run(route, x, y, csls, k, True, world)
    for r in res:                                                  # every rank ends with the full result
        assert r.info["shard"] == evaluate.shard_bounds(n, world, r.info["rank"])
        ee.assert_equal_to_oracle(r, ref, csls, True)


_DEGENERATE = [(route,) + c for route in ee.ROUTES for c in ee.degenerate_cases(route) if c[1] <= N_MAX]


@pytest.mark.parametrize("route,table,n,d", _DEGENERATE, ids=_ids(_DEGENERATE))
@pytest.mark.parametrize("world", [1, 3])
def test_degenerate_tables_through_the_stand_ins(route, table, n, d, world):
    x, y = ee.degenerate(table, n, d, n + d)
    res, ref = _run(route, x, y, True, 10, True, world)
    if table == "one_row":
        np.testing.assert_array_equal(ref["rank_l2r"], np.arange(n))          # every element a tie: stable order
        np.testing.assert_array_equal(ref["top3"], np.tile(np.arange(3), (n, 1)))
    for r in res:
        ee.assert_equal_to_oracle(r, ref, True, True)


def test_the_table_covers_every_size_and_width():
    for route in ee.ROUTES:
        cases = ee.edge_cases(route)
        for n in ee.N_EDGES:
            assert len({c[1] for c in cases if c[0] == n}) >= 2, (route, n)
        for d in ee.D_EDGES:
            assert len({c[0] for c in cases if c[1] == d}) >= 2, (route, d)
        assert {c[2] for c in cases} == {True, False} and {c[5] for c in cases} == set(ee.PATHS[route])
        assert {c[3] for c in cases if c[0] > 16} >= {1, 3, 16} and all(c[3] == c[0] for c in cases if c[0] == 1)
        assert {c[2] for c in ee.sharded_cases(route)} >= {2, 3, 8}
        for n, _d, world, _csls, _k in ee.sharded_cases(route):
            assert min(ee.shard_sizes(n, world)) <= 1
    # L1 operands are padded to a multiple of 8: the table has widths on both sides of it
    assert {d % 8 == 0 for d in ee.D_EDGES} == {True, False}
