"""Exact Viterbi hand-overs for models that do not forget their start, without a GPU: the host max-product composition
(engine.compose_shard_operators, semiring 'max') against a serial max-product recursion, the max-product scan and the operator
exchange across time shards through the whole C ABI on the CPU emulator (tests/emu/viterbi_scan_emu_driver.py), and the
exchange (TimeShardedTrajectories.viterbi_operator_exchange) on a gloo world of two processes."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from test_engine_emulated_cpu import engine_emu  # noqa: F401  (builds tests/emu/engine_emu.so when it is stale)

EMU = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'emu')


def _maxprod_op(p, A, frames):
    """Max-product operator of `frames` as [row normalised to sum one | log-scale]: row i = e_i carried through the frames."""
    N = A.shape[0]
    M, L = np.eye(N), np.zeros(N)
    for t in frames:
        M = (M[:, :, None] * A[None, :, :]).max(axis=1) * p[t]
        s = M.sum(axis=1)
        M, L = M / s[:, None], L + np.log(s)
    return np.concatenate([M, L[:, None]], axis=1)


def _serial(p, A, pi):
    """Normalised max-product vectors of every frame (_hidden.c:229-265 without back-pointers)."""
    T, N = p.shape
    d = np.zeros((T, N))
    v = pi * p[0]
    d[0] = v / v.sum()
    for t in range(1, T):
        v = (d[t - 1][:, None] * A).max(axis=0) * p[t]
        d[t] = v / v.sum()
    return d


def _shards(world, lengths, p_by_traj, A, pi):
    N = A.shape[0]
    ops = [np.zeros((len(lengths), N, N + 1)) for _ in range(world)]
    borders = [np.zeros((len(lengths), 2, N)) for _ in range(world)]
    owns = [[False] * len(lengths) for _ in range(world)]
    ser = [_serial(p, A, pi) for p in p_by_traj]
    for k, T in enumerate(lengths):
        for r in range(world):
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            owns[r][k] = hi > lo
            if hi > lo:
                ops[r][k] = _maxprod_op(p_by_traj[k], A, range(lo, hi))
                borders[r][k][1] = ser[k][hi - 1]
            else:
                ops[r][k] = np.concatenate([np.eye(N), np.zeros((N, 1))], axis=1)
    return ops, borders, owns, ser


def _model(N, rng, sticky):
    X = rng.random((N, N)) + (50.0 * np.eye(N) if sticky else 0.0)
    return X / X.sum(axis=1)[:, None], np.full(N, 1.0 / N)


@pytest.mark.parametrize('N,world', [(3, 2), (7, 5), (20, 3), (40, 4)])
def test_max_product_composition_equals_a_serial_recursion(N, world):
    """The exact vector at lo - 1 of every shard, composed from the first owner's end and the operators of the shards after
    it, equals the serial max-product vector there (ragged lengths, a 3-frame trajectory that leaves shards owning nothing)."""
    from bhmm_b200.engine import compose_shard_operators
    rng = np.random.default_rng(31 * N + world)
    A, pi = _model(N, rng, sticky=(N % 2 == 1))
    lengths = [400, 3, 97]
    p_by_traj = [rng.random((T, N)) + 1e-3 for T in lengths]
    ops, borders, owns, ser = _shards(world, lengths, p_by_traj, A, pi)
    fwd = compose_shard_operators(ops, borders, owns, semiring='max')
    assert fwd.shape == (world, len(lengths), N)
    for k, T in enumerate(lengths):
        first = True
        for r in range(world):
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            if hi <= lo or first:
                assert not fwd[r][k].any()
                first = first and hi <= lo
                continue
            np.testing.assert_allclose(fwd[r][k], ser[k][lo - 1], rtol=1e-11, atol=0)


def _drive(specs, **env):
    e = dict(os.environ, BHMM_B200_PANEL='1', BHMM_B200_LANE_VITERBI='0', **env)
    r = subprocess.run([sys.executable, os.path.join(EMU, 'viterbi_scan_emu_driver.py')] + specs, env=e,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert 'all ok' in r.stdout and 'FAIL' not in r.stdout
    return r.stdout


@pytest.mark.parametrize('N', [6, 20, 40])
def test_max_product_scan_in_one_batch(engine_emu, N):  # noqa: F811
    """A model that does not forget, in one batch: the chain-parallel pass takes its starts from the max-product scan (at
    most 4 fix-up sweeps) and its paths equal the oracle's."""
    _drive(['batch,%d' % N])


def test_margin_redo_returns_the_oracle_path(engine_emu):  # noqa: F811
    """With the guessed bound at 0 and a widened margin, the pass after the scan is redone at the measured bound (a second
    scan) and still returns the oracle's paths."""
    _drive(['redo,20'], BHMM_B200_VITERBI_SCAN_GUESS='0')


@pytest.mark.parametrize('N,world', [(6, 2), (20, 3)])
def test_exact_viterbi_borders_on_the_emulator(engine_emu, N, world):  # noqa: F811
    """Two-frame halos on 2-3 shards: the borders fail, the shards' max-product operators give exact starts, the borders
    certify after phase 1 again and the joined paths equal the oracle's; the first owned chain of a shard keeps its halo
    warm-up in the exact pass after the in-shard scan."""
    _drive(['shards,%d,%d' % (N, world)])


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _exchange_data(world, lengths, N):
    rng = np.random.default_rng(19)
    A, pi = _model(N, rng, sticky=True)
    p_by_traj = [rng.random((T, N)) + 1e-3 for T in lengths]
    return _shards(world, lengths, p_by_traj, A, pi)


def _gloo_worker(rank, world, port, out):
    import torch.distributed as td
    from bhmm_b200.engine import TimeShardedTrajectories
    td.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    lengths, N = [500, 1, 17], 5
    ops, borders, _, _ = _exchange_data(world, lengths, N)
    terms = np.array([10.0 + rank, 1e-13 * (rank + 1), -1.0])
    fwd, margin = TimeShardedTrajectories.viterbi_operator_exchange(ops[rank], terms, borders, lengths, rank, world, 'cpu')
    out[rank] = (fwd.tolist(), float(margin))
    td.destroy_process_group()


def test_viterbi_operator_exchange_world2():
    import torch.multiprocessing as mp
    from bhmm_b200.engine import TimeShardedTrajectories, compose_shard_operators
    world, lengths, N = 2, [500, 1, 17], 5
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    ops, borders, owns, ser = _exchange_data(world, lengths, N)
    fwd = compose_shard_operators(ops, borders, owns, semiring='max')
    for r in range(world):
        np.testing.assert_array_equal(np.array(out[r][0]), fwd[r])
    np.testing.assert_allclose(fwd[1][0], ser[0][249], rtol=1e-12)
    # shard 1's margin: shard 0's chains x worst plus the guessed border mismatch, times c
    want = TimeShardedTrajectories.VITERBI_MARGIN_C * (10.0 * 1e-13 + TimeShardedTrajectories.VITERBI_BORDER_GUESS)
    assert out[0][1] == 0.0 and out[1][1] == pytest.approx(want, rel=1e-12)


def _gloo_missing_halo_worker(rank, world, port, out):
    import torch.distributed as td
    from bhmm_b200.engine import TimeShardedTrajectories
    td.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    lengths, N = [500, 1, 17], 5
    ops, borders, _, _ = _exchange_data(world, lengths, N)
    terms = np.array([10.0, 1e-13, 0.0 if rank == 1 else -1.0])     # rank 1 has no halo frame before trajectory 0
    try:
        TimeShardedTrajectories.viterbi_operator_exchange(ops[rank], terms, borders, lengths, rank, world, 'cpu')
        out[rank] = 'returned'
    except RuntimeError as e:
        out[rank] = str(e)
    td.destroy_process_group()


def test_viterbi_operator_exchange_refuses_together():
    """A shard without the halo frame its exact start needs makes EVERY rank raise after the one gather (none is left
    waiting in a collective), with a RuntimeError (the estimator turns it into a warning and paths left at None)."""
    import torch.multiprocessing as mp
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_missing_halo_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    assert all('rank 1 holds no halo frame' in out[r] for r in range(2)), dict(out)


def test_margin_that_cannot_certify_is_refused():
    """A near-tie margin of 1 or more would flag every decision: refused, not clamped."""
    from bhmm_b200.engine import TimeShardedTrajectories
    with pytest.raises(RuntimeError, match='too wide'):
        TimeShardedTrajectories._viterbi_check_exchange([np.array([1e12, 1e-11, -1.0])] * 2, np.array([0.0, 25.0]))
    TimeShardedTrajectories._viterbi_check_exchange([np.array([10.0, 1e-13, -1.0])] * 2, np.array([0.0, 1e-11]))
