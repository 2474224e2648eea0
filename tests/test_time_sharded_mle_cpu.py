"""Host side of the exact shard borders of the time-sharded E-step: the composition of the shards' operators
(engine.compose_shard_operators) against a serial numpy forward / backward, the library's operator kernels and border starts on
the CPU emulator (tests/emu) against a numpy product and the oracle, and the operator exchange
(TimeShardedTrajectories.operator_exchange) on a gloo world of two processes."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from test_engine_emulated_cpu import engine_emu  # noqa: F401  (builds tests/emu/engine_emu.so when it is stale)

HERE = os.path.dirname(os.path.abspath(__file__))


def _scaled_ops(p, A, frames):
    """prod over `frames` of (A D_t) in the library's representation: rows normalised to one, log of every row's scale."""
    N = A.shape[0]
    M, L = np.eye(N), np.zeros(N)
    for t in frames:
        M = M @ (A * p[t][None, :])
        s = M.sum(axis=1)
        M /= s[:, None]
        L += np.log(s)
    return np.concatenate([M, L[:, None]], axis=1)


def _serial(p, A, pi):
    """Scaled forward and backward variables of one trajectory (_hidden.c: alpha rows and beta rows normalised to one)."""
    T, N = p.shape
    alpha, beta = np.zeros((T, N)), np.zeros((T, N))
    a = pi * p[0]
    alpha[0] = a / a.sum()
    for t in range(1, T):
        a = (alpha[t - 1] @ A) * p[t]
        alpha[t] = a / a.sum()
    beta[T - 1] = 1.0 / N
    for t in range(T - 2, -1, -1):
        b = A @ (p[t + 1] * beta[t + 1])
        beta[t] = b / b.sum()
    return alpha, beta


def _shards(world, lengths, p_by_traj, A, pi):
    """Every shard's operators and border vectors as the library reports them, from the serial recursions."""
    K, N = len(lengths), A.shape[0]
    ops = [np.zeros((K, 2, N, N + 1)) for _ in range(world)]
    borders = [np.zeros((K, 4, N)) for _ in range(world)]
    owns = [[False] * K for _ in range(world)]
    ser = [_serial(p, A, pi) for p in p_by_traj]
    for r in range(world):
        for k, T in enumerate(lengths):
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            eye = np.concatenate([np.eye(N), np.zeros((N, 1))], axis=1)
            ops[r][k][0] = ops[r][k][1] = eye
            if hi <= lo:
                continue
            owns[r][k] = True
            p = p_by_traj[k]
            ops[r][k][0] = _scaled_ops(p, A, range(lo, hi))
            if hi < T:
                ops[r][k][1] = _scaled_ops(p, A, range(lo + 1, hi + 1))
            alpha, beta = ser[k]
            borders[r][k][1] = alpha[hi - 1]
            borders[r][k][3] = beta[lo]
            # what a too-short halo reports at the other two places: something else
            borders[r][k][0] = np.full(N, 1.0 / N)
            borders[r][k][2] = np.full(N, 1.0 / N)
    return ops, borders, owns, ser


@pytest.mark.parametrize('seed', range(8))
def test_compose_equals_a_serial_forward_backward(seed):
    from bhmm_b200.engine import compose_shard_operators
    rng = np.random.default_rng(seed)
    world, N = int(rng.integers(1, 6)), int(rng.integers(1, 9))
    lengths = [int(rng.integers(1, 60)) for _ in range(int(rng.integers(1, 4)))] + [1, 3]   # 1-frame ranges, empty shards
    X = rng.random((N, N)) + 3.0 * rng.random() * np.eye(N)
    A = X / X.sum(axis=1)[:, None]
    pi = rng.random(N)
    pi /= pi.sum()
    p_by_traj = [rng.random((T, N)) * np.exp(rng.normal(0, 3, (T, 1))) for T in lengths]   # wildly scaled emissions
    ops, borders, owns, ser = _shards(world, lengths, p_by_traj, A, pi)
    fwd, bwd = compose_shard_operators(ops, borders, owns)
    assert fwd.shape == bwd.shape == (world, len(lengths), N)
    for k, T in enumerate(lengths):
        alpha, beta = ser[k]
        owners = [r for r in range(world) if owns[r][k]]
        for r in range(world):
            lo, hi = (T * r) // world, (T * (r + 1)) // world
            if r in owners and r != owners[0]:
                np.testing.assert_allclose(fwd[r, k], alpha[lo - 1], rtol=1e-12, atol=1e-300)
            else:
                assert not fwd[r, k].any()
            if r in owners and r != owners[-1]:
                np.testing.assert_allclose(bwd[r, k], beta[hi], rtol=1e-12, atol=1e-300)
            else:
                assert not bwd[r, k].any()


def test_compose_passes_through_shards_that_own_nothing():
    from bhmm_b200.engine import compose_shard_operators
    N = 3
    rng = np.random.default_rng(1)
    A = rng.random((N, N))
    A /= A.sum(axis=1)[:, None]
    pi = np.full(N, 1.0 / N)
    # one trajectory of 2 frames on 4 shards: shards 0 and 2 own nothing, 1 and 3 own a frame each
    p = rng.random((2, N))
    ops, borders, owns, ser = _shards(4, [2], [p], A, pi)
    assert [o[0] for o in owns] == [False, True, False, True]
    fwd, bwd = compose_shard_operators(ops, borders, owns)
    alpha, beta = ser[0]
    np.testing.assert_allclose(fwd[3, 0], alpha[0], rtol=1e-13)
    np.testing.assert_allclose(bwd[1, 0], beta[1], rtol=1e-13)
    assert not fwd[1, 0].any() and not bwd[3, 0].any() and not fwd[0].any() and not bwd[2].any()


def _drive(specs, mode='0'):
    env = dict(os.environ, BHMM_B200_PANEL=mode)
    r = subprocess.run([sys.executable, os.path.join(HERE, 'emu', 'estep_shard_emu_driver.py')] + specs, env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert ' ok ' in r.stdout and 'FAIL' not in r.stdout
    return r


@pytest.mark.parametrize('spec', ['ops,3,3', 'ops,20,2', 'ops,40,3'])
def test_shard_operators_on_the_emulator(engine_emu, spec):  # noqa: F811
    """k_chain_operator[_wide] + k_compose_operators against a numpy product of (A D_t) over each shard's owned frames:
    7-frame chains give odd chain counts, 2-chain and single-chain runs; a 2-frame trajectory leaves shards owning nothing."""
    _drive([spec])


@pytest.mark.parametrize('spec', ['estep,3,2', 'estep,6,3', 'estep,3,5'])
def test_exact_border_starts_on_the_emulator(engine_emu, spec):  # noqa: F811
    """Two-frame halos on a sticky model: the borders fail, the composed operators give exact starts, the second E-step's
    borders certify and the summed statistics equal the oracle's; cleared starts warm up on the halo again."""
    _drive([spec])


def test_exact_border_starts_on_the_panel_kernels(engine_emu):  # noqa: F811
    """The same through the tensor-pipe (panel) kernels that serve 17 <= N <= 104 (wide layout at N = 20)."""
    _drive(['estep,20,2'], mode='1')


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _exchange_data(world, lengths, N):
    rng = np.random.default_rng(9)
    X = rng.random((N, N)) + np.eye(N)
    A = X / X.sum(axis=1)[:, None]
    pi = np.full(N, 1.0 / N)
    p_by_traj = [rng.random((T, N)) for T in lengths]
    return _shards(world, lengths, p_by_traj, A, pi)


def _gloo_worker(rank, world, port, out):
    import torch.distributed as td
    from bhmm_b200.engine import TimeShardedTrajectories
    td.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    lengths, N = [500, 1, 17], 5
    ops, borders, _, _ = _exchange_data(world, lengths, N)
    fwd, bwd = TimeShardedTrajectories.operator_exchange(ops[rank], borders, lengths, rank, world, 'cpu')
    out[rank] = (fwd.tolist(), bwd.tolist())
    td.destroy_process_group()


def test_operator_exchange_world2():
    import torch.multiprocessing as mp
    from bhmm_b200.engine import compose_shard_operators
    world, lengths, N = 2, [500, 1, 17], 5
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    ops, borders, owns, ser = _exchange_data(world, lengths, N)
    fwd, bwd = compose_shard_operators(ops, borders, owns)
    for r in range(world):
        np.testing.assert_array_equal(np.array(out[r][0]), fwd[r])
        np.testing.assert_array_equal(np.array(out[r][1]), bwd[r])
    np.testing.assert_allclose(fwd[1][0], ser[0][0][249], rtol=1e-12)
    np.testing.assert_allclose(bwd[0][0], ser[0][1][250], rtol=1e-12)
