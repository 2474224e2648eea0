"""Host side of the Gibbs sweep on time shards: the composition of the shards' whole-shard maps (engine.compose_shard_maps)
against a serial walk, the library's sampling phases on the CPU emulator (tests/emu) against the oracle, and the
distributed exchange (TimeShardedTrajectories.gibbs_exchange) on a gloo world of two processes."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

from test_engine_emulated_cpu import engine_emu  # noqa: F401  (builds tests/emu/engine_emu.so when it is stale)

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.parametrize('seed', range(6))
def test_compose_equals_a_serial_walk(seed):
    from bhmm_b200.engine import compose_shard_maps
    rng = np.random.default_rng(seed)
    world, K, N = int(rng.integers(1, 9)), int(rng.integers(1, 5)), int(rng.integers(1, 40))
    maps = [rng.integers(0, N, size=(K, N)).astype(np.uint8) for _ in range(world)]
    owns = [[bool(rng.random() < 0.7) for _ in range(K)] for _ in range(world)]
    owns[world - 1][0] = False                         # a trajectory too short for the last shard
    enter = compose_shard_maps(maps, owns)
    assert enter.shape == (world, K)
    for k in range(K):
        owners = [r for r in range(world) if owns[r][k]]
        # serial: start anywhere at the end (the last owner's map ignores it), hop from owner to owner
        states = {}
        s = 0
        for r in reversed(owners):
            states[r] = s
            s = int(maps[r][k][s])
        for i, r in enumerate(owners):
            if i + 1 < len(owners):
                q = owners[i + 1]
                # the state at q's first owned frame is q's map applied to what enters q
                assert enter[r, k] == maps[q][k][max(enter[q, k], 0)]
            else:
                assert enter[r, k] == -1
        for r in range(world):
            if not owns[r][k]:
                later = [q for q in owners if q > r]
                if not later:
                    assert enter[r, k] == -1
                else:
                    q = later[0]
                    assert enter[r, k] == maps[q][k][max(enter[q, k], 0)]     # passed through unchanged


def test_compose_with_identity_maps_of_empty_shards():
    from bhmm_b200.engine import compose_shard_maps
    N = 5
    ident = np.arange(N, dtype=np.uint8)[None, :]
    last = np.full((1, N), 3, dtype=np.uint8)           # the end of the trajectory: a constant map
    mid = np.array([[4, 0, 1, 2, 3]], dtype=np.uint8)
    enter = compose_shard_maps([mid, ident, last], [[True], [False], [True]])
    assert enter[:, 0].tolist() == [3, 3, -1]
    enter = compose_shard_maps([mid, ident, last], [[True], [True], [True]])   # an owning shard with the identity map
    assert enter[:, 0].tolist() == [3, 3, -1]


@pytest.mark.parametrize('spec', ['3,2', '3,3', '20,2', '20,3'])
def test_sampling_phases_on_the_emulator(engine_emu, spec):  # noqa: F811
    env = dict(os.environ, BHMM_B200_PANEL='0', BHMM_B200_EXACT_SCAN='0')
    r = subprocess.run([sys.executable, os.path.join(HERE, 'emu', 'gibbs_shard_emu_driver.py'), spec], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert ' ok ' in r.stdout and 'FAIL' not in r.stdout


def test_tiled_link_with_entering_states_on_the_emulator(engine_emu):  # noqa: F811
    env = dict(os.environ, BHMM_B200_PANEL='0', BHMM_B200_EXACT_SCAN='0', BHMM_B200_CHASE_TILED='1')
    r = subprocess.run([sys.executable, os.path.join(HERE, 'emu', 'gibbs_shard_emu_driver.py'), '3,3'], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _exchange_data(world, K, N, lengths):
    """Every shard's maps and border vectors, the same in every process (seeded)."""
    rng = np.random.default_rng(5)
    maps = [rng.integers(0, N, size=(K, N)).astype(np.uint8) for _ in range(world)]
    v = rng.random((K, N)) + 0.1
    borders = [np.stack([v, v], axis=1) for _ in range(world)]     # used at lo - 1 == end at hi - 1 of the left neighbour
    return maps, borders


def _gloo_worker(rank, world, port, out):
    import torch.distributed as td
    from bhmm_b200.engine import TimeShardedTrajectories
    td.init_process_group('gloo', init_method='tcp://127.0.0.1:%d' % port, rank=rank, world_size=world)
    K, N, lengths = 3, 7, [1000, 1, 17]
    maps, borders = _exchange_data(world, K, N, lengths)
    enter, worst = TimeShardedTrajectories.gibbs_exchange(maps[rank], borders[rank], lengths, rank, world, 1e-11, 'cpu')
    out[rank] = (list(map(int, enter)), worst)
    td.destroy_process_group()


def test_distributed_exchange_world2():
    import torch.multiprocessing as mp
    from bhmm_b200.engine import compose_shard_maps
    world = 2
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_gloo_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    K, N, lengths = 3, 7, [1000, 1, 17]
    maps, _ = _exchange_data(world, K, N, lengths)
    owns = [[(T * (r + 1)) // world > (T * r) // world for T in lengths] for r in range(world)]
    want = compose_shard_maps(maps, owns)
    for r in range(world):
        assert out[r][0] == want[r].tolist()
        assert out[r][1] == 0.0
    # the one-frame trajectory lives on the last shard only: the first shard passes that shard's state through
    assert want[1][1] == -1 and want[0][1] == maps[1][1][0]
