"""The panel kernels' actual CUDA source (bhmm_b200/csrc/panel_kernels.cu) executed on the CPU by tests/emu/warp_emu.h
(every CUDA thread a fiber, warp collectives and mma.sync.m8n8k4.f64 emulated from their PTX definitions) and compared
with a plain scaled forward-backward on whole trajectories (the algorithm of bhmm/hidden/impl_c/_hidden.c:16-183).

Written because the kernels could not be run on a GPU in the round they were written in: this executes their control
flow, indexing and collectives for real -- several blocks, partially filled warps, the persistent stride loop, warm-up
and exact (fix-up) starts, ragged trajectories, the three emission kinds, the outlier rule -- and would abort on a
divergent collective (a hang on hardware).  What it cannot show: race conditions between warps, ptxas behaviour, speed.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
EMU = os.path.join(HERE, 'emu')
PN = 32
EM_POBS, EM_GAUSS, EM_DISC = 0, 1, 2


@pytest.fixture(scope='module')
def emu():
    so = os.path.join(EMU, 'panel_emu.so')
    deps = [os.path.join(EMU, 'panel_emu.cpp'), os.path.join(EMU, 'warp_emu.h'),
            os.path.join(HERE, '..', 'bhmm_b200', 'csrc', 'panel_kernels.cu'), os.path.join(HERE, '..', 'bhmm_b200', 'csrc', 'kernels.h'),
            os.path.join(HERE, '..', 'bhmm_b200', 'csrc', 'common.cuh')]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        cuda_inc = os.path.join(os.environ.get('CUDA_HOME', '/usr/local/cuda'), 'include')
        if not os.path.exists(os.path.join(cuda_inc, 'cuda_runtime.h')):
            pytest.skip('CUDA headers not found')
        subprocess.run(['g++', '-O1', '-std=c++17', '-shared', '-fPIC', '-w', '-I' + cuda_inc, '-o', so,
                        os.path.join(EMU, 'panel_emu.cpp')], check=True)
    return C.CDLL(so)


@pytest.fixture
def request_cleanup():
    todo = []
    yield todo
    for fn in todo:
        fn()


def gauss(o, mu, sigma):
    return np.exp(-0.5 * ((o - mu) / sigma) ** 2) / (np.sqrt(2 * np.pi) * sigma)


def plain_estep(ps, A, pi):
    """ps: list of (T,N) emission tables.  Per-frame normalised forward-backward, gamma, xi counts; lc: the log of every
    frame's normaliser (row by row, its sum is ll)."""
    N = len(pi)
    out = dict(alpha=[], beta=[], gamma=[], ll=0.0, lc=[], C=np.zeros((N, N)), g0=np.zeros(N))
    for p in ps:
        T = len(p)
        al, be = np.zeros((T, N)), np.zeros((T, N))
        for t in range(T):
            v = pi * p[0] if t == 0 else al[t - 1].dot(A) * p[t]
            out['ll'] += np.log(v.sum())
            out['lc'].append(np.log(v.sum()))
            al[t] = v / v.sum()
        be[T - 1] = 1.0 / N
        for t in range(T - 2, -1, -1):
            v = A.dot(p[t + 1] * be[t + 1])
            be[t] = v / v.sum()
        gam = al * be
        gam /= gam.sum(axis=1)[:, None]
        for t in range(T - 1):
            x = al[t][:, None] * A * (p[t + 1] * be[t + 1])[None, :]
            out['C'] += x / x.sum()
        out['g0'] += gam[0]
        out['alpha'].append(al)
        out['beta'].append(be)
        out['gamma'].append(gam)
    for k in ('alpha', 'beta', 'gamma'):
        out[k] = np.vstack(out[k])
    out['lc'] = np.array(out['lc'])
    return out


def make_plan(Ts, chunk):
    row0, ln, t0, TT, row = [], [], [], [], 0
    for T in Ts:
        for a in range(0, T, chunk):
            row0.append(row + a)
            ln.append(min(chunk, T - a))
            t0.append(a)
            TT.append(T)
        row += T
    return (np.array(row0, dtype=np.int64), np.array(ln, dtype=np.int32), np.array(t0, dtype=np.int32),
            np.array(TT, dtype=np.int32))


def ptr(a, t=C.c_double):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


class Run(object):
    def __init__(self, emu, plan, A, pi, em_kind, obs=None, pobs=None, sym=None, mu=None, sigma=None, Bt=None, M=0,
                 ignore_outliers=0):
        self.emu, self.plan, self.A, self.pi, self.kind = emu, plan, np.ascontiguousarray(A), np.ascontiguousarray(pi), em_kind
        self.N = PN = len(pi)
        self.wide32 = False
        self.em = (ptr(pobs), ptr(obs), ptr(sym, C.c_int), ptr(mu), ptr(sigma), ptr(Bt), C.c_int(M), C.c_int(ignore_outliers))
        self._keep = (obs, pobs, sym, mu, sigma, Bt)
        n = len(plan[0])
        rows = int(plan[0][-1] + plan[1][-1])
        self.n, self.rows = n, rows
        self.alpha = np.zeros((rows, PN))
        self.chain_ll = np.zeros(n)
        self.hu_f, self.he_f = np.zeros((n, PN)), np.zeros((n, PN))
        self.hu_b, self.he_b = np.zeros((n, PN)), np.zeros((n, PN))

    def _chains(self, warm, exact, chain_list):
        row0, ln, t0, TT = self.plan
        lst = None if chain_list is None else np.array(chain_list, dtype=np.int32)
        n_run = self.n if lst is None else len(lst)
        return (ptr(row0, C.c_longlong), ptr(ln, C.c_int), ptr(t0, C.c_int), ptr(TT, C.c_int), ptr(lst, C.c_int),
                C.c_int(n_run), C.c_int(warm), None, C.c_int(exact)), lst

    def forward(self, grid, warm, exact=0, chain_list=None):
        ch, keep = self._chains(warm, exact, chain_list)
        rc = self.emu.panel_emu_forward(C.c_int(self.N), C.c_int(self.kind), C.c_int(grid), *ch, *self.em, ptr(self.A), ptr(self.pi),
                                        ptr(self.alpha), ptr(self.chain_ll), ptr(self.hu_f), ptr(self.he_f))
        assert rc == 0

    def backward_stats(self, grid, warm, alpha, exact=0, gamma=None, Bnum=None):
        ch, keep = self._chains(warm, exact, None)
        PN = self.N
        pw = self.emu.panel_emu_warps_per_block() if (PN == 32 and not self.wide32) else 1
        partials = np.full((grid * pw, PN * PN + 4 * PN), np.nan)     # every row must be written by its warp / block
        rc = self.emu.panel_emu_backward_stats(C.c_int(PN), C.c_int(self.kind), C.c_int(grid), *ch, *self.em, ptr(self.A),
                                               ptr(np.ascontiguousarray(alpha)), ptr(gamma), ptr(Bnum), ptr(partials),
                                               ptr(self.hu_b), ptr(self.he_b))
        assert rc == 0
        assert not np.isnan(partials).any()
        s = partials.sum(axis=0)
        return dict(C=self.A * s[:PN * PN].reshape(PN, PN), g0=s[PN * PN:PN * PN + PN], sg=s[PN * PN + PN:PN * PN + 2 * PN],
                    sgd=s[PN * PN + 2 * PN:PN * PN + 3 * PN], sgdd=s[PN * PN + 3 * PN:])


def model(seed, mixing=3.0, N=PN):
    rng = np.random.default_rng(seed)
    A = rng.random((N, N)) + mixing * np.eye(N)            # fast mixing: a 48-frame warm-up forgets its start
    A /= A.sum(axis=1)[:, None]
    pi = rng.random(N)
    pi /= pi.sum()
    return rng, A, pi, np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)


def check_handovers(run, ref, plan):
    row0, ln, t0, TT = plan
    for c in range(len(row0)):
        np.testing.assert_allclose(run.he_f[c], ref['alpha'][row0[c] + ln[c] - 1], rtol=1e-10)
        if t0[c] > 0:
            np.testing.assert_allclose(run.hu_f[c], ref['alpha'][row0[c] - 1], rtol=1e-10)
            np.testing.assert_allclose(run.he_b[c], ref['beta'][row0[c]], rtol=1e-10)
        if t0[c] + ln[c] < TT[c]:
            np.testing.assert_allclose(run.hu_b[c], ref['beta'][row0[c] + ln[c]], rtol=1e-10)


@pytest.mark.parametrize('grid', [2, 1])
def test_gaussian_estep_warm_up_mode(emu, grid):
    """42 chains of ragged trajectories (one of a single frame, one shorter than a chunk): grid = 2 leaves the second block
    partly idle, grid = 1 makes the warps stride over two chain groups."""
    rng, A, pi, mu, sigma = model(11)
    Ts = [130, 97, 1, 64, 20, 111, 75, 33, 128, 60, 90, 45]
    trajs = [mu[rng.integers(0, PN, T)] + 0.7 * rng.standard_normal(T) for T in Ts]
    obs = np.concatenate(trajs)
    plan = make_plan(Ts, 24)
    assert len(plan[0]) == 42
    ref = plain_estep([gauss(o[:, None], mu[None, :], sigma[None, :]) for o in trajs], A, pi)
    run = Run(emu, plan, A, pi, EM_GAUSS, obs=obs, mu=mu, sigma=sigma, ignore_outliers=1)
    run.forward(grid, warm=48)
    np.testing.assert_allclose(run.alpha, ref['alpha'], rtol=1e-10, atol=1e-300)
    assert abs(run.chain_ll.sum() - ref['ll']) <= 1e-12 * abs(ref['ll'])
    gamma = np.zeros((run.rows, PN))
    st = run.backward_stats(grid, 48, run.alpha, gamma=gamma)
    np.testing.assert_allclose(gamma, ref['gamma'], rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9)
    np.testing.assert_allclose(st['g0'], ref['g0'], rtol=1e-10)
    np.testing.assert_allclose(st['sg'], ref['gamma'].sum(axis=0), rtol=1e-10)
    d = obs[:, None] - mu[None, :]
    np.testing.assert_allclose(st['sgd'], (ref['gamma'] * d).sum(axis=0), rtol=1e-9, atol=1e-10)
    np.testing.assert_allclose(st['sgdd'], (ref['gamma'] * d * d).sum(axis=0), rtol=1e-10)
    assert abs(st['C'].sum() - (sum(Ts) - len(Ts))) < 1e-8
    check_handovers(run, ref, plan)


def test_exact_fix_up_pass_over_a_chain_list(emu):
    """Slow mixing and a warm-up that is too short: the hand-overs disagree; an exact pass over the listed chains (each
    starting from its predecessor's recorded last row, in order) repairs them -- the certification's fix-up sweep."""
    rng, A, pi, mu, sigma = model(5, mixing=40.0)
    Ts = [90, 70]
    trajs = [mu[rng.integers(0, PN, T)] + 2.5 * rng.standard_normal(T) for T in Ts]
    obs = np.concatenate(trajs)
    plan = make_plan(Ts, 30)
    ref = plain_estep([gauss(o[:, None], mu[None, :], sigma[None, :]) for o in trajs], A, pi)
    run = Run(emu, plan, A, pi, EM_GAUSS, obs=obs, mu=mu, sigma=sigma, ignore_outliers=1)
    run.forward(1, warm=2)
    assert np.max(np.abs(run.alpha - ref['alpha'])) > 1e-6
    t0 = plan[2]
    for c in range(len(t0)):               # chains that do not start a trajectory, one after the other
        if t0[c] > 0:
            run.forward(1, warm=2, exact=1, chain_list=[c])
    np.testing.assert_allclose(run.alpha, ref['alpha'], rtol=1e-10, atol=1e-300)
    assert abs(run.chain_ll.sum() - ref['ll']) <= 1e-12 * abs(ref['ll'])
    # exact backward start: every chain enters with the true beta of the frame after it
    row0, ln = plan[0], plan[1]
    for c in range(len(t0)):
        run.he_b[c] = ref['beta'][row0[c]]
    st = run.backward_stats(1, 2, ref['alpha'], exact=1)
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9)
    np.testing.assert_allclose(st['sg'], ref['gamma'].sum(axis=0), rtol=1e-10)


def test_discrete_and_table_emissions_with_outlier_frames(emu):
    rng, A, pi, mu, sigma = model(23)
    M = 12
    B = rng.random((PN, M)) ** 3 + 1e-4
    B[:, 7] = 0.0                                           # a symbol no state emits: an outlier frame
    B /= B.sum(axis=1)[:, None]
    Ts = [70, 41, 9]
    syms = [rng.integers(0, M, T).astype(np.int32) for T in Ts]
    syms[0][33] = 7
    syms[1][0] = 7
    sym = np.concatenate(syms)
    Bt = np.ascontiguousarray(B.T)
    plan = make_plan(Ts, 16)
    ps = []
    for s in syms:
        p = B[:, s].T.copy()
        p[p.sum(axis=1) == 0] = 1.0                         # outputmodel.py:126-130
        ps.append(p)
    ref = plain_estep(ps, A, pi)
    run = Run(emu, plan, A, pi, EM_DISC, sym=sym, Bt=Bt, M=M, ignore_outliers=1)
    run.forward(1, warm=40)
    np.testing.assert_allclose(run.alpha, ref['alpha'], rtol=1e-10, atol=1e-300)
    assert abs(run.chain_ll.sum() - ref['ll']) <= 1e-12 * abs(ref['ll'])
    Bnum = np.zeros((PN, M))
    st = run.backward_stats(1, 40, run.alpha, Bnum=Bnum)
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9)
    np.testing.assert_allclose(st['g0'], ref['g0'], rtol=1e-10)
    want = np.zeros((PN, M))
    np.add.at(want.T, sym, ref['gamma'])
    np.testing.assert_allclose(Bnum, want, rtol=1e-9, atol=1e-14)
    # the same frames through a caller's p_obs table (EM_POBS: no outlier rule inside the kernel)
    pobs = np.ascontiguousarray(np.vstack(ps))
    run2 = Run(emu, plan, A, pi, EM_POBS, pobs=pobs)
    run2.forward(1, warm=40)
    np.testing.assert_allclose(run2.alpha, ref['alpha'], rtol=1e-10, atol=1e-300)
    st2 = run2.backward_stats(1, 40, run2.alpha)
    np.testing.assert_allclose(st2['C'], ref['C'], rtol=1e-9)


def test_exp8_tail_far_observations(emu):
    """Observations tens of sigma away from most states: the polynomial exp's tail (exact zeros below -746, the library
    exp in the denormal band) must agree with libm's densities."""
    rng, A, pi, mu, sigma = model(31)
    T = 40
    o = np.concatenate([rng.standard_normal(T - 6) * 4.0, [19.0, -19.5, 21.0, 18.7, -20.3, 0.0]])
    ref = plain_estep([gauss(o[:, None], mu[None, :], sigma[None, :])], A, pi)
    plan = make_plan([T], 64)
    run = Run(emu, plan, A, pi, EM_GAUSS, obs=o, mu=mu, sigma=sigma, ignore_outliers=1)
    run.forward(1, warm=0)
    np.testing.assert_allclose(run.alpha, ref['alpha'], rtol=1e-9, atol=1e-300)
    assert abs(run.chain_ll.sum() - ref['ll']) <= 1e-12 * abs(ref['ll'])


# ------------------------------------------------------------------------------------------------ wide kernels, 32 < N <= 104
@pytest.mark.parametrize('N,grid', [(100, 2), (37, 1), (64, 1), (32, 2), (21, 1)])
def test_wide_gaussian_estep(emu, N, grid, request_cleanup):
    """The wide kernels as the launchers dispatch them: a block of N/8 warps, state tiles exchanged through shared memory;
    k_forward_wide2 / k_backward_stats_wide2 (two sets of 8 chains per block, outlier machinery compiled in) at N = 100
    (C4's state count, padded to 104: 13 warps, B fragments in shared memory, one backward chain set per block), an odd N
    with a half-empty last tile and a full 64; the one-set k_forward_wide / k_backward_stats_wide (4 warps per 8 chains) at
    N = 32 (the alternative to the one-warp kernels there) and N = 21.  tests/test_panel_family_emulated_cpu.py covers
    every tile occupancy."""
    rng, A, pi, mu, sigma = model(100 + N, N=N)
    Ts = [50, 33, 1, 41, 18, 29]
    trajs = [mu[rng.integers(0, N, T)] + 0.7 * rng.standard_normal(T) for T in Ts]
    trajs[3][7] = 400.0                                     # far from every state: all densities underflow (outlier rule)
    obs = np.concatenate(trajs)
    plan = make_plan(Ts, 13)
    ps = []
    for o in trajs:
        p = gauss(o[:, None], mu[None, :], sigma[None, :])
        p[p.sum(axis=1) == 0] = 1.0
        ps.append(p)
    ref = plain_estep(ps, A, pi)
    run = Run(emu, plan, A, pi, EM_GAUSS, obs=obs, mu=mu, sigma=sigma, ignore_outliers=1)
    run.wide32 = True
    emu.panel_emu_force_wide(1)                             # N = 32 on the wide kernels too (BHMM_B200_PANEL=2)
    request_cleanup.append(lambda: emu.panel_emu_force_wide(0))
    run.forward(grid, warm=30)
    np.testing.assert_allclose(run.alpha, ref['alpha'], rtol=1e-10, atol=1e-300)
    assert abs(run.chain_ll.sum() - ref['ll']) <= 1e-12 * abs(ref['ll'])
    gamma = np.zeros((run.rows, N))
    st = run.backward_stats(grid, 30, run.alpha, gamma=gamma)
    np.testing.assert_allclose(gamma, ref['gamma'], rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(st['g0'], ref['g0'], rtol=1e-10)
    np.testing.assert_allclose(st['sg'], ref['gamma'].sum(axis=0), rtol=1e-10)
    d = obs[:, None] - mu[None, :]
    np.testing.assert_allclose(st['sgdd'], (ref['gamma'] * d * d).sum(axis=0), rtol=1e-10)
    np.testing.assert_allclose(st['sgd'], (ref['gamma'] * d).sum(axis=0), rtol=1e-9, atol=1e-7)
    assert abs(st['C'].sum() - (sum(Ts) - len(Ts))) < 1e-8
    row0, ln, t0, TT = plan
    for c in range(len(row0)):
        np.testing.assert_allclose(run.he_f[c], ref['alpha'][row0[c] + ln[c] - 1], rtol=1e-10, atol=1e-300)
        if t0[c] > 0:
            np.testing.assert_allclose(run.hu_f[c], ref['alpha'][row0[c] - 1], rtol=1e-10, atol=1e-300)
            np.testing.assert_allclose(run.he_b[c], ref['beta'][row0[c]], rtol=1e-10)
        if t0[c] + ln[c] < TT[c]:
            np.testing.assert_allclose(run.hu_b[c], ref['beta'][row0[c] + ln[c]], rtol=1e-10)


def test_wide_discrete_c4_shape_and_fix_up(emu):
    """N = 100 states, discrete symbols (the C4 model family) with a symbol no state emits, B-numerators, and an exact
    fix-up pass over a chain list after a warm-up that is too short, on k_forward_wide2 / k_backward_stats_wide2 at 13
    tiles with the outlier rule on."""
    N, M = 100, 30
    rng, A, pi, mu, sigma = model(77, mixing=25.0, N=N)
    B = rng.random((N, M)) ** 3 + 1e-4
    B[:, 5] = 0.0
    B /= B.sum(axis=1)[:, None]
    Ts = [40, 26]
    syms = [rng.integers(0, M, T).astype(np.int32) for T in Ts]
    syms[0][17] = 5
    sym = np.concatenate(syms)
    Bt = np.ascontiguousarray(B.T)
    plan = make_plan(Ts, 11)
    ps = []
    for s_ in syms:
        p = B[:, s_].T.copy()
        p[p.sum(axis=1) == 0] = 1.0
        ps.append(p)
    ref = plain_estep(ps, A, pi)
    run = Run(emu, plan, A, pi, EM_DISC, sym=sym, Bt=Bt, M=M, ignore_outliers=1)
    run.forward(1, warm=1)
    assert np.max(np.abs(run.alpha - ref['alpha'])) > 1e-8
    t0 = plan[2]
    for c in range(len(t0)):
        if t0[c] > 0:
            run.forward(1, warm=1, exact=1, chain_list=[c])
    np.testing.assert_allclose(run.alpha, ref['alpha'], rtol=1e-10, atol=1e-300)
    assert abs(run.chain_ll.sum() - ref['ll']) <= 1e-12 * abs(ref['ll'])
    Bnum = np.zeros((N, M))
    st = run.backward_stats(1, 60, ref['alpha'], Bnum=Bnum)            # warm-up longer than the trajectories: exact
    np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9, atol=1e-300)
    np.testing.assert_allclose(st['g0'], ref['g0'], rtol=1e-10)
    want = np.zeros((N, M))
    np.add.at(want.T, sym, ref['gamma'])
    np.testing.assert_allclose(Bnum, want, rtol=1e-9, atol=1e-14)


# ------------------------------------------------------------------------------------------------ Viterbi, 32 < N <= 104
def _resolve(F, T):
    """Path from the shifted back-pointer map (CHASE layout of k_viterbi_team / k_viterbi_regs)."""
    path = np.zeros(T, dtype=np.int32)
    path[T - 1] = F[T - 1, 0]
    for t in range(T - 2, -1, -1):
        path[t] = F[t, path[t + 1]]
    return path


@pytest.mark.parametrize('N', [100, 40, 64])
def test_viterbi_regs_is_bit_exact(emu, oracle_port, N):
    """k_viterbi_regs (matrix column in registers, four interleaved first-maximum scans, unrolled sequential row sum) against
    the oracle's restatement of _compute_viterbi (_hidden.c:203-281): identical paths, including exact ties (a model with
    repeated rows / columns and repeated emission values makes ties common) and an outlier frame in the discrete model."""
    rng = np.random.default_rng(N)
    M = 9
    X = rng.integers(1, 4, size=(N, N)).astype(float)       # small integers: many exactly equal products
    X += 6.0 * np.eye(N)
    A = X / X.sum(axis=1)[:, None]
    pi = np.ones(N) / N
    B = rng.integers(0, 3, size=(N, M)).astype(float) + 0.0
    B[:, 4] = 0.0
    B[:, 0] += 1.0
    B /= B.sum(axis=1)[:, None]
    Ts = [57, 1, 23, 40, 2]
    syms = [rng.integers(0, M, T).astype(np.int32) for T in Ts]
    syms[0][20] = 4                                         # no state emits symbol 4
    sym = np.concatenate(syms)
    offsets = np.concatenate([[0], np.cumsum(Ts)]).astype(np.int64)
    Bt = np.ascontiguousarray(B.T)
    A = np.ascontiguousarray(A)
    rows = int(offsets[-1])
    for grid in (2, 7):
        F = np.full((rows, N), 255, dtype=np.uint8)
        rc = emu.panel_emu_viterbi(C.c_int(N), C.c_int(EM_DISC), C.c_int(grid), C.c_int(len(Ts)), ptr(offsets, C.c_longlong),
                                   None, None, ptr(sym, C.c_int), None, None, ptr(Bt), C.c_int(M), C.c_int(1), ptr(A),
                                   ptr(pi), F.ctypes.data_as(C.POINTER(C.c_ubyte)))
        assert rc == 0
        for k, T in enumerate(Ts):
            pobs = oracle_port.discrete_p_obs(syms[k], B)
            pobs[pobs.sum(axis=1) == 0] = 1.0
            want = oracle_port.viterbi(A, pobs, pi)
            got = _resolve(F[offsets[k]:offsets[k + 1]], T)
            assert np.array_equal(got, want), (N, grid, k)
    # structural ties ACROSS the four scan blocks: a rank-one transition matrix and emission rows that repeat with period 3,
    # so every state has N/3 exact twins and only the first-maximum rule decides
    A1 = np.full((N, N), 1.0 / N)
    B1 = np.array([[0.5, 0.25, 0.25], [0.25, 0.5, 0.25], [0.125, 0.125, 0.75]])[np.arange(N) % 3]
    s1 = rng.integers(0, 3, 50).astype(np.int32)
    off1 = np.array([0, 50], dtype=np.int64)
    F = np.zeros((50, N), dtype=np.uint8)
    rc = emu.panel_emu_viterbi(C.c_int(N), C.c_int(EM_DISC), C.c_int(1), C.c_int(1), ptr(off1, C.c_longlong), None, None,
                               ptr(s1, C.c_int), None, None, ptr(np.ascontiguousarray(B1.T)), C.c_int(3), C.c_int(0),
                               ptr(A1), ptr(pi), F.ctypes.data_as(C.POINTER(C.c_ubyte)))
    assert rc == 0
    want = oracle_port.viterbi(A1, oracle_port.discrete_p_obs(s1, B1), pi)
    assert np.array_equal(_resolve(F, 50), want)
    assert len(set(want.tolist())) <= 3 and want.max() <= 2          # always the FIRST of the twins
    # caller's table (EM_POBS), continuous densities
    T = 35
    pobs = np.ascontiguousarray(rng.random((T, N)) ** 4)
    F = np.zeros((T, N), dtype=np.uint8)
    off1 = np.array([0, T], dtype=np.int64)
    rc = emu.panel_emu_viterbi(C.c_int(N), C.c_int(EM_POBS), C.c_int(1), C.c_int(1), ptr(off1, C.c_longlong), ptr(pobs),
                               None, None, None, None, None, C.c_int(0), C.c_int(0), ptr(A), ptr(pi),
                               F.ctypes.data_as(C.POINTER(C.c_ubyte)))
    assert rc == 0
    assert np.array_equal(_resolve(F, T), oracle_port.viterbi(A, pobs, pi))


# ------------------------------------------------------------------------------------------------ time-chunked Viterbi, N <= 32
def _viterbi_chain(emu, N, em_kind, plan, A, pi, grid, warm, exact=0, chain_list=None, pobs=None, sym=None, Bt=None, M=0,
                   F=None, hu=None, he=None, margin_min=1e-9, ignore_outliers=0):
    row0, ln, t0, TT = plan
    lst = None if chain_list is None else np.array(chain_list, dtype=np.int32)
    rows = int(row0[-1] + ln[-1])
    flagmap = np.full(rows, 0xdeadbeef, dtype=np.uint32)    # every row must be written
    rc = emu.panel_emu_viterbi_chain(C.c_int(N), C.c_int(em_kind), C.c_int(grid), ptr(row0, C.c_longlong), ptr(ln, C.c_int),
                                     ptr(t0, C.c_int), ptr(TT, C.c_int), ptr(lst, C.c_int),
                                     C.c_int(len(row0) if lst is None else len(lst)), C.c_int(warm), None, C.c_int(exact),
                                     ptr(pobs), None, ptr(sym, C.c_int), None, None, ptr(Bt), C.c_int(M),
                                     C.c_int(ignore_outliers), ptr(A), ptr(pi), F.ctypes.data_as(C.POINTER(C.c_ubyte)),
                                     ptr(hu), ptr(he), flagmap.ctypes.data_as(C.POINTER(C.c_uint)), C.c_double(margin_min))
    assert rc == 0
    return flagmap


@pytest.mark.parametrize('N', [32, 10, 3])
def test_time_chunked_viterbi_matches_sequential(emu, oracle_port, N):
    """k_viterbi_chain32: two trajectories cut into 15 chains that run in parallel after a warm-up reproduce the oracle's
    sequential Viterbi paths bit for bit, the hand-overs agree to rounding, and no decision is flagged as a near-tie."""
    rng = np.random.default_rng(50 + N)
    X = rng.random((N, N)) + 2.0 * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = rng.random(N)
    pi /= pi.sum()
    Ts = [400, 173]
    pobs = [np.ascontiguousarray(rng.random((T, N)) ** 3 + 1e-6) for T in Ts]
    cat = np.ascontiguousarray(np.vstack(pobs))
    plan = make_plan(Ts, 40)
    n = len(plan[0])
    assert n == 15
    F = np.full((cat.shape[0], N), 255, dtype=np.uint8)
    hu, he = np.zeros((n, N)), np.zeros((n, N))
    flagmap = _viterbi_chain(emu, N, EM_POBS, plan, A, pi, grid=2, warm=80, pobs=cat, F=F, hu=hu, he=he, margin_min=1e-11)
    assert not np.any(flagmap == 0xdeadbeef)                # every row of the map got its flag word
    row, paths = 0, []
    for T, p in zip(Ts, pobs):
        paths.append(_resolve(F[row:row + T], T))
        assert np.array_equal(paths[-1], oracle_port.viterbi(A, p, pi))
        row += T
    # no decision ON the resolved paths is a near-tie (k_viterbi_path_flags)
    path = np.ascontiguousarray(np.concatenate(paths), dtype=np.int32)
    offs = np.concatenate([[0], np.cumsum(Ts)]).astype(np.int64)
    assert emu.panel_emu_viterbi_path_flags(flagmap.ctypes.data_as(C.POINTER(C.c_uint)), path.ctypes.data_as(C.POINTER(C.c_int)),
                                            ptr(offs, C.c_longlong), len(Ts), C.c_longlong(len(path))) == 0
    # with an absurdly large threshold every decision is "near": one hit per row
    flag_all = _viterbi_chain(emu, N, EM_POBS, plan, A, pi, grid=2, warm=80, pobs=cat, F=F, hu=hu, he=he, margin_min=2.0)
    hits = emu.panel_emu_viterbi_path_flags(flag_all.ctypes.data_as(C.POINTER(C.c_uint)), path.ctypes.data_as(C.POINTER(C.c_int)),
                                            ptr(offs, C.c_longlong), len(Ts), C.c_longlong(len(path)))
    assert hits == (len(path) - len(Ts) if N > 1 else 0) + (len(Ts) if N > 1 else 0)
    t0 = plan[2]
    for c in range(n):
        if t0[c] > 0:
            np.testing.assert_allclose(hu[c], he[c - 1], rtol=1e-11, atol=1e-300)


def test_time_chunked_viterbi_fix_up_and_tie_flag(emu, oracle_port):
    """(1) A warm-up that is too short on a slowly mixing model leaves wrong hand-overs; exact passes over the failing chains,
    in order, repair the map.  (2) A model with structural ties is flagged (the caller then runs the sequential kernel)."""
    N = 8
    rng = np.random.default_rng(4)
    X = rng.random((N, N)) + 60.0 * np.eye(N)
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = np.ones(N) / N
    T = 240
    pobs = np.ascontiguousarray(0.3 + 0.7 * rng.random((T, N)))         # weakly informative: the start matters for long
    plan = make_plan([T], 30)
    n = len(plan[0])
    F = np.zeros((T, N), dtype=np.uint8)
    hu, he = np.zeros((n, N)), np.zeros((n, N))
    _viterbi_chain(emu, N, EM_POBS, plan, A, pi, grid=1, warm=1, pobs=pobs, F=F, hu=hu, he=he)
    bad = [c for c in range(1, n) if np.max(np.abs(hu[c] - he[c - 1]) / np.maximum(hu[c], he[c - 1])) > 1e-11]
    assert bad, 'the one-frame warm-up should have failed somewhere'
    while bad:                                              # certification loop: earliest failing chain first
        c = bad[0]
        _viterbi_chain(emu, N, EM_POBS, plan, A, pi, grid=1, warm=1, exact=1, chain_list=[c], pobs=pobs, F=F, hu=hu, he=he)
        bad = [k for k in range(1, n) if np.max(np.abs(hu[k] - he[k - 1]) / np.maximum(hu[k], he[k - 1])) > 1e-11]
    assert np.array_equal(_resolve(F, T), oracle_port.viterbi(A, pobs, pi))
    # (2) structural ties
    A1 = np.full((N, N), 1.0 / N)
    p1 = np.ascontiguousarray(np.tile(np.array([[0.5, 0.25] * (N // 2)]), (60, 1)))
    plan1 = make_plan([60], 20)
    F1 = np.zeros((60, N), dtype=np.uint8)
    h1, h2 = np.zeros((3, N)), np.zeros((3, N))
    fm = _viterbi_chain(emu, N, EM_POBS, plan1, A1, pi, grid=1, warm=10, pobs=p1, F=F1, hu=h1, he=h2)
    assert np.count_nonzero(fm) > 30                        # ties at (almost) every frame
