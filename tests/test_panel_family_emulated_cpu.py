"""The tensor-pipe ("panel") family as it ships for 17 <= N <= 104, executed on the CPU by tests/emu/warp_emu.h and compared
with a plain float64 forward-backward and with the oracle's Viterbi.  tests/emu/panel_emu.cpp dispatches like the launchers:
the one-set kernels at 4 state tiles (N <= 32), the two-set kernels k_forward_wide2 / k_backward_stats_wide2 at 8 and 13
tiles with the outlier machinery compiled in only when the rule is on, and k_viterbi_multi for the batched Viterbi.

Every tile occupancy: a last tile holding one state (17, 25, 33, 41, 65, 97), full tiles (24, 32, 40, 64, 72, 104), odd N
(every store on the scalar path), the most empty warps (3 at N = 33, 4 at N = 65).  Every chain layout of a block: chain
counts with n mod 16 in {0, 5, 8, 13} (second set full, empty, exactly empty, partial), grid = 1 (the persistent loop walks
3 or more rounds) and the launchers' grid (the last block partly idle), trajectories of 1 and 2 frames.  Every start: the
trajectory's pi, a uniform warm-up, a warm-up longer than the chain's offset (clipped to pi), per-chain warm-ups, exact
starts over a chain list.  Dynamic shared memory holds NaN at every launch and every output row NaN before it, so a word
read before it is written, or a row never written, fails the comparison.  What this cannot show: races between warps and
the named barriers of k_viterbi_multi's sub-blocks (nsub > 1), which tests/test_panel_family_cuda.py covers on the GPU.
"""
import ctypes as C

import numpy as np
import pytest

from test_panel_emulated_cpu import emu, gauss, make_plan, plain_estep, ptr, _resolve  # noqa: F401  (emu: fixture)

EM_POBS, EM_GAUSS, EM_DISC = 0, 1, 2
E_NS = (17, 24, 25, 31, 32, 33, 40, 41, 63, 64, 65, 72, 97, 103, 104)
# one N per occupancy class for the discrete and table emissions: NT = 4 odd with a one-state tile, NT = 8 with 3 empty warps,
# NT = 8 full, NT = 13 with 4 empty warps, NT = 13 odd, NT = 13 full
CLASS_NS = (25, 33, 64, 65, 103, 104)
LAYOUTS = (48, 37, 40, 45)                  # n mod 16 = 0, 5, 8, 13
CHUNK, WARM, M_SYM, NO_SYM = 6, 20, 11, 5     # chains start at t0 = 0, 6, ..., 30: warm-ups clipped to pi and real ones
V_NS = (33, 40, 64, 65, 100, 103, 104)


def ragged(n, rng):
    """trajectory lengths that cut into exactly n chains of CHUNK frames, among them trajectories of 1 and 2 frames"""
    Ts, left = [1, 2], n - 2
    while left > 0:
        k = min(left, int(rng.integers(1, 7)))
        Ts.append((k - 1) * CHUNK + int(rng.integers(1, CHUNK + 1)))
        left -= k
    rng.shuffle(Ts)
    return Ts


def wide_model(seed, N, mixing=1.0):
    rng = np.random.default_rng(seed)
    A = rng.random((N, N)) + mixing * np.eye(N)
    A /= A.sum(axis=1)[:, None]
    pi = rng.random(N)
    pi /= pi.sum()
    return rng, A, pi


class Problem(object):
    """trajectories of one emission kind, the kernels' inputs and the float64 reference"""

    def __init__(self, rng, N, kind, outl, Ts, A, pi):
        self.N, self.kind, self.outl, self.Ts, self.A, self.pi = N, kind, outl, Ts, A, pi
        self.mu, self.sigma = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
        self.obs = self.sym = self.Bt = self.pobs = None
        self.M = 0
        if kind == EM_GAUSS:
            trajs = [self.mu[rng.integers(0, N, T)] + 0.7 * rng.standard_normal(T) for T in Ts]
            if outl:                                        # far from every state: all densities underflow
                trajs[int(np.argmax(Ts))][3] = 400.0
            self.obs = np.concatenate(trajs)
            ps = [gauss(o[:, None], self.mu[None, :], self.sigma[None, :]) for o in trajs]
        elif kind == EM_DISC:
            B = rng.random((N, M_SYM)) ** 3 + 1e-4
            B[:, NO_SYM] = 0.0                              # a symbol no state emits
            B /= B.sum(axis=1)[:, None]
            syms = [rng.choice([m for m in range(M_SYM) if m != NO_SYM], T).astype(np.int32) for T in Ts]
            if outl:
                syms[int(np.argmax(Ts))][3] = NO_SYM
            self.sym = np.concatenate(syms)
            self.Bt = np.ascontiguousarray(B.T)
            self.M = M_SYM
            ps = [B[:, s].T.copy() for s in syms]
        else:
            ps = [rng.random((T, N)) ** 3 + 1e-3 for T in Ts]
            self.pobs = np.ascontiguousarray(np.vstack(ps))
        if kind != EM_POBS and outl:
            for p in ps:
                p[p.sum(axis=1) == 0] = 1.0                 # outputmodel.py:126-130
        assert kind == EM_POBS or outl == any((p == 1.0).all(axis=1).any() for p in ps)
        self.ref = plain_estep(ps, A, pi)
        self.plan = make_plan(Ts, CHUNK)
        self.rows = int(self.plan[0][-1] + self.plan[1][-1])
        n = len(self.plan[0])
        self.alpha = np.full((self.rows, N), np.nan)
        self.chain_ll = np.full(n, np.nan)
        self.hu_f, self.he_f, self.hu_b, self.he_b = (np.full((n, N), np.nan) for _ in range(4))

    def _em(self):
        return (ptr(self.pobs), ptr(self.obs), ptr(self.sym, C.c_int), ptr(self.mu), ptr(self.sigma), ptr(self.Bt),
                C.c_int(self.M), C.c_int(self.outl))

    def _chains(self, warm, warmv, exact, chain_list):
        row0, ln, t0, TT = self.plan
        self._lst = None if chain_list is None else np.array(chain_list, dtype=np.int32)
        self._wv = None if warmv is None else np.ascontiguousarray(warmv, dtype=np.int32)
        n_run = len(row0) if self._lst is None else len(self._lst)
        return (ptr(row0, C.c_longlong), ptr(ln, C.c_int), ptr(t0, C.c_int), ptr(TT, C.c_int), ptr(self._lst, C.c_int),
                C.c_int(n_run), C.c_int(warm), ptr(self._wv, C.c_int), C.c_int(exact))

    def forward(self, emu, grid, warm, warmv=None, exact=0, chain_list=None):
        rc = emu.panel_emu_forward(C.c_int(self.N), C.c_int(self.kind), C.c_int(grid),
                                   *self._chains(warm, warmv, exact, chain_list), *self._em(), ptr(self.A), ptr(self.pi),
                                   ptr(self.alpha), ptr(self.chain_ll), ptr(self.hu_f), ptr(self.he_f))
        assert rc == 0

    def backward(self, emu, grid, warm, alpha, warmv=None, exact=0, chain_list=None):
        N = self.N
        gamma = np.full((self.rows, N), np.nan)
        Bnum = np.zeros((N, self.M)) if self.kind == EM_DISC else None
        partials = np.full((grid, N * N + 4 * N), np.nan)  # one row per block, every row written
        rc = emu.panel_emu_backward_stats(C.c_int(N), C.c_int(self.kind), C.c_int(grid),
                                          *self._chains(warm, warmv, exact, chain_list), *self._em(), ptr(self.A),
                                          ptr(np.ascontiguousarray(alpha)), ptr(gamma), ptr(Bnum), ptr(partials),
                                          ptr(self.hu_b), ptr(self.he_b))
        assert rc == 0
        assert not np.isnan(partials).any()
        s = partials.sum(axis=0)
        return dict(gamma=gamma, Bnum=Bnum, C=self.A * s[:N * N].reshape(N, N), g0=s[N * N:N * N + N],
                    sg=s[N * N + N:N * N + 2 * N], sgd=s[N * N + 2 * N:N * N + 3 * N], sgdd=s[N * N + 3 * N:])

    # ---- comparisons with the float64 reference
    def check_forward(self):
        ref, (row0, ln, t0, TT) = self.ref, self.plan
        np.testing.assert_allclose(self.alpha, ref['alpha'], rtol=1e-10, atol=1e-300)
        want = np.array([ref['lc'][row0[c]:row0[c] + ln[c]].sum() for c in range(len(row0))])
        np.testing.assert_allclose(self.chain_ll, want, rtol=1e-10, atol=1e-12)
        for c in range(len(row0)):
            np.testing.assert_allclose(self.he_f[c], ref['alpha'][row0[c] + ln[c] - 1], rtol=1e-10, atol=1e-300)
            if t0[c] > 0:
                np.testing.assert_allclose(self.hu_f[c], ref['alpha'][row0[c] - 1], rtol=1e-10, atol=1e-300)

    def check_backward(self, st):
        ref, (row0, ln, t0, TT), N = self.ref, self.plan, self.N
        np.testing.assert_allclose(st['gamma'], ref['gamma'], rtol=1e-10, atol=1e-300)
        np.testing.assert_allclose(st['C'], ref['C'], rtol=1e-9, atol=1e-300)
        np.testing.assert_allclose(st['g0'], ref['g0'], rtol=1e-10, atol=1e-300)
        np.testing.assert_allclose(st['sg'], ref['gamma'].sum(axis=0), rtol=1e-10)
        assert abs(st['C'].sum() - (sum(self.Ts) - len(self.Ts))) < 1e-9 * sum(self.Ts)
        if self.kind == EM_GAUSS:
            d = self.obs[:, None] - self.mu[None, :]
            g = ref['gamma']
            np.testing.assert_allclose(st['sgd'], (g * d).sum(axis=0), rtol=1e-9, atol=1e-12 * (g * np.abs(d)).sum())
            np.testing.assert_allclose(st['sgdd'], (g * d * d).sum(axis=0), rtol=1e-9)
        if self.kind == EM_DISC:
            want = np.zeros((N, self.M))
            np.add.at(want.T, self.sym, ref['gamma'])
            np.testing.assert_allclose(st['Bnum'], want, rtol=1e-9, atol=1e-14)
        for c in range(len(row0)):
            if t0[c] > 0:
                np.testing.assert_allclose(self.he_b[c], ref['beta'][row0[c]], rtol=1e-10, atol=1e-300)
            if t0[c] + ln[c] < TT[c]:
                np.testing.assert_allclose(self.hu_b[c], ref['beta'][row0[c] + ln[c]], rtol=1e-10, atol=1e-300)


@pytest.fixture
def wide_mode(emu):
    """N = 32 runs on the wide kernels (BHMM_B200_PANEL=2) for the test"""
    emu.panel_emu_force_wide(1)
    yield
    emu.panel_emu_force_wide(0)


def run_estep(emu, N, kind, outl, n, seed, one_first):
    """forward and backward + statistics, one of them on a single block (one_first: the forward), the other on the
    launchers' grid"""
    rng, A, pi = wide_model(seed, N)
    Ts = ragged(n, rng)
    pb = Problem(rng, N, kind, outl, Ts, A, pi)
    assert len(pb.plan[0]) == n
    cpb, cpb_bwd = emu.panel_emu_wide_cpb(N), emu.panel_emu_wide_cpb_bwd(N)
    assert (cpb, cpb_bwd) == ((8, 8) if N <= 32 else ((16, 16) if N <= 64 else (16, 8)))
    assert n > 2 * cpb                                      # grid = 1: three rounds or more
    assert 0 < (pb.plan[2] > WARM).sum() < (pb.plan[2] > 0).sum()
    grid_f, grid_b = (1, -(-n // cpb_bwd)) if one_first else (-(-n // cpb), 1)
    pb.forward(emu, grid_f, WARM)
    pb.check_forward()
    st = pb.backward(emu, grid_b, WARM, pb.alpha)
    pb.check_backward(st)


@pytest.mark.parametrize('outl', [1, 0])
@pytest.mark.parametrize('N', E_NS)
def test_gaussian_estep_every_tile_occupancy(emu, wide_mode, N, outl):
    """Gaussian E-step with the outlier rule on (a frame where every density underflows) and off (OUTL = false on wide2)"""
    i = E_NS.index(N)
    run_estep(emu, N, EM_GAUSS, outl, LAYOUTS[(i + 2 * outl) % 4], 1000 + 10 * N + outl, outl == 1)


@pytest.mark.parametrize('kind,outl', [(EM_DISC, 0), (EM_DISC, 1), (EM_POBS, 0)])
@pytest.mark.parametrize('N', CLASS_NS)
def test_discrete_and_table_estep_per_occupancy_class(emu, N, kind, outl):
    """discrete symbols with the rule off, with the rule on and a symbol no state emits, and the caller's p_obs table"""
    i = CLASS_NS.index(N) + kind + outl
    run_estep(emu, N, kind, outl, LAYOUTS[i % 4], 2000 + 10 * N + 3 * kind + outl, i % 2 == 0)


@pytest.mark.parametrize('N', [25, 41, 65])
def test_start_modes_and_exact_fix_up(emu, N):
    """(1) Per-chain warm-ups (warmv) of WARM frames, or reaching past the trajectory's start (forward) or end (backward), are
    exact where the scalar warm-up of one frame is not.  (2) On a slowly mixing model a warm-up of 2 frames fails in both directions; exact starts over chain lists, each
    chain after the one it starts from (forward in order, backward in reverse), repair every output and hand-over, and one
    exact pass over the list of all interior chains then leaves them unchanged."""
    rng, A, pi = wide_model(3000 + N, N)
    Ts = [57, 1, 34, 2, 61, 25, 48, 9, 40]
    pb = Problem(rng, N, EM_GAUSS, 1, Ts, A, pi)
    row0, ln, t0, TT = pb.plan
    n = len(row0)
    cpb = emu.panel_emu_wide_cpb(N)
    # a real warm-up of WARM frames where the chain starts later than that, else one that reaches back to the start
    pb.forward(emu, 2, 1, warmv=np.where(t0 > WARM, WARM, t0 + rng.integers(0, 3, n)))
    pb.check_forward()
    rest = TT - (t0 + ln)
    st = pb.backward(emu, 2, 1, pb.alpha, warmv=np.where(rest > WARM, WARM, rest + rng.integers(0, 3, n)))
    pb.check_backward(st)
    pb.forward(emu, 2, 1)
    assert np.max(np.abs(pb.alpha - pb.ref['alpha'])) > 1e-6   # the warm-up of one frame alone does not forget

    rng, A, pi = wide_model(3100 + N, N, mixing=40.0)
    pb = Problem(rng, N, EM_GAUSS, 0, Ts, A, pi)
    pb.forward(emu, 1, 2)
    assert np.max(np.abs(pb.alpha - pb.ref['alpha'])) > 1e-6
    interior = [c for c in range(n) if t0[c] > 0]
    for c in interior:
        pb.forward(emu, 1, 2, exact=1, chain_list=[c])
    pb.check_forward()
    st = pb.backward(emu, 1, 2, pb.ref['alpha'])
    assert np.max(np.abs(st['gamma'] - pb.ref['gamma'])) > 1e-6
    for c in reversed([c for c in range(n) if t0[c] + ln[c] < TT[c]]):
        pb.backward(emu, 1, 2, pb.ref['alpha'], exact=1, chain_list=[c])
    st = pb.backward(emu, -(-n // emu.panel_emu_wide_cpb_bwd(N)), 2, pb.ref['alpha'], exact=1)
    pb.check_backward(st)
    assert len(interior) > cpb                              # both chain sets of a block, more than one round at grid = 1
    pb.alpha[:] = np.nan
    pb.forward(emu, 1, 2, exact=1, chain_list=interior)
    first = [c for c in range(n) if t0[c] == 0]
    pb.forward(emu, 1, 2, chain_list=first)
    pb.check_forward()


def test_unsupported_state_counts(emu):
    """N <= 16 belongs to the lane family, N > 104 to the team kernels; the batched Viterbi starts above 32"""
    for N in (16, 105):
        args = (C.c_int(N), C.c_int(EM_POBS), C.c_int(1)) + (None,) * 5 + (C.c_int(0), C.c_int(0), None, C.c_int(0)) + \
               (None,) * 6 + (C.c_int(0), C.c_int(0))
        assert emu.panel_emu_forward(*args, *(None,) * 6) == 2
        assert emu.panel_emu_backward_stats(*args, *(None,) * 7) == 2
        assert emu.panel_emu_wide_cpb(N) == 0 and emu.panel_emu_wide_cpb_bwd(N) == 0
    for N in (32, 105):
        assert emu.panel_emu_viterbi_multi(C.c_int(N), C.c_int(EM_POBS), C.c_int(1), C.c_int(0), *(None,) * 7,
                                           C.c_int(0), C.c_int(0), None, None, None) == 2


# ------------------------------------------------------------------------------------------------ k_viterbi_multi
def viterbi_multi(emu, N, kind, grid, Ts, A, pi, pobs=None, obs=None, sym=None, mu=None, sigma=None, Bt=None, M=0, outl=0):
    offsets = np.concatenate([[0], np.cumsum(Ts)]).astype(np.int64)
    F = np.full((int(offsets[-1]), N), 255, dtype=np.uint8)
    rc = emu.panel_emu_viterbi_multi(C.c_int(N), C.c_int(kind), C.c_int(grid), C.c_int(len(Ts)), ptr(offsets, C.c_longlong),
                                     ptr(pobs), ptr(obs), ptr(sym, C.c_int), ptr(mu), ptr(sigma), ptr(Bt), C.c_int(M),
                                     C.c_int(outl), ptr(np.ascontiguousarray(A)), ptr(pi),
                                     F.ctypes.data_as(C.POINTER(C.c_ubyte)))
    assert rc == 0
    assert F.max() < N                                      # every entry of the map written
    return [_resolve(F[offsets[k]:offsets[k + 1]], T) for k, T in enumerate(Ts)]


@pytest.mark.parametrize('N', V_NS)
def test_viterbi_multi_is_bit_exact(emu, oracle_port, N):
    """k_viterbi_multi (A in shared memory, R = 4 trajectories per group in lock step, two predecessors per scan step, odd N
    on the single-predecessor tail) against the oracle's _compute_viterbi: identical paths for K = 1, 3, 4, 5, 9 (groups
    partly filled, several rounds at grid = 1), trajectories of 1 and 2 frames, the three emission kinds with the outlier
    rule, a tie-heavy model, and a rank-one model whose states have exact twins across the scan."""
    R = emu.panel_emu_viterbi_multi_r()
    assert R == 4
    rng = np.random.default_rng(700 + N)
    X = rng.integers(1, 4, size=(N, N)).astype(float) + 6.0 * np.eye(N)    # small integers: many exactly equal products
    A = np.ascontiguousarray(X / X.sum(axis=1)[:, None])
    pi = np.ones(N) / N
    B = rng.integers(0, 3, size=(N, 9)).astype(float)
    B[:, 4] = 0.0                                           # no state emits symbol 4
    B[:, 0] += 1.0
    B /= B.sum(axis=1)[:, None]
    mu, sigma = np.linspace(-5, 5, N), np.linspace(0.5, 2.0, N)
    for K, grid in ((9, 1), (5, 2), (4, 1), (3, 1), (1, 1)):
        Ts = [int(t) for t in rng.integers(3, 40, K)]
        Ts[0] = 1
        if K > 1:
            Ts[-1] = 2
        # discrete, outlier rule on, a frame with symbol 4
        syms = [rng.integers(0, 9, T).astype(np.int32) for T in Ts]
        syms[-1][-1] = 4
        got = viterbi_multi(emu, N, EM_DISC, grid, Ts, A, pi, sym=np.concatenate(syms), Bt=np.ascontiguousarray(B.T), M=9,
                            outl=1)
        for k in range(K):
            assert np.array_equal(got[k], oracle_port.viterbi(A, oracle_port.discrete_p_obs(syms[k], B, True), pi)), (K, k)
        # Gaussian, outlier rule on (a frame far from every state) and off
        for outl in (1, 0):
            trajs = [mu[rng.integers(0, N, T)] + 0.7 * rng.standard_normal(T) for T in Ts]
            if outl:
                trajs[-1][-1] = 400.0
            got = viterbi_multi(emu, N, EM_GAUSS, grid, Ts, A, pi, obs=np.concatenate(trajs), mu=mu, sigma=sigma, outl=outl)
            for k in range(K):
                want = oracle_port.viterbi(A, oracle_port.gaussian_p_obs(trajs[k], mu, sigma, bool(outl)), pi)
                assert np.array_equal(got[k], want), (K, k, outl)
        # the caller's table
        ps = [rng.random((T, N)) ** 4 for T in Ts]
        got = viterbi_multi(emu, N, EM_POBS, grid, Ts, A, pi, pobs=np.ascontiguousarray(np.vstack(ps)))
        for k in range(K):
            assert np.array_equal(got[k], oracle_port.viterbi(A, ps[k], pi)), (K, k)
    # structural ties ACROSS the scan: a rank-one transition matrix and emission rows that repeat with period 3, so every
    # state has N/3 exact twins and only the first-maximum rule decides
    A1 = np.full((N, N), 1.0 / N)
    B1 = np.array([[0.5, 0.25, 0.25], [0.25, 0.5, 0.25], [0.125, 0.125, 0.75]])[np.arange(N) % 3]
    Ts = [50, 1, 31, 2, 17]
    syms = [rng.integers(0, 3, T).astype(np.int32) for T in Ts]
    got = viterbi_multi(emu, N, EM_DISC, 1, Ts, A1, pi, sym=np.concatenate(syms), Bt=np.ascontiguousarray(B1.T), M=3)
    for k in range(len(Ts)):
        want = oracle_port.viterbi(A1, oracle_port.discrete_p_obs(syms[k], B1), pi)
        assert np.array_equal(got[k], want)
        assert want.max() <= 2                              # always the FIRST of the twins
