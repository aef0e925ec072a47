"""Host checks of the float64 references and error bounds in tests/helpers/policy_reference.py (no GPU): the vectorised
Philox is the scalar spec, and each bound holds for a float32 emulation of its kernel's arithmetic while it rejects
the same emulation with one term missing -- a bound that cannot tell those apart is too loose to test a kernel with."""
import numpy as np
import pytest

from tests.helpers import policy_reference as P


def test_vectorised_philox_equals_the_scalar_spec():
    rng = np.random.Generator(np.random.PCG64(1))
    quads = [0, 1, 2 ** 32 - 1, 2 ** 32, 2 ** 34 + 2, 2 ** 64 - 1] + [int(q) for q in rng.integers(0, 2 ** 63, 10)]
    steps = [0, 7, 2 ** 32 - 1, 2 ** 32, 2 ** 33 + 5, 2 ** 64 - 1] + [int(s) for s in rng.integers(0, 2 ** 63, 10)]
    for seed in (0, 543, 2 ** 32 + 17, 2 ** 64 - 1):
        got = P.philox4_np(seed, np.array(quads, dtype=np.uint64)[:, None], np.array(steps, dtype=np.uint64)[None, :])
        assert got.shape == (4, len(quads), len(steps)) and got.dtype == np.uint32
        for i, q in enumerate(quads):
            for j, s in enumerate(steps):
                assert got[:, i, j].tolist() == P.philox4(seed, q, s), (seed, q, s)
    # sample_bits: key seed ^ 0x5A4D504C45, counter (env >> 2, step), word env & 3
    envs = np.array([0, 1, 2, 3, 4, 5, 2 ** 34 + 8, 2 ** 34 + 11, 2 ** 40 + 3], dtype=np.uint64)
    for step in (0, 2 ** 32 - 1, 2 ** 32):
        bits = P.sample_bits(11, envs, step)
        for g, b in zip(envs.tolist(), bits.tolist()):
            assert b == P.philox4(11 ^ 0x5A4D504C45, g >> 2, step)[g & 3]


def _planes_like(rng, n, cells, n_chars):
    """0/1 inputs shaped like a layered board: exactly one channel set per cell (Hello World: 7 x 468 inputs)."""
    x = np.zeros((n, n_chars, cells), dtype=np.float32)
    k = rng.integers(0, n_chars, (n, cells))
    x[np.arange(n)[:, None], k, np.arange(cells)[None, :]] = 1.0
    return x.reshape(n, -1)


@pytest.mark.parametrize("case", ["dense_175", "planes_3276"])
def test_logit_bound_holds_for_the_kernel_arithmetic_and_rejects_a_missing_term(case):
    rng = np.random.Generator(np.random.PCG64(2))
    n, A = 256, 5
    if case == "dense_175":
        n_in, n_hidden = 175, 17
        x = rng.normal(0.0, 1.0, (n, n_in)).astype(np.float32)
    else:
        n_in, n_hidden = 3276, 32
        x = _planes_like(rng, n, 468, 7)
    w = P.policy_weights(rng, n_in, n_hidden, A, fan_in=np.count_nonzero(x[0]))
    want, mag = P.mlp_logits(x, *w)
    bound = P.logit_bound(x, n_hidden, mag)
    err = np.abs(P.mlp_logits_f32(x, *w) - want)
    assert (err <= bound).all(), float((err / bound).max())
    assert float((err / bound).max()) > 1e-4                  # the emulation does round: the check is not vacuous
    # one input term dropped: out of bound in nearly every row (a dropped term can be small by chance)
    miss = (np.abs(P.mlp_logits_f32(x, *w, skip_last_input=True) - want) > bound).any(axis=1)
    assert miss.mean() > 0.9, miss.mean()
    # no output bias: out of bound in every row
    assert (np.abs(P.mlp_logits_f32(x, *w, skip_b2=True) - want) > bound).any(axis=1).all()


def _sample_f32(p, bits, shift=8):
    """sample_categorical_bits (cx_policy.cuh) on probabilities in numpy float32 (exact emulation: every operation is a
    correctly rounded float32 add, multiply or compare); shift = 9 is a defect the draw check must expose."""
    p = np.asarray(p, dtype=np.float32)
    n, A = p.shape
    w = np.where(p > 0, p, np.float32(0))
    total = np.zeros(n, dtype=np.float32)
    for a in range(A):
        total = (total + w[:, a]).astype(np.float32)
    u = ((bits >> np.uint32(shift)).astype(np.float32) * np.float32(1.0 / 16777216.0)).astype(np.float32) * total
    pick, cum, found = np.full(n, A - 1), np.zeros(n, dtype=np.float32), np.zeros(n, dtype=bool)
    for a in range(A):
        cum = (cum + w[:, a]).astype(np.float32)
        hit = ~found & (u < cum)
        pick[hit], found = a, found | hit
    for a in range(A - 1, 0, -1):
        pick[(pick == a) & ~(w[:, a] > 0)] = a - 1
    return pick


def test_draw_check_passes_the_sampler_arithmetic_and_rejects_a_wrong_uniform():
    rng = np.random.Generator(np.random.PCG64(3))
    n, A = 1 << 16, 5
    p = rng.random((n, A)).astype(np.float32)
    p[rng.random((n, A)) < 0.2] = 0.0                         # zero-probability actions are never drawn
    p[:, 0] = np.maximum(p[:, 0], np.float32(1e-3))
    bits = P.sample_bits(5, np.arange(n), 2 ** 32 - 1)
    w, err = P.weights_of(p, False)
    measure, observed = P.check_draws(_sample_f32(p, bits), w, err, bits)
    assert measure < 1e-4 and observed < 1e-3
    with pytest.raises(AssertionError):
        P.check_draws(_sample_f32(p, bits, shift=9), w, err, bits)


def test_returns_bound_holds_for_the_kernel_arithmetic_and_rejects_an_uncut_return():
    rng = np.random.Generator(np.random.PCG64(4))
    T, n, gamma = 300, 64, 0.999
    r = (np.where(rng.random((T, n)) < 0.5, -1.0, 1.0) * 10.0 ** rng.uniform(-3, 3, (T, n))).astype(np.float32)
    d = rng.random((T, n)).astype(np.float32)
    f = np.where(rng.random((T, n)) < 0.02, P.TRUNCATED, 0).astype(np.uint8)
    boot = rng.normal(0, 100, n).astype(np.float32)
    want, mag = P.returns64(r, f, gamma, d, boot)
    bound = P.returns_bound(mag)

    def kernel(cut):
        g, out = boot.copy(), np.empty((T, n), dtype=np.float32)
        for t in range(T - 1, -1, -1):
            c = np.where((f[t] & cut) != 0, np.float32(0), d[t])
            gc = (np.float32(gamma) * c).astype(np.float32)
            g = (gc.astype(np.float64) * g + r[t]).astype(np.float32)       # fmaf: one rounding
            out[t] = g
        return out

    assert (np.abs(kernel(P.TERMINATED | P.TRUNCATED) - want) <= bound).all()
    assert (np.abs(kernel(P.TERMINATED) - want) > bound).any()


def test_chi2_survival_function():
    # 5 % and 1e-6 quantiles of chi-square with 1 .. 7 degrees of freedom
    for dof, q05, q1e6 in [(1, 3.8414588206941285, 23.928126976934827), (2, 5.991464547107983, 27.631021115928547),
                           (4, 9.487729036781158, 33.37684158171984), (7, 14.067140449340167, 40.521831234179864)]:
        assert abs(P.chi2_sf(q05, dof) - 0.05) < 1e-12
        assert abs(P.chi2_sf(q1e6, dof) / 1e-6 - 1.0) < 1e-9
