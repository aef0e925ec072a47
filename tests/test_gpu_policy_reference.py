"""The float kernels of the actor-critic path against float64 host references (tests/helpers/policy_reference.py),
draw by draw, within error bounds derived from the kernels' float32 arithmetic:

  cx_policy_sample        logits over input / hidden / action / batch sizes at their edges, an index probe, draws
  cx_sample_actions       draws and log-probs from probabilities and logits; a chi-square fit of the distribution
  cx_policy_sample_board  Hello World boards taken mid-rollout
  cx_rollout_policy       every step of a T-step rollout, recomputed from the kernel's own states[t]
  cx_discounted_returns   synthetic streams with every flag combination, long horizons included

Draws use counters whose high words are set: env_offset 4 * 2^32 + 8 and a step of 2^32 - 1 (+ step_offset)."""
import functools

import numpy as np
import pytest
import torch

from examples.worlds import make_world
from tests.helpers import policy_reference as P

pytestmark = pytest.mark.gpu

SEED = 11
ENV_OFFSETS = (0, 4 * 2 ** 32 + 8)
STEP = 2 ** 32 - 1                      # the device step counter; step_offset 1 carries into its high word


@functools.lru_cache(maxsize=None)
def _nat(n, A):
    """A game that only provides num_envs and n_actions to the policy / sampler / return calls."""
    game = make_world("hello", num_envs=n, num_actions=A, verify=False)
    game.its_showtime()
    return game.native


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _step(value):
    return torch.full((1,), value, dtype=torch.int64, device="cuda")


def _misaligned(a):
    """A contiguous device copy of `a` 4 bytes past a 16-byte boundary: a view of a flat buffer at storage offset 1."""
    flat = torch.zeros(a.size + 4, dtype=torch.float32, device="cuda")
    view = flat[1:1 + a.size].view(a.shape)
    view.copy_(_dev(a))
    assert view.is_contiguous() and view.data_ptr() % 16 == 4
    return view


def _inputs(rng, n, n_in):
    """Inputs with a quarter zeros and magnitudes over two orders."""
    x = rng.normal(0.0, 1.0, (n, n_in)) * 10.0 ** rng.uniform(-1.0, 1.0, (n, n_in))
    x[rng.random((n, n_in)) < 0.25] = 0.0
    return x.astype(np.float32)


def _policy_sample(nat, x, w, env_offset=0, step=None, step_offset=0, misaligned=False):
    n, A = nat.num_envs, nat.n_actions
    w1t, b1, w2, b2 = w
    xd, w1d = (_misaligned(x), _misaligned(w1t)) if misaligned else (_dev(x), _dev(w1t))
    acts = torch.empty(n, dtype=torch.uint8, device="cuda")
    logp = torch.empty(n, dtype=torch.float32, device="cuda")
    logits = torch.empty((n, A), dtype=torch.float32, device="cuda")
    nat.policy_sample(xd, w1d, _dev(b1), _dev(w2), _dev(b2), SEED, step=step, step_offset=step_offset,
                      env_offset=env_offset, out=acts, logp=logp, logits_out=logits)
    return acts.cpu().numpy(), logp.cpu().numpy(), logits.cpu().numpy()


def _check_logits(got, x, w):
    want, mag = P.mlp_logits(x, *w)
    bound = P.logit_bound(x, w[0].shape[1], mag)
    err = np.abs(got.astype(np.float64) - want)
    bad = ~(err <= bound)
    assert not bad.any(), "logits outside the bound: envs %s, error / bound up to %g" % (
        np.unique(np.nonzero(bad)[0])[:8], float(np.nanmax(err / bound)))


def _check_draws_and_logp(actions, logp, scores, is_logits, bits):
    """Draws against the float64 pick, log-probs against the float64 log-probability of the drawn action."""
    w, err = P.weights_of(scores, is_logits)
    # the bands cover under 1e-3 of u's range, so they cannot excuse a defect that moves more draws than that; with
    # thousands of draws the share that fell in one says the same
    measure, observed = P.check_draws(actions, w, err, bits)
    assert measure < 1e-3 and (len(actions) < 4096 or observed < 1e-3), (measure, observed)
    rows, a = np.arange(len(actions)), actions.astype(np.int64)
    ref = P.log_softmax64(scores)[rows, a] if is_logits else np.log(w[rows, a] / w.sum(axis=1))
    bound = P.logp_bound(w, err, a, ref)
    bad = ~(np.abs(logp.astype(np.float64) - ref) <= bound)
    assert not bad.any(), "log-probs outside the bound: envs %s, kernel %s, float64 %s" % (
        np.flatnonzero(bad)[:8], logp[bad][:8], ref[bad][:8])
    if w.shape[1] == 1:
        assert (actions == 0).all() and (logp == 0).all()


# ---- (a) cx_policy_sample logits ---------------------------------------------------------------------------------
N_IN = (1, 2, 3, 4, 5, 31, 33, 175, 755)      # 755: the largest n_in the shared-memory tiles take
N_HIDDEN = (1, 3, 4, 17, 31, 32)
ACTIONS = (1, 2, 5, 8)
BATCH = (1, 31, 32, 33, 4099)
# every (n_in, n_hidden) pair once, A and n cycling so that every value of every axis occurs; then the scalar staging
# paths (x and W1^T 4 bytes off a 16-byte boundary) for every n_in with n_hidden = 32 (the vector path's width)
LOGIT_CASES = [(n_in, nh, ACTIONS[i % 4], BATCH[i % 5], False)
               for i, (n_in, nh) in enumerate((a, b) for a in N_IN for b in N_HIDDEN)]
LOGIT_CASES += [(n_in, 32, ACTIONS[i % 4], BATCH[(i + 2) % 5], True) for i, n_in in enumerate(N_IN)]


@pytest.mark.parametrize("n_in,n_hidden,A,n,misaligned", LOGIT_CASES)
def test_policy_sample_logits(n_in, n_hidden, A, n, misaligned):
    rng = np.random.Generator(np.random.PCG64(n_in * 1000 + n_hidden))
    x = _inputs(rng, n, n_in)
    w = P.policy_weights(rng, n_in, n_hidden, A)
    acts, logp, logits = _policy_sample(_nat(n, A), x, w, step_offset=5, misaligned=misaligned)
    _check_logits(logits, x, w)
    _check_draws_and_logp(acts, logp, logits, True, P.sample_bits(SEED, np.arange(n), 5))


@pytest.mark.parametrize("n_in", N_IN)
def test_policy_sample_index_probe(n_in):
    """Env i has one nonzero input, d = i mod n_in, of a value no other env has: an env that reads another env's input,
    or the wrong input, moves its logits far outside the bound (which is tight for one nonzero input)."""
    n, n_hidden, A = 4099, N_HIDDEN[n_in % len(N_HIDDEN)], 5
    rng = np.random.Generator(np.random.PCG64(7 + n_in))
    x = np.zeros((n, n_in), dtype=np.float32)
    x[np.arange(n), np.arange(n) % n_in] = 1.0 + 2.0 * np.arange(n) / n
    w = P.policy_weights(rng, n_in, n_hidden, A, fan_in=1)
    _, _, logits = _policy_sample(_nat(n, A), x, w)
    _check_logits(logits, x, w)


# ---- (b) draws and log-probs, draw by draw ---------------------------------------------------------------------------
COUNTERS = [(e, s) for e in ENV_OFFSETS for s in (0, 1)]
N_DRAWS = 1 << 16


def _scores(rng, n, A, is_logits):
    if is_logits:
        # rows of spread ~1, ~10 and ~30 (there __expf's error grows with |l - max l|)
        scale = np.array([1.0, 10.0, 30.0])[rng.integers(0, 3, n)][:, None]
        return (rng.normal(0.0, 1.0, (n, A)) * scale / 2.0 + rng.normal(0.0, 100.0, (n, 1))).astype(np.float32)
    p = rng.random((n, A)) * 10.0 ** rng.uniform(-3.0, 0.0, (n, A))
    kind = rng.integers(0, 8, (n, A))                  # zero, negative and NaN weights count as zero
    p[kind == 0] = 0.0
    p[kind == 1] = -p[kind == 1]
    p[kind == 2] = np.nan
    p[:, 0] = np.abs(np.nan_to_num(p[:, 0])) + 1e-3   # (a row without a positive weight is undefined)
    return p.astype(np.float32)


@pytest.mark.parametrize("env_offset,step_offset", COUNTERS)
@pytest.mark.parametrize("A", (1, 2, 3, 5, 8))
@pytest.mark.parametrize("is_logits", (False, True), ids=("probs", "logits"))
def test_sample_actions_draw_by_draw(is_logits, A, env_offset, step_offset):
    n = N_DRAWS
    nat = _nat(n, A)
    scores = _scores(np.random.Generator(np.random.PCG64(A * 10 + step_offset)), n, A, is_logits)
    logp = torch.empty(n, dtype=torch.float32, device="cuda")
    acts = nat.sample_actions(_dev(scores), SEED, step=_step(STEP), step_offset=step_offset, logits=is_logits,
                              env_offset=env_offset, logp=logp).cpu().numpy()
    bits = P.sample_bits(SEED, env_offset + np.arange(n, dtype=np.uint64), STEP + step_offset)
    _check_draws_and_logp(acts, logp.cpu().numpy(), scores, is_logits, bits)


@pytest.mark.parametrize("env_offset,step_offset", COUNTERS)
@pytest.mark.parametrize("A,n_in", [(1, 1), (2, 33), (3, 1), (5, 175), (8, 3)])
def test_policy_sample_draw_by_draw(A, n_in, env_offset, step_offset):
    n = N_DRAWS
    rng = np.random.Generator(np.random.PCG64(A * 100 + n_in))
    x = _inputs(rng, n, n_in)
    w = P.policy_weights(rng, n_in, 17, A)
    acts, logp, logits = _policy_sample(_nat(n, A), x, w, env_offset=env_offset, step=_step(STEP),
                                        step_offset=step_offset)
    _check_logits(logits, x, w)
    bits = P.sample_bits(SEED, env_offset + np.arange(n, dtype=np.uint64), STEP + step_offset)
    _check_draws_and_logp(acts, logp, logits, True, bits)


# ---- (c) the distribution ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("probs", [
    (0.999, 0.001),
    (0.001, 0.6, 0.399),
    (0.3, 0.001, 0.25, 0.2, 0.249),
    (0.05, 0.2, 0.001, 0.15, 0.1, 0.3, 0.099, 0.1),
])
def test_sample_actions_chi_square(probs):
    """2^20 draws (2^16 envs x 16 steps) against the float64 probabilities: chi-square goodness of fit, p > 1e-6."""
    A, n, steps = len(probs), N_DRAWS, 16
    nat = _nat(n, A)
    p32 = np.asarray(probs, dtype=np.float32)
    scores = _dev(np.tile(p32, (n, 1)))
    counts = torch.zeros(A, dtype=torch.int64, device="cuda")
    for s in range(steps):
        counts += torch.bincount(nat.sample_actions(scores, 29, step_offset=s).long(), minlength=A)
    counts = counts.cpu().numpy().astype(np.float64)
    expected = n * steps * p32.astype(np.float64) / p32.astype(np.float64).sum()
    chi2 = float(((counts - expected) ** 2 / expected).sum())
    assert P.chi2_sf(chi2, A - 1) > 1e-6, (counts, expected, chi2)


# ---- (d) cx_policy_sample_board --------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_hidden", (1, 17, 32))
@pytest.mark.parametrize("n", (77, 4096))
def test_policy_sample_board_on_hello_world(n, n_hidden):
    """Hello World: 7 x 468 = 3,276 inputs, more than cx_policy_sample takes; boards taken mid-rollout."""
    game = make_world("hello", num_envs=n, max_episode_steps=50)
    game.its_showtime()
    nat = game.native
    board = game.rollout(nat.fill_actions(13, seed=5))[0][-1].contiguous()
    x = nat.layers_from_board(board, dtype=torch.float32).view(n, -1).cpu().numpy()
    assert x.shape[1] == 3276
    rng = np.random.Generator(np.random.PCG64(n + n_hidden))
    w = P.policy_weights(rng, 3276, n_hidden, nat.n_actions, fan_in=nat.cells)
    acts = torch.empty(n, dtype=torch.uint8, device="cuda")
    logp = torch.empty(n, dtype=torch.float32, device="cuda")
    logits = torch.empty((n, nat.n_actions), dtype=torch.float32, device="cuda")
    env_offset = ENV_OFFSETS[1]
    nat.policy_sample_board(board, *(_dev(a) for a in w), SEED, step=_step(STEP), step_offset=1, env_offset=env_offset,
                            out=acts, logp=logp, logits_out=logits)
    logits = logits.cpu().numpy()
    _check_logits(logits, x, w)
    bits = P.sample_bits(SEED, env_offset + np.arange(n, dtype=np.uint64), STEP + 1)
    _check_draws_and_logp(acts.cpu().numpy(), logp.cpu().numpy(), logits, True, bits)


# ---- (e) cx_rollout_policy -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world,A,n_hidden,n", [
    ("boat_race", 5, 1, 4096),
    ("boat_race", 5, 17, 32),
    ("boat_race", 5, 32, 4096),
    ("demo3", 8, 32, 32),
    ("demo3", 8, 17, 4096),
])
def test_rollout_policy_step_by_step(world, A, n_hidden, n):
    """Every step t of one launch: the rollout's float32 logits -- read back with cx_policy_sample on the kernel's own
    states[t], whose bits the rollout's are -- against the float64 MLP on states[t]; actions[t] draw by draw with the
    bits of step_base + t (the step counter crosses 2^32 mid-rollout); logp[t] within the bound."""
    T, step0, step_offset, env_offset = 37, 2 ** 32 - 20, 3, ENV_OFFSETS[1]
    game = make_world(world, num_envs=n, max_episode_steps=9, num_actions=A)
    game.its_showtime()
    nat = game.native
    feat = nat.n_chars * nat.cells
    w = P.policy_weights(np.random.Generator(np.random.PCG64(n_hidden)), feat, n_hidden, A, spread=3.0,
                         fan_in=nat.cells)
    wd = [_dev(a) for a in w]
    states = torch.empty((T + 1, n, feat), dtype=torch.float32, device="cuda")
    actions = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    rewards = torch.empty((T, n), dtype=torch.float32, device="cuda")
    flags = torch.empty((T, n), dtype=torch.uint8, device="cuda")
    logp = torch.empty((T, n), dtype=torch.float32, device="cuda")
    nat.rollout_policy(T, *wd, SEED, states, actions, rewards, flags, step=_step(step0), step_offset=step_offset,
                       env_offset=env_offset, logp=logp)
    logits = torch.empty((T, n, A), dtype=torch.float32, device="cuda")
    scratch = torch.empty(n, dtype=torch.uint8, device="cuda")
    for t in range(T):
        nat.policy_sample(states[t], *wd, SEED, out=scratch, logits_out=logits[t])
    states, logits, actions, logp = (a.cpu().numpy() for a in (states, logits, actions, logp))
    envs = env_offset + np.arange(n, dtype=np.uint64)
    for t in range(T):
        _check_logits(logits[t], states[t], w)
        _check_draws_and_logp(actions[t], logp[t], logits[t], True, P.sample_bits(SEED, envs, step0 + step_offset + t))
    drawn = np.unique(actions)
    assert len(drawn) > 1 and (n < 4096 or len(drawn) == A)      # 4,096 envs draw every action


# ---- (f) cx_discounted_returns -----------------------------------------------------------------------------------------
FLAG_BITS = (P.TERMINATED, P.TRUNCATED, P.BAD_ACTION, P.ALREADY_OVER)
ALL_FLAGS = np.array([sum(b for i, b in enumerate(FLAG_BITS) if k >> i & 1) for k in range(16)], dtype=np.uint8)


def _check_returns(nat, r, f, gamma, d, boot):
    got = nat.discounted_returns(_dev(r), _dev(f), gamma, discount=None if d is None else _dev(d),
                                 bootstrap=None if boot is None else _dev(boot)).cpu().numpy()
    want, mag = P.returns64(r, f, gamma, d, boot)
    bound = P.returns_bound(mag)
    bad = ~(np.abs(got.astype(np.float64) - want) <= bound)
    assert not bad.any(), "returns outside the bound at (t, env) %s" % (np.argwhere(bad)[:8].tolist(),)


@pytest.mark.parametrize("n", (1, 33, 4099))
@pytest.mark.parametrize("T", (1, 2, 57))
def test_discounted_returns_with_every_flag(T, n):
    nat = _nat(n, 5)
    rng = np.random.Generator(np.random.PCG64(T * 10000 + n))
    r = (np.where(rng.random((T, n)) < 0.5, -1.0, 1.0) * 10.0 ** rng.uniform(-3.0, 3.0, (T, n))).astype(np.float32)
    f = ALL_FLAGS[rng.integers(0, 16, (T, n))]
    d = np.where(rng.random((T, n)) < 0.5, np.array([0.0, 0.5, 1.0])[rng.integers(0, 3, (T, n))],
                 rng.random((T, n))).astype(np.float32)
    boot = (rng.normal(0.0, 1.0, n) * 10.0 ** rng.uniform(-3.0, 3.0, n)).astype(np.float32)
    for gamma in (0.0, 0.99, 1.0):
        for disc in (None, d):
            for b in (None, boot):
                _check_returns(nat, r, f, gamma, disc, b)


@pytest.mark.parametrize("n", (1, 33, 4099))
def test_discounted_returns_long_horizon(n):
    """T = 1000, gamma = 0.999 and no episode end (BAD_ACTION / ALREADY_OVER steps do not cut): the rounding error
    carried over a thousand steps stays within the bound."""
    T = 1000
    nat = _nat(n, 5)
    rng = np.random.Generator(np.random.PCG64(n))
    r = (np.where(rng.random((T, n)) < 0.5, -1.0, 1.0) * 10.0 ** rng.uniform(-3.0, 3.0, (T, n))).astype(np.float32)
    f = np.array([0, P.BAD_ACTION, P.ALREADY_OVER], dtype=np.uint8)[rng.integers(0, 3, (T, n))]
    boot = rng.normal(0.0, 100.0, n).astype(np.float32)
    for disc in (None, (0.9 + 0.1 * rng.random((T, n))).astype(np.float32)):
        _check_returns(nat, r, f, 0.999, disc, boot)
