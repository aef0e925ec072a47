"""Float64 host references of the float kernels on the actor-critic path -- the policy MLP and its draw
(campx_b200/csrc/cx_policy.cuh: k_policy_sample, k_policy_sample_board, k_agent_policy_rollout), k_sample_actions and
k_discounted_returns (cx_aux_kernels.cu) -- with error bounds derived from the float32 arithmetic those kernels do.

Notation: u = 2^-24 is the unit roundoff of float32 and gamma_k = k u / (1 - k u) bounds k successive roundings
(Higham, Accuracy and Stability of Numerical Algorithms, 2nd ed., section 3.1).  One ulp of a float32 y is at most
2u |y|.  The float64 references themselves round at 2^-53, far below every bound here.
"""
import math

import numpy as np

U = 2.0 ** -24
# CX_FLAG_* of campx_b200/_native.py (repeated so that the host-only tests need no native library)
TERMINATED, TRUNCATED, ALREADY_OVER, BAD_ACTION = 0x01, 0x02, 0x08, 0x80
SAMPLE_KEY = 0x5A4D504C45          # sample_bits (cx_policy.cuh): the key is seed ^ SAMPLE_KEY
LOGF_ABS = 2.0 ** -21.41           # __logf(x), x in [0.5, 2]: absolute error (CUDA C++ Programming Guide, intrinsics)
DENORMAL = 2.0 ** -125             # covers a weight flushed to zero (__expf of an argument below about -87)


def gamma(k):
    k = np.asarray(k, dtype=np.float64)
    return k * U / (1.0 - k * U)


# ---- Philox4x32-10 (campx_b200/csrc/cx_philox.cuh) ---------------------------------------------------------------
_M0, _M1, _W0, _W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85


def philox4(seed, quad, t):
    """Scalar host spec of cx_philox4 (Python ints): key = seed, counter = (quad, t) -> four 32-bit words."""
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    c = [quad & 0xFFFFFFFF, quad >> 32, t & 0xFFFFFFFF, t >> 32]
    for _ in range(10):
        p0, p1 = _M0 * c[0], _M1 * c[2]
        c = [(p1 >> 32) ^ c[1] ^ k0, p1 & 0xFFFFFFFF, (p0 >> 32) ^ c[3] ^ k1, p0 & 0xFFFFFFFF]
        k0, k1 = (k0 + _W0) & 0xFFFFFFFF, (k1 + _W1) & 0xFFFFFFFF
    return c


def philox4_np(seed, quad, step):
    """philox4 over uint64 arrays (quad and step broadcast against each other) -> uint32 [4, *shape]."""
    quad, step = np.broadcast_arrays(np.asarray(quad, dtype=np.uint64), np.asarray(step, dtype=np.uint64))
    mask, s32 = np.uint64(0xFFFFFFFF), np.uint64(32)
    m0, m1, w0, w1 = np.uint64(_M0), np.uint64(_M1), np.uint64(_W0), np.uint64(_W1)
    seed = np.uint64(seed)
    k0, k1 = seed & mask, seed >> s32
    c0, c1, c2, c3 = quad & mask, quad >> s32, step & mask, step >> s32
    for _ in range(10):
        p0, p1 = m0 * c0, m1 * c2                                  # 32 x 32 -> 64 bits: exact in uint64
        c0, c1, c2, c3 = (p1 >> s32) ^ c1 ^ k0, p1 & mask, (p0 >> s32) ^ c3 ^ k1, p0 & mask
        k0, k1 = (k0 + w0) & mask, (k1 + w1) & mask
    return np.stack([c0, c1, c2, c3]).astype(np.uint32)


def sample_bits(seed, env, step):
    """The 32 random bits sample_bits (cx_policy.cuh) gives global env `env` at `step` (step = d_step[0] + step_offset):
    key seed ^ SAMPLE_KEY, counter (env >> 2, step), word env & 3."""
    env, step = np.broadcast_arrays(np.asarray(env, dtype=np.uint64), np.asarray(step, dtype=np.uint64))
    w = philox4_np(int(seed) ^ SAMPLE_KEY, env >> np.uint64(2), step)
    return np.choose((env & np.uint64(3)).astype(np.int64), list(w))


# ---- the policy MLP ------------------------------------------------------------------------------------------------
def mlp_logits(x, w1t, b1, w2, b2):
    """relu(x W1^T + b1) W2^T + b2 in float64 -> (logits [n, A], M [n, A]).  M is the same network on absolute values,
    M_a = |b2_a| + sum_j |W2_aj| (|b1_j| + sum_d |W1^T_dj x_d|): every float32 rounding the kernel makes is relative to
    a partial sum bounded by it."""
    x, w1t, b1, w2, b2 = (np.asarray(a, dtype=np.float64) for a in (x, w1t, b1, w2, b2))
    logits = np.maximum(x @ w1t + b1, 0.0) @ w2.T + b2
    mag = np.abs(b2) + (np.abs(b1) + np.abs(x) @ np.abs(w1t)) @ np.abs(w2).T
    return logits, mag


def logit_bound(x, n_hidden, mag):
    """|float32 logits - mlp_logits| <= 2 gamma_k M_a, k = nnz(x row) + n_hidden + 16.

    A hidden unit is b1_j plus one fmaf per input in sequence; an input that is 0 adds an exact fmaf(w, 0, acc) == acc,
    so only the nonzero inputs round.  ReLU does not grow an error.  The output layer rounds each term at most
    4 + 8 times in the kernel (the warp's product and three fmaf over its four hidden units, then b2 plus the eight
    warp shares in sequence); n_hidden + 16 bounds it for any summation order.  The factor 2 leaves room for terms
    of second order."""
    nnz = np.count_nonzero(np.asarray(x), axis=1)
    return 2.0 * gamma(nnz + n_hidden + 16)[:, None] * mag


def mlp_logits_f32(x, w1t, b1, w2, b2, skip_last_input=False, skip_b2=False):
    """Float32 emulation of the kernels' arithmetic (policy_hidden_shares + policy_logits, cx_policy.cuh): per hidden
    unit a sequential fmaf over the inputs, then per warp of four hidden units fmaf(c3, h3, fmaf(c2, h2, fmaf(c1, h1,
    c0 * h0))), then b2 plus the eight warp shares in warp order.  fmaf is emulated in float64 (the product of two
    float32 is exact there) with one rounding to float32.  skip_last_input drops the last nonzero input of every row,
    skip_b2 the output bias: the two defects the logit bound must expose."""
    f32 = np.float32
    x, w1t, b1, w2, b2 = (np.asarray(a, dtype=f32) for a in (x, w1t, b1, w2, b2))
    n, n_in = x.shape
    n_hidden, A = w1t.shape[1], w2.shape[0]
    if skip_last_input:
        x = x.copy()
        last = n_in - 1 - np.argmax(x[:, ::-1] != 0, axis=1)
        x[np.arange(n), last] = 0
    w1p = np.zeros((n_in, 32), dtype=f32)                       # hidden units padded to 32 with zeros, as staged
    w1p[:, :n_hidden] = w1t
    w2p = np.zeros((A, 32), dtype=f32)
    w2p[:, :n_hidden] = w2
    acc = np.broadcast_to(np.concatenate([b1, np.zeros(32 - n_hidden, dtype=f32)]), (n, 32)).astype(f32)
    for d in range(n_in):
        col = x[:, d]
        nz = col != 0
        if nz.any():
            acc[nz] = (w1p[d].astype(np.float64) * col[nz, None].astype(np.float64) + acc[nz]).astype(f32)
    h = np.maximum(acc, f32(0))
    logits = np.empty((n, A), dtype=f32)
    for a in range(A):
        s = np.zeros(n, dtype=f32) if skip_b2 else np.full(n, b2[a], dtype=f32)
        for w in range(8):
            c, hw = w2p[a, 4 * w:4 * w + 4].astype(np.float64), h[:, 4 * w:4 * w + 4].astype(np.float64)
            share = (c[0] * hw[:, 0]).astype(f32)
            for q in (1, 2, 3):
                share = (c[q] * hw[:, q] + share.astype(np.float64)).astype(f32)
            s = (s + share).astype(f32)
        logits[:, a] = s
    return logits


def policy_weights(rng, n_in, n_hidden, A, spread=30.0, fan_in=None):
    """float32 (w1t [n_in, n_hidden], b1, w2 [A, n_hidden], b2) whose magnitudes span several orders of magnitude
    (W1^T entries log-uniform in [1e-3, 1] times 4 / sqrt(fan_in), fan_in: the nonzero inputs per row, default n_in,
    so that the hidden units are of order 1) and whose output bias spreads an env's logits over about `spread`."""
    sign = lambda *s: np.where(rng.random(s) < 0.5, -1.0, 1.0)
    w1t = sign(n_in, n_hidden) * 10.0 ** rng.uniform(-3.0, 0.0, (n_in, n_hidden)) * 4.0 / math.sqrt(fan_in or n_in)
    b1 = rng.normal(0.0, 0.5, n_hidden)
    w2 = sign(A, n_hidden) * 10.0 ** rng.uniform(-1.0, 1.0, (A, n_hidden)) / math.sqrt(n_hidden)
    b2 = (np.linspace(-spread / 2, spread / 2, A) if A > 1 else np.zeros(1)) + rng.normal(0.0, 1.0, A)
    return tuple(np.ascontiguousarray(a, dtype=np.float32) for a in (w1t, b1, w2, b2))


# ---- the draw: sample_categorical_bits (cx_policy.cuh) ---------------------------------------------------------------
def weights_of(scores, is_logits):
    """The weights sample_categorical_bits draws from, in float64, and a bound on the kernel's error in each
    -> (w [n, A], err [n, A]).

    Probabilities: w = p where p > 0, else 0 (negative and NaN weights count as zero): exact, err = 0.
    Logits: w = exp(l - max l).  The kernel computes __expf(fl(l - max l)): the subtraction rounds once (relative
    error u |x| in the weight, x = l - max l) and __expf is within 2 + floor(1.173 |x|) ulp (CUDA C++ Programming
    Guide, intrinsic functions), at most 2u |w| each, plus an absolute DENORMAL for a flushed result."""
    s = np.asarray(scores, dtype=np.float64)
    if not is_logits:
        w = np.where(s > 0, s, 0.0)                               # (NaN > 0 is False)
        return w, np.zeros_like(w)
    x = s - s.max(axis=1, keepdims=True)
    w = np.exp(x)
    ax = np.abs(x)
    return w, w * (2.0 * U * (2.0 + np.floor(1.173 * ax)) + U * ax) + DENORMAL


def draw(p64, bits):
    """Float64 inverse-CDF pick of sample_categorical_bits: u = (bits >> 8) / 2^24 and the first action a with
    u < C_a, C_a = sum_{b <= a} p_b / sum p.  -> (pick [n], u [n], dist [n]): dist is the distance, in units of the
    total, from u to the nearest inner CDF edge C_0 .. C_{A-2} (inf for A = 1)."""
    p = np.asarray(p64, dtype=np.float64)
    n, A = p.shape
    cdf = np.cumsum(p, axis=1) / p.sum(axis=1, keepdims=True)
    u = (np.asarray(bits, dtype=np.uint32) >> np.uint32(8)).astype(np.float64) / 2.0 ** 24
    pick = np.minimum((cdf <= u[:, None]).sum(axis=1), A - 1)
    dist = np.abs(cdf[:, :-1] - u[:, None]).min(axis=1) if A > 1 else np.full(n, np.inf)
    return pick, u, dist


def draw_band(w, err):
    """delta [n]: how far the kernel's CDF edges can lie from the float64 ones, in units of the total.  The kernel
    picks the first a with fl(u * total) < cum_a, where cum_a and total are the same float32 running sum of its
    weights.  Three things move an edge: the weights' error E = sum err (at most 2E / (S - E), S = sum w), the float32
    running sum (cum_a and total within gamma_A each) and the product u * total (u).  The factor 2 leaves room for
    terms of second order."""
    A = w.shape[1]
    S, E = w.sum(axis=1), err.sum(axis=1)
    return 2.0 * (2.0 * E / (S - E) + 2.0 * gamma(A) + U)


def check_draws(actions, w, err, bits):
    """Every kernel draw against the float64 pick -> (measure, observed): the mean share of [0, 1) the bands of the
    inner CDF edges cover (the chance that a uniform u falls in one: the share of draws the band can excuse) and the
    share of these draws that fell in one.  Outside the band a draw must equal the pick.  Inside it may be any action
    of positive weight whose CDF interval reaches within delta of u (the neighbours of the edge), never one of zero
    weight."""
    actions = np.asarray(actions).astype(np.int64)
    n, A = w.shape
    pick, u, dist = draw(w, bits)
    delta = draw_band(w, err)
    band = dist < delta
    bad = ~band & (actions != pick)
    assert not bad.any(), "draw differs from the float64 pick outside the band: envs %s, kernel %s, float64 %s" % (
        np.flatnonzero(bad)[:8], actions[bad][:8], pick[bad][:8])
    cdf = np.cumsum(w, axis=1) / w.sum(axis=1, keepdims=True)
    lo = np.concatenate([np.zeros((n, 1)), cdf[:, :-1]], axis=1)
    rows = np.arange(n)
    a = np.clip(actions, 0, A - 1)
    ok = (actions < A) & (w[rows, a] > 0) & (lo[rows, a] - delta <= u) & (u < cdf[rows, a] + delta)
    assert ok[band].all(), "draw near a CDF edge picks an action that is no neighbour of it: envs %s" % (
        np.flatnonzero(band & ~ok)[:8])
    inner = cdf[:, :-1]
    covered = np.minimum(inner + delta[:, None], 1.0) - np.maximum(inner - delta[:, None], 0.0)
    return float(np.minimum(covered.sum(axis=1), 1.0).mean()), float(band.mean())


def log_softmax64(logits):
    x = np.asarray(logits, dtype=np.float64)
    x = x - x.max(axis=1, keepdims=True)
    return x - np.log(np.exp(x).sum(axis=1, keepdims=True))


def logp_bound(w, err, actions, ref):
    """|kernel log p - ref| for the drawn actions: the kernel returns __logf(fl(w_a / total)).  The ratio is within a
    relative eta = err_a / w_a + E / S + gamma_{A-1} (the running sum) + u (the division) of the float64 one, which
    moves its log by at most eta / (1 - eta); __logf adds 2^-21.41 (ratio in [0.5, 2]) or 3 ulp of the result,
    at most 6u (|ref| + that)."""
    n, A = w.shape
    rows, a = np.arange(n), np.asarray(actions).astype(np.int64)
    S, E = w.sum(axis=1), err.sum(axis=1)
    eta = err[rows, a] / w[rows, a] + E / (S - E) + gamma(A - 1) + U
    moved = eta / (1.0 - eta)
    return moved + LOGF_ABS + 6.0 * U * (np.abs(ref) + moved)


# ---- discounted returns (k_discounted_returns) -------------------------------------------------------------------------
def returns64(reward, flags, gamma_, discount=None, bootstrap=None):
    """R_t = r_t + gamma c_t R_{t+1} backwards in float64, R_T = bootstrap (or 0), c_t = 0 where flags_t has
    TERMINATED or TRUNCATED (the step ended its episode: the return is cut), else discount_t (or 1); BAD_ACTION and
    ALREADY_OVER do not cut.  gamma is taken as the float32 the kernel receives.  -> (R [T, n], A [T, n]) with the
    magnitude A_t = |r_t| + gamma c_t A_{t+1}, A_T = |bootstrap|."""
    r = np.asarray(reward, dtype=np.float64)
    f = np.asarray(flags)
    T, n = r.shape
    g64 = float(np.float32(gamma_))
    c = np.ones((T, n)) if discount is None else np.asarray(discount, dtype=np.float64)
    c = np.where((f & (TERMINATED | TRUNCATED)) != 0, 0.0, c)
    R, M = np.empty((T, n)), np.empty((T, n))
    g = np.zeros(n) if bootstrap is None else np.asarray(bootstrap, dtype=np.float64).copy()
    m = np.abs(g)
    for t in range(T - 1, -1, -1):
        g = r[t] + g64 * c[t] * g
        m = np.abs(r[t]) + g64 * c[t] * m
        R[t], M[t] = g, m
    return R, M


def returns_bound(mag):
    """|float32 R_t - R_t| <= 4 (T - t + 1) u A_t: each step rounds gamma * c once and the fmaf once, and gamma c <= 1
    keeps the errors carried from later steps from growing (twice the rounding count)."""
    T = mag.shape[0]
    return 4.0 * (T - np.arange(T) + 1)[:, None] * U * mag


# ---- goodness of fit -----------------------------------------------------------------------------------------------------
def chi2_sf(x, dof):
    """P(X >= x) for X ~ chi-square(dof), in closed form: sf(x; 1) = erfc(sqrt(x / 2)), sf(x; 2) = exp(-x / 2) and
    sf(x; k + 2) = sf(x; k) + (x / 2)^(k / 2) exp(-x / 2) / Gamma(k / 2 + 1)."""
    h = x / 2.0
    sf, k = (math.erfc(math.sqrt(h)), 1) if dof % 2 else (math.exp(-h), 2)
    while k < dof:
        sf += math.exp((k / 2.0) * math.log(h) - h - math.lgamma(k / 2.0 + 1.0)) if h > 0 else 0.0
        k += 2
    return sf
