"""Per-joint feedback policies (include/rem2d_policy.h): the weight layout, the features and the network in numpy float64.

Every joint has its own network with H hidden units (1 <= H <= 16) and P = 10 * H + 1 weights: W1 (H x 8, row-major), b1 (H),
w2 (H), b2. Its inputs are the sine controller's output s and the end-of-tick observations (``features``); its output u is
added to s, and the P-controller drives the joint to s + u. ``forward`` is the definition the CUDA library and the oracle
compute, bit for bit: element-wise operations in the stated order (no BLAS, whose sums may be reordered)."""
import numpy as np

N_FEATURES = 8
MAX_HIDDEN = 16


def n_params(H):
    """Weights per joint for H hidden units."""
    if not 1 <= int(H) <= MAX_HIDDEN:
        raise ValueError("the hidden layer has 1..%d units, not %r" % (MAX_HIDDEN, H))
    return 10 * int(H) + 1


def hidden_size(P):
    """H for P weights per joint; ValueError unless P = 10 * H + 1 with 1 <= H <= 16."""
    P = int(P)
    if P < 11 or (P - 1) % 10 or (P - 1) // 10 > MAX_HIDDEN:
        raise ValueError("a policy has 10 * H + 1 weights per joint with 1 <= H <= %d, not %d" % (MAX_HIDDEN, P))
    return (P - 1) // 10


def _joints(table):
    """(creature, A, B) of every joint in table order: its creature and the global indices of its parent and child bodies."""
    body_off = np.asarray(table.body_off, np.int64)
    nbs = np.diff(body_off)
    c = np.repeat(np.arange(table.n_creatures), nbs - 1)
    k = np.arange(table.n_bodies - table.n_creatures) - (body_off[:-1] - np.arange(table.n_creatures))[c]
    return c, body_off[c] + np.asarray(table.joint_parent, np.int64), body_off[c] + k + 1


def features(obs, sine, table):
    """float64[n_joints, 8] inputs of every joint's network: the sine outputs ``sine`` of this tick and the observations
    ``obs`` of the state at its start (``Engine.read_observations``): s, joint angle, joint speed, ground[B], ground[A], root
    angle, root vx, root vy."""
    c, A, B = _joints(table)
    root = np.asarray(obs["root"])
    ground = np.asarray(obs["ground"])
    x = np.empty((len(c), N_FEATURES), np.float64)
    x[:, 0] = sine
    x[:, 1] = np.asarray(obs["joint_angle"], np.float32)
    x[:, 2] = np.asarray(obs["joint_speed"], np.float32)
    x[:, 3] = ground[B]
    x[:, 4] = ground[A]
    x[:, 5] = root[c, 2]
    x[:, 6] = root[c, 3]
    x[:, 7] = root[c, 4]
    return x


def forward(weights, x):
    """u = float64[n_joints]: every joint's network on its features x[n_joints, 8], in the order of include/rem2d_policy.h."""
    W = np.asarray(weights, np.float64)
    H = hidden_size(W.shape[1])
    x = np.asarray(x, np.float64)
    u = W[:, 10 * H].copy()
    for k in range(H):
        acc = W[:, 8 * H + k].copy()
        for i in range(N_FEATURES):
            acc = acc + W[:, 8 * k + i] * x[:, i]
        u = u + W[:, 9 * H + k] * (acc / (1.0 + np.abs(acc)))
    return u


def random_weights(n_joints, H, scale=1.0, rng=None):
    """float64[n_joints, 10 * H + 1], normal with standard deviation ``scale``."""
    rng = np.random.default_rng(rng)
    return rng.normal(0.0, scale, (int(n_joints), n_params(H)))
