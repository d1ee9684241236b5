"""numpy (float64) Kronecker factors of the per-point empirical Fisher  --  TEST INFRASTRUCTURE ONLY.

For every Linear layer: the per-point inputs a~_i = [a_i; 1] (a_i without a bias) and the pre-activation gradients
delta_i = d log p_i / d z of point i's data term -0.5 ||y_i - f(x_i)||^2 / sigma^2, restated from
oracle.quinn_oracle.logpost_grad, and the raw sums kernel 6 (qb_logpost_kfac) returns:
    A = sum_i a_i a_i^T,   s = sum_i a_i (bias only),   G = sum_i delta_i delta_i^T.
It sits next to the oracle rather than in it because oracle/quinn_oracle.py is pinned against fixtures recorded from the
reference, which has no such function.  tests/test_kfac_cpu.py checks outer(delta_i, a~_i) against torch autograd.
"""
import numpy as np

from oracle.quinn_oracle import _act, _dact, _layer_wb


def per_point(layers, theta, x, y, sigma, final=None):
    """Per layer (a~ [N, n_in (+1)], delta [N, n_out]); a~ carries the trailing 1 column for layers with a bias."""
    theta = np.asarray(theta, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    h = np.asarray(x, dtype=np.float64)
    cache = []
    for L in layers:
        if len(L.get('terms', [None])) > 1:
            raise ValueError('Kronecker factors need plain layers (no polynomial-in-depth weights)')
        W, b = _layer_wb(L, theta)
        z = h @ W.T + (b if b is not None else 0.0)
        a = _act(L['act'], z)
        cache.append((h, z, a, W))
        h = h + L['res_step'] * a if L['res_step'] != 0.0 else a
    out = np.exp(h) if final == 'exp' else h
    da = (y - out) / sigma ** 2
    if final == 'exp':
        da = da * out
    res = []
    for L, (hin, z, a, W) in zip(reversed(layers), reversed(cache)):
        scale = L['res_step'] if L['res_step'] != 0.0 else 1.0
        dz = scale * da * _dact(L['act'], z, a)
        at = np.hstack([hin, np.ones((hin.shape[0], 1))]) if L['b_off'] >= 0 else hin
        res.append((at, dz))
        dprev = dz @ W
        da = dprev + da if L['res_step'] != 0.0 else dprev
    return res[::-1]


def factors(layers, theta, x, y, sigma, final=None):
    """Per layer dict(A, s, G) of raw sums over the points (s is None without a bias)."""
    out = []
    for L, (at, d) in zip(layers, per_point(layers, theta, x, y, sigma, final)):
        a = at[:, :L['n_in']]
        out.append(dict(A=a.T @ a, s=a.sum(0) if L['b_off'] >= 0 else None, G=d.T @ d))
    return out


def layer_index(L):
    """theta index of entry (j, i) of the layer's [W | b] matrix, row-major: [n_out, n_in (+1)]"""
    n_in, n_out = L['n_in'], L['n_out']
    idx = L['w_off'] + np.arange(n_out)[:, None] * n_in + np.arange(n_in)[None, :]
    if L['b_off'] >= 0:
        idx = np.hstack([idx, (L['b_off'] + np.arange(n_out))[:, None]])
    return idx


def kron_precision(layers, theta, x, y, sigma, tau=0.0, final=None):
    """Dense (P, P) block-diagonal Lambda in theta order: per layer G/N (x) A~/N + tau I, A~ = [[A, s], [s^T, N]]."""
    N = np.asarray(x).shape[0]
    P = np.asarray(theta).size
    Lam = np.zeros((P, P))
    for L, f in zip(layers, factors(layers, theta, x, y, sigma, final)):
        A = f['A']
        if f['s'] is not None:
            A = np.block([[A, f['s'][:, None]], [f['s'][None, :], np.array([[float(N)]])]])
        blk = np.kron(f['G'] / N, A / N) + tau * np.eye(A.shape[0] * f['G'].shape[0])
        idx = layer_index(L).ravel()
        Lam[np.ix_(idx, idx)] = blk
    return Lam
