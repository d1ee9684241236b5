"""numpy (float64) Hessian-vector products of the log-posterior  --  TEST INFRASTRUCTURE ONLY.

A forward-over-reverse restatement of oracle.quinn_oracle.logpost_grad: the tangent of every forward quantity along a
direction v, then the tangent of the reverse sweep.  It sits next to the oracle rather than in it because
oracle/quinn_oracle.py is pinned against fixtures recorded from the reference, which has no such function.
tests/test_hessian_cpu.py checks it against torch autograd; kernel 5 (qb_logpost_hvp) is checked against it.
"""
import numpy as np

from oracle.quinn_oracle import _layer_wb


def _act_d12(name, z):
    """act'(z), act''(z)"""
    if name == 'tanh':
        t = np.tanh(z)
        return 1.0 - t * t, -2.0 * t * (1.0 - t * t)
    if name == 'relu':
        return (z > 0).astype(z.dtype), np.zeros_like(z)
    return np.ones_like(z), np.zeros_like(z)


def _act(name, z):
    if name == 'tanh':
        return np.tanh(z)
    if name == 'relu':
        return np.maximum(z, 0.0)
    return z


def logpost_hvp(layers, theta, x, y, sigma, fulldatasize=None, prior=None, final=None, v=None):
    """(d^2 lp / d theta^2) v with lp = oracle.logpost (same terms, same sign).  v: (P,) or (K, P); returns the same
    shape."""
    v = np.asarray(v, dtype=np.float64)
    if v.ndim == 2:
        return np.stack([logpost_hvp(layers, theta, x, y, sigma, fulldatasize, prior, final, vk) for vk in v])
    theta = np.asarray(theta, dtype=np.float64)
    y = np.asarray(y, dtype=np.float64)
    h = np.asarray(x, dtype=np.float64)
    hd = np.zeros_like(h)
    cache = []
    for L in layers:
        W, b = _layer_wb(L, theta)
        V, vb = _layer_wb(L, v)
        z = h @ W.T + (b if b is not None else 0.0)
        zd = hd @ W.T + h @ V.T + (vb if vb is not None else 0.0)
        d1, d2 = _act_d12(L['act'], z)
        s, sd = _act(L['act'], z), d1 * zd
        cache.append((h, hd, z, zd, W, V))
        if L['res_step'] != 0.0:
            h, hd = h + L['res_step'] * s, hd + L['res_step'] * sd
        else:
            h, hd = s, sd
    u, ud = h, hd
    if final == 'exp':
        e = np.exp(u)
        r = y - e
        da, dda = r * e / sigma ** 2, e * ud * (r - e) / sigma ** 2
    else:
        da, dda = (y - u) / sigma ** 2, -ud / sigma ** 2
    hv = np.zeros_like(theta)
    for L, (hin, hdin, z, zd, W, V) in zip(reversed(layers), reversed(cache)):
        scale = L['res_step'] if L['res_step'] != 0.0 else 1.0
        d1, d2 = _act_d12(L['act'], z)
        dz = scale * d1 * da
        ddz = scale * (d1 * dda + d2 * zd * da)
        hW, hb = (ddz.T @ hin + dz.T @ hdin).ravel(), ddz.sum(axis=0)
        for c, wo, bo in L.get('terms', [(1.0, L['w_off'], L['b_off'])]):
            hv[wo:wo + L['n_in'] * L['n_out']] += c * hW
            if bo >= 0:
                hv[bo:bo + L['n_out']] += c * hb
        da_in, dda_in = dz @ W, ddz @ W + dz @ V
        if L['res_step'] != 0.0:
            da_in, dda_in = da_in + da, dda_in + dda
        da, dda = da_in, dda_in
    if prior is not None:
        hv -= (y.shape[0] / fulldatasize) * v / prior['sigma'] ** 2
    return hv


def logpost_hessian(layers, theta, x, y, sigma, fulldatasize=None, prior=None, final=None):
    """Full (P, P) Hessian of lp: one product per unit direction."""
    P = np.asarray(theta).size
    return logpost_hvp(layers, theta, x, y, sigma, fulldatasize, prior, final, np.eye(P))

