"""numpy (float64) output Jacobians and the linearised (GLM) predictive  --  TEST INFRASTRUCTURE ONLY.

For every point x_n and output j: the Jacobian J[n, j, :] = d f_j(x_n) / d theta, and the per-layer pairs kernel 7
(qb_predict_jac) returns, a_l = the layer's input [n_in, N] and d_l[j] = d f_j / d z_l [o, n_out, N], restated from the
forward pass of oracle.quinn_oracle.  Layer l's part of J is outer(d_l[j, :, n], [a_l[:, n]; 1]), times coef_m at each
polynomial term, summed over layers that share weights.  The GLM moments of one member are f(mu) and cov_scale J Sigma
J^T; members mix with equal weights.  It sits next to the oracle rather than in it because oracle/quinn_oracle.py is
pinned against fixtures recorded from the reference, which has no such function.  tests/test_glm_cpu.py checks J against
torch autograd.
"""
import numpy as np

from oracle.quinn_oracle import _act, _dact, _layer_wb


def pairs(layers, theta, x, final=None):
    """(f [N, o], per layer dict(a=[n_in, N], d=[o, n_out, N]))"""
    theta = np.asarray(theta, dtype=np.float64)
    h = np.asarray(x, dtype=np.float64)
    cache = []
    for L in layers:
        W, b = _layer_wb(L, theta)
        z = h @ W.T + (b if b is not None else 0.0)
        a = _act(L['act'], z)
        cache.append((h, z, a, W))
        h = h + L['res_step'] * a if L['res_step'] != 0.0 else a
    f = np.exp(h) if final == 'exp' else h
    N, o = f.shape
    res = [dict(a=hin.T.copy(), d=np.zeros((o, L['n_out'], N))) for L, (hin, *_) in zip(layers, cache)]
    for j in range(o):
        da = np.zeros((N, o))
        da[:, j] = f[:, j] if final == 'exp' else 1.0
        for l in range(len(layers) - 1, -1, -1):
            L, (hin, z, a, W) = layers[l], cache[l]
            scale = L['res_step'] if L['res_step'] != 0.0 else 1.0
            dz = scale * da * _dact(L['act'], z, a)
            res[l]['d'][j] = dz.T
            dprev = dz @ W
            da = dprev + da if L['res_step'] != 0.0 else dprev
    return f, res


def assemble(layers, P, prs):
    """J [N, o, P] from per-layer pairs (polynomial terms scaled by coef, shared weights summed)"""
    N = prs[0]['a'].shape[1]
    o = prs[0]['d'].shape[0]
    J = np.zeros((N, o, P))
    for L, p in zip(layers, prs):
        gW = np.einsum('jun,in->njui', p['d'], p['a']).reshape(N, o, -1)
        gb = p['d'].transpose(2, 0, 1)
        for c, wo, bo in L.get('terms', [(1.0, L['w_off'], L['b_off'])]):
            J[:, :, wo:wo + gW.shape[2]] += c * gW
            if bo >= 0:
                J[:, :, bo:bo + L['n_out']] += c * gb
    return J


def jacobian(layers, theta, x, final=None):
    """(f [N, o], J [N, o, P])"""
    f, prs = pairs(layers, theta, x, final)
    return f, assemble(layers, np.asarray(theta).size, prs)


def glm_moments(members, cov_scale):
    """Mixture of the members' linearised predictives, members = [(f [N, o], J [N, o, P], Sigma [P, P])]:
    (mean [N, o], var [N, o], cov [N, N, o]) by the law of total (co)variance, equal weights."""
    fs = np.stack([f for f, _, _ in members])
    mean = fs.mean(0)
    N, o = mean.shape
    cov = np.zeros((N, N, o))
    for f, J, S in members:
        for j in range(o):
            cov[:, :, j] += cov_scale * J[:, j] @ S @ J[:, j].T + np.outer(f[:, j] - mean[:, j], f[:, j] - mean[:, j])
    cov /= len(members)
    var = np.stack([np.diag(cov[:, :, j]) for j in range(o)], 1)
    return mean, var, cov
