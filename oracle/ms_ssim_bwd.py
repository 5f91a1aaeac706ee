"""Closed-form gradient of oracle.metrics.ms_ssim with respect to its FIRST argument (TEST INFRASTRUCTURE, see oracle/__init__.py).

The derivation ``nic_ms_ssim_bwd`` (csrc/metrics.cu) implements, restated in torch CPU ops so that it can be checked against
autograd over ``oracle.metrics.ms_ssim`` without a GPU (tests/test_ms_ssim_loss_host.py).

Level l (0..4) has input planes x_l, y_l (x_0 = x, y_0 = y; x_{l+1} = avg_pool2d(x_l, 2, padding = size % 2)) and a VALID
output of ho x wo pixels.  Its statistic t_l is the mean of the cs map (l < 4) or of the ssim map (l = 4) over that output.
The gradient is written in the difference u = x - y: with G the separable 11-tap Gaussian (VALID) and the moment maps
m1 = G x, m2 = G y, exx = G x^2, eyy = G y^2, mu = G u, euu = G u^2,

    D = exx - m1^2 + eyy - m2^2 + C2,  V = euu - mu^2 (= s1 + s2 - 2 s12),  cs = 1 - V / D
    L = 1 - mu^2 / B with B = m1^2 + m2^2 + C1 (= (2 m1 m2 + C1) / B),  ssim = L cs

cs depends on x through m1, exx, mu and euu: d cs = a dm1 + b dexx + e (dmu-term of V ...) with
    a = 2 (mu - m1 V / D) / D,  b = V / D^2,  e = -1 / D     (d cs / d m1 incl. the mu path, d cs / d exx, d cs / d euu)
and at l = 4 (ssim): a <- (d L / d m1) cs + L a, b <- L b, e <- L e, d L / d m1 = 2 (m1 mu^2 / B - mu) / B.
All three are scaled by g_l / (ho wo), g_l = d loss / d t_l.  The gradient of the level's input is then
G^T a + 2 x_l (G^T b) + 2 u_l (G^T e) (G^T: the full, transposed filter), plus the coarser level's gradient handed down through
the pooling adjoint g_{l-1}[i, j] += g_l[(i + ph) / 2, (j + pw) / 2] / 4.

Written this way no term is a difference of two large, nearly equal numbers when x_hat is close to x: the textbook form
G^T (d/dm1) + 2 x G^T(-cs / D) + y G^T(2 / D) cancels to O(x - y) from O(x / D) terms and, in fp32, loses about 1e-4 of the
gradient's norm at 1 % noise.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .metrics import WEIGHTS, _filter, _gauss


def pyramid(x, y):
    """[(x_l, y_l)] for the five levels."""
    out = [(x, y)]
    for _ in range(4):
        pad = [s % 2 for s in x.shape[2:]]
        x, y = F.avg_pool2d(x, kernel_size=2, padding=pad), F.avg_pool2d(y, kernel_size=2, padding=pad)
        out.append((x, y))
    return out


def _moments(x, y, win):
    return _filter(x, win), _filter(y, win), _filter(x * x, win), _filter(y * y, win), _filter(x * y, win)


def level_stats(x, y, data_range=1.0):
    """[5, N, C]: mean cs of levels 0-3 and mean ssim of level 4 (the terms ms_ssim raises to the weights)."""
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    win = _gauss(dtype=x.dtype)
    t = []
    for l, (xl, yl) in enumerate(pyramid(x, y)):
        m1, m2, exx, eyy, exy = _moments(xl, yl, win)
        cs = (2 * (exy - m1 * m2) + c2) / (exx - m1 * m1 + eyy - m2 * m2 + c2)
        v = cs if l < 4 else (2 * m1 * m2 + c1) / (m1 * m1 + m2 * m2 + c1) * cs
        t.append(v.flatten(2).mean(-1))
    return torch.stack(t)


def term_grads(t):
    """d v / d t_l for v = prod_l relu(t_l)^w_l per plane ([5, N, C] -> [5, N, C]): w_l v / t_l where t_l > 0, else 0 (so a channel
    with any term <= 0 has v = 0 and no gradient at all) - what autograd gives through relu and pow."""
    w = torch.tensor(WEIGHTS, dtype=t.dtype).view(-1, *([1] * (t.dim() - 1)))
    v = torch.prod(torch.relu(t) ** w, dim=0)
    pos = t > 0
    return torch.where(pos, w * v / torch.where(pos, t, torch.ones_like(t)), torch.zeros_like(t))


def _filter_t(a, win):
    """G^T: the adjoint of _filter (full convolution with the same separable window)."""
    c = a.shape[1]
    k = win.to(a.dtype)
    a = F.conv_transpose2d(a, k.view(1, 1, 1, -1).repeat(c, 1, 1, 1), groups=c)
    return F.conv_transpose2d(a, k.view(1, 1, -1, 1).repeat(c, 1, 1, 1), groups=c)


def backward(x, y, g_level, data_range=1.0):
    """d loss / d x for g_level [5, N, C] = d loss / d t_l (t_l as in level_stats)."""
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    win = _gauss(dtype=x.dtype)
    levels = pyramid(x, y)
    g = None
    for l in range(4, -1, -1):
        xl, yl = levels[l]
        ul = xl - yl
        m1, m2, exx, eyy = _filter(xl, win), _filter(yl, win), _filter(xl * xl, win), _filter(yl * yl, win)
        mu, euu = _filter(ul, win), _filter(ul * ul, win)
        d = exx - m1 * m1 + eyy - m2 * m2 + c2
        v = euu - mu * mu
        a, b, e = 2 * (mu - m1 * v / d) / d, v / (d * d), -1 / d
        if l == 4:
            bl = m1 * m1 + m2 * m2 + c1
            lum, cs = 1 - mu * mu / bl, 1 - v / d
            a, b, e = 2 * (m1 * mu * mu / bl - mu) / bl * cs + lum * a, lum * b, lum * e
        scale = (g_level[l] / (m1.shape[2] * m1.shape[3]))[..., None, None]
        a, b, e = a * scale, b * scale, e * scale
        gl = _filter_t(a, win) + 2 * xl * _filter_t(b, win) + 2 * ul * _filter_t(e, win)
        if g is not None:
            ph, pw = (s % 2 for s in xl.shape[2:])
            iy = (torch.arange(xl.shape[2]) + ph) // 2
            ix = (torch.arange(xl.shape[3]) + pw) // 2
            gl = gl + g[:, :, iy][:, :, :, ix] / 4
        g = gl
    return g


def ms_ssim_grad(x, y, data_range=1.0):
    """d mean_{N, C}(ms_ssim per plane) / d x - the gradient autograd gives over oracle.metrics.ms_ssim(x, y)."""
    t = level_stats(x, y, data_range)
    return backward(x, y, term_grads(t) / (t.shape[1] * t.shape[2]), data_range)
