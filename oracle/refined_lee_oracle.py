"""
TEST INFRASTRUCTURE ONLY.  NumPy float64 statement of the refined Lee filter of include/ndchg.h
(`ndchg_refined_lee`): for every pixel of every time step, the edge-aligned mask of its N x N window chosen from the
3 x 3 subwindow means of the span, and out = M + b (x - M) with the local statistics of the span over that mask.

It shares no code with the kernel.  It is vectorised over pixels and loops over the window offsets in the stated
order, accumulating `acc = acc + term` (never `np.sum` / `.mean` over a window axis, whose pairwise summation would
change the order); a mask sum adds the terms of the offsets inside the mask and keeps the others out with
`np.where`.  The reflect edge is `np.pad(mode='symmetric')`; the diagonal bands of a layout are read from
`nd_b200.change.POLS`.
"""
import numpy as np

from nd_b200.change import POLS

WINDOWS = (7, 11, 15)


def sizes(window):
    """(h, s, c): half window, subwindow side and subwindow spacing of an N = 4m + 3 window."""
    h = window // 2
    s = (window - 1) // 2
    return h, s, (window - s) // 2


def span(x, pol):
    """C11 + C22 (+ C33), added left to right in band order; single-pol: C11."""
    diag = [POLS[pol].index(b) for b in ('C11', 'C22', 'C33') if b in POLS[pol]]
    y = x[..., diag[0]]
    for d in diag[1:]:
        y = y + x[..., d]
    return y


def selection(values, window, pol):
    """Per sample (rows, cols, k): the subwindow means `m` (3, 3, rows, cols, k), the edge `e` (0 .. 3) and `second`
    (True where the second mask of the edge is taken), in float64."""
    x = np.asarray(values).astype(np.float64)
    rows, cols = x.shape[:2]
    h, s, c = sizes(window)
    yp = np.pad(span(x, pol), ((h, h), (h, h), (0, 0)), mode='symmetric')
    r = (s - 1) // 2
    m = np.empty((3, 3) + x.shape[:3])
    for u in range(3):
        for v in range(3):
            acc = np.zeros(x.shape[:3])
            for a in range(-r, r + 1):
                for b in range(-r, r + 1):
                    dy, dx = (u - 1) * c + a, (v - 1) * c + b
                    acc = acc + yp[h + dy:h + dy + rows, h + dx:h + dx + cols]
            m[u, v] = acc / (s * s)
    G = [np.abs((m[0, 2] + m[1, 2] + m[2, 2]) - (m[0, 0] + m[1, 0] + m[2, 0])),
         np.abs((m[2, 0] + m[2, 1] + m[2, 2]) - (m[0, 0] + m[0, 1] + m[0, 2])),
         np.abs((m[0, 1] + m[0, 2] + m[1, 2]) - (m[1, 0] + m[2, 0] + m[2, 1])),
         np.abs((m[0, 0] + m[0, 1] + m[1, 0]) - (m[1, 2] + m[2, 1] + m[2, 2]))]
    e = np.zeros(x.shape[:3], np.int64)
    Ge = G[0]
    for i in (1, 2, 3):
        win = G[i] > Ge                                          # strict: the first maximum wins, NaN never wins
        e = np.where(win, i, e)
        Ge = np.where(win, G[i], Ge)
    pairs = [((1, 0), (1, 2)), ((0, 1), (2, 1)), ((0, 2), (2, 0)), ((0, 0), (2, 2))]
    first = np.choose(e, [m[p[0]] for p in pairs])
    second = np.choose(e, [m[p[1]] for p in pairs])
    return m, e, np.abs(second - m[1, 1]) < np.abs(first - m[1, 1])


def in_mask(e, second, dy, dx):
    """True where offset (dy, dx) lies in the mask of (e, second): d <= 0 (first) or d >= 0 (second), with
    d = dx, dy, dy - dx, dy + dx for e = 0 .. 3."""
    d = np.choose(e, [dx, dy, dy - dx, dy + dx])
    return np.where(second, d >= 0, d <= 0)


def statistics(values, looks, window, pol):
    """Per sample: e, second, ybar, var_y, b (rows, cols, k) and the masked band means M (rows, cols, k, bands),
    float64."""
    x = np.asarray(values).astype(np.float64)
    rows, cols = x.shape[:2]
    h = window // 2
    n = window * (window + 1) // 2
    _, e, second = selection(x, window, pol)
    xp = np.pad(x, ((h, h), (h, h), (0, 0), (0, 0)), mode='symmetric')
    yp = np.pad(span(x, pol), ((h, h), (h, h), (0, 0)), mode='symmetric')
    offsets = [(dy, dx) for dy in range(-h, h + 1) for dx in range(-h, h + 1)]        # row-major
    sy = np.zeros(x.shape[:3])
    for dy, dx in offsets:
        sy = np.where(in_mask(e, second, dy, dx), sy + yp[h + dy:h + dy + rows, h + dx:h + dx + cols], sy)
    ybar = sy / n
    vy = np.zeros(x.shape[:3])
    sx = np.zeros(x.shape)
    for dy, dx in offsets:
        inside = in_mask(e, second, dy, dx)
        d = yp[h + dy:h + dy + rows, h + dx:h + dx + cols] - ybar
        vy = np.where(inside, vy + d * d, vy)
        sx = np.where(inside[..., None], sx + xp[h + dy:h + dy + rows, h + dx:h + dx + cols], sx)
    var_y = vy / n
    sv2 = 1.0 / float(looks)
    with np.errstate(invalid='ignore', divide='ignore'):
        var_x = (var_y - (ybar * ybar) * sv2) / (1.0 + sv2)
        b = np.where(var_x > 0, var_x / var_y, 0.0)
    return dict(e=e, second=second, ybar=ybar, var_y=var_y, b=b, M=sx / n)


def refined_lee(values, looks, window=7, pol='dual'):
    """The filtered samples, (rows, cols, k, bands) in the data type of `values`."""
    values = np.asarray(values)
    if window not in WINDOWS or window > min(values.shape[:2]):
        raise ValueError('window %r' % (window,))
    st = statistics(values, looks, window, pol)
    x = values.astype(np.float64)
    M = st['M']
    with np.errstate(invalid='ignore'):
        out = M + st['b'][..., None] * (x - M)
    return out.astype(values.dtype)
