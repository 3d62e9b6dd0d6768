"""TEST INFRASTRUCTURE ONLY -- numpy restatement of the reference's layout post-processing.

Follows inference.py:21-29 (find_N_peaks) and :90-139 (plane, peaks, wall fitting, validity check with the
cuboid fallback, corner assembly), and the misc/post_proc.py functions they call: np_coorx2u :22, np_coory2v :26,
np_coor2xy :30-40, np_x_u_solve_y :43-45, np_y_u_solve_x :48-50, np_xy2coor :53-66, mean_percentile :69-72,
vote :75-98, np_refine_by_fix_z :109-123, infer_coory :126-131, get_gpid :134-139, gen_ww_cuboid :205-238,
gen_ww_general :241-334, gen_ww :337-359.  Pinned by tests/golden/layout.npz (minted from the real reference's
``inference()`` by tests/golden/make_golden_layout.py).

Two additions the reference does not have:
  * ``vote_fast``: the O(n) two-pointer form of ``vote`` (the O(n^2) masked argmax reduces to "widest window of
    the sorted segment whose spread is within tol, leftmost first"); tests prove it equal to ``vote``.
  * ``ring_is_valid``: an exact simple-ring predicate standing in for shapely's ``Polygon(xy2d).is_valid`` on the
    float32 vertices (rational arithmetic via fractions.Fraction)."""
from fractions import Fraction

import numpy as np
from scipy.ndimage import maximum_filter

PI = float(np.pi)
STATUS_OK, STATUS_ASSERT, STATUS_RING = 0, 1, 2


# ------------------------------------------------------------------------------------------ inference.py:21-29
def find_n_peaks(signal, r=29, min_v=0.05, N=None):
    max_v = maximum_filter(signal, size=r, mode='wrap')
    pk_loc = np.where(max_v == signal)[0]
    pk_loc = pk_loc[signal[pk_loc] > min_v]                  # float32 vs python float: NEP 50 compares in float32
    if N is not None:
        order = np.lexsort((pk_loc, -signal[pk_loc]))        # argsort(-value); ties (excluded by the corpora) by column
        pk_loc = pk_loc[order[:N]]
        pk_loc = pk_loc[np.argsort(pk_loc)]
    return pk_loc, signal[pk_loc]


# ------------------------------------------------------------------------------------------ post_proc.py
def np_coorx2u(coorx, coorW=1024):
    return ((coorx + 0.5) / coorW - 0.5) * 2 * PI


def np_coory2v(coory, coorH=512):
    return -((coory + 0.5) / coorH - 0.5) * PI


def np_coor2xy(coor, z=50, coorW=1024, coorH=512, floorW=1024, floorH=512):
    coor = np.array(coor)
    u = np_coorx2u(coor[:, 0], coorW)
    v = np_coory2v(coor[:, 1], coorH)
    c = z / np.tan(v)
    x = c * np.sin(u) + floorW / 2 - 0.5
    y = -c * np.cos(u) + floorH / 2 - 0.5
    return np.hstack([x[:, None], y[:, None]])


def np_x_u_solve_y(x, u, floorW=1024, floorH=512):
    c = (x - floorW / 2 + 0.5) / np.sin(u)
    return -c * np.cos(u) + floorH / 2 - 0.5


def np_y_u_solve_x(y, u, floorW=1024, floorH=512):
    c = -(y - floorH / 2 + 0.5) / np.cos(u)
    return c * np.sin(u) + floorW / 2 - 0.5


def np_xy2coor(xy, z=50, coorW=1024, coorH=512, floorW=1024, floorH=512):
    x = xy[:, 0] - floorW / 2 + 0.5
    y = xy[:, 1] - floorH / 2 + 0.5
    u = np.arctan2(x, -y)
    v = np.arctan(z / np.sqrt(x ** 2 + y ** 2))
    coorx = (u / (2 * PI) + 0.5) * coorW - 0.5
    coory = (-v / PI + 0.5) * coorH - 0.5
    return np.hstack([coorx[:, None], coory[:, None]])


def mean_percentile(vec, p1=25, p2=75):
    vmin = np.percentile(vec, p1)
    vmax = np.percentile(vec, p2)
    return vec[(vmin <= vec) & (vec <= vmax)].mean()


def vote(vec, tol):
    """post_proc.py:75-98 as written: O(n^2) masks over all (row, col) pairs of the sorted segment."""
    vec = np.sort(vec)
    n = np.arange(len(vec))[::-1]
    n = n[:, None] - n[None, :] + 1.0
    d = np.abs(vec[:, None] - vec[None, :]) + 1e-9            # squareform(pdist(.., p=1) + 1e-9): diagonal stays 0
    np.fill_diagonal(d, 0.0)
    invalid = (n < len(vec) * 0.4) | (d > tol)
    if (~invalid).sum() == 0 or len(vec) < tol:
        best_fit = np.median(vec)
        p_score = 0
    else:
        n[invalid] = -1
        max_idx = n.argmax()
        max_row = max_idx // len(vec)
        max_col = max_idx % len(vec)
        assert max_col > max_row
        best_fit = vec[max_row:max_col + 1].mean()
        p_score = (max_col - max_row + 1) / len(vec)
    l1_score = np.abs(vec - best_fit).mean()
    return best_fit, p_score, l1_score


def vote_fast(vec, tol):
    """``vote`` in O(n) after the sort.  Row i of the mask is valid exactly for the columns i..J(i), J(i) the last
    column whose distance (+1e-9 off the diagonal) is within tol (J is non-decreasing in i), and n = j - i + 1.  So the
    first row-major maximum is the widest such window, leftmost on ties, when it reaches 0.4 * len."""
    vec = np.sort(vec)
    L = len(vec)
    best_i, best_w = -1, -1
    j = 0
    for i in range(L):
        j = max(j, i)
        while j + 1 < L and (vec[j + 1] - vec[i]) + 1e-9 <= tol:
            j += 1
        w = j - i + 1
        if w >= L * 0.4 and w > best_w:
            best_i, best_w = i, w
    if best_w < 0 or L < tol:
        best_fit = np.median(vec)
        p_score = 0
    else:
        assert best_w > 1                                     # vote's `assert max_col > max_row`
        best_fit = vec[best_i:best_i + best_w].mean()
        p_score = best_w / L
    l1_score = np.abs(vec - best_fit).mean()
    return best_fit, p_score, l1_score


def np_refine_by_fix_z(coory0, coory1, z0=50, coorH=512):
    v0 = np_coory2v(coory0, coorH)
    v1 = np_coory2v(coory1, coorH)
    c0 = z0 / np.tan(v0)
    z1 = c0 * np.tan(v1)
    z1_mean = mean_percentile(z1)
    v1_refine = np.arctan2(z1_mean, c0)
    coory1_refine = (-v1_refine / PI + 0.5) * coorH - 0.5
    return coory1_refine, z1_mean


def infer_coory(coory0, h, z0=50, coorH=512):
    v0 = np_coory2v(coory0, coorH)
    c0 = z0 / np.tan(v0)
    z1 = z0 + h
    v1 = np.arctan2(z1, c0)
    return (-v1 / PI + 0.5) * coorH - 0.5


def get_gpid(coorx, coorW):
    gpid = np.zeros(coorW)
    gpid[np.round(coorx).astype(int)] = 1
    gpid = np.cumsum(gpid).astype(int)
    gpid[gpid == gpid[-1]] = 0
    return gpid


def gen_ww_cuboid(xy, gpid, tol, vote_fn=vote):
    xy_cor = []
    assert len(np.unique(gpid)) == 4
    for j in range(4):
        new_x, x_score, x_l1 = vote_fn(xy[gpid == j, 0], tol)
        new_y, y_score, y_l1 = vote_fn(xy[gpid == j, 1], tol)
        if (x_score, -x_l1) > (y_score, -y_l1):
            xy_cor.append({'type': 0, 'val': new_x, 'score': x_score})
        else:
            xy_cor.append({'type': 1, 'val': new_y, 'score': y_score})
    scores = [0, 0]                                           # sanity fallback, :220-236 (types only; vals kept)
    for j in range(4):
        scores[j % 2] += xy_cor[j]['score'] if xy_cor[j]['type'] == 0 else -xy_cor[j]['score']
    types = (0, 1, 0, 1) if scores[0] > scores[1] else (1, 0, 1, 0)
    for j in range(4):
        xy_cor[j]['type'] = types[j]
    return xy_cor


def gen_ww_general(init_coorx, xy, gpid, tol, vote_fn=vote, events=None):
    """:241-334; ``events`` (a set) collects the loop's actions: 'requeue', 'forced_infer', 'forced_change',
    'insert'."""
    events = set() if events is None else events
    xy_cor = []
    K = len(init_coorx)
    assert K == len(np.unique(gpid))
    for j in range(K):
        new_x, x_score, x_l1 = vote_fn(xy[gpid == j, 0], tol)
        new_y, y_score, y_l1 = vote_fn(xy[gpid == j, 1], tol)
        u0 = np_coorx2u(init_coorx[(j - 1 + K) % K])
        u1 = np_coorx2u(init_coorx[j])
        if (x_score, -x_l1) > (y_score, -y_l1):
            xy_cor.append({'type': 0, 'val': new_x, 'score': x_score, 'gpid': j, 'u0': u0, 'u1': u1, 'tbd': True})
        else:
            xy_cor.append({'type': 1, 'val': new_y, 'score': y_score, 'gpid': j, 'u0': u0, 'u1': u1, 'tbd': True})
    while True:
        tbd = -1
        for i in range(len(xy_cor)):
            if xy_cor[i]['tbd'] and (tbd == -1 or xy_cor[i]['score'] > xy_cor[tbd]['score']):
                tbd = i
        if tbd == -1:
            break
        xy_cor[tbd]['tbd'] = False
        p_idx = (tbd - 1 + len(xy_cor)) % len(xy_cor)
        n_idx = (tbd + 1) % len(xy_cor)
        num_tbd_neighbor = xy_cor[p_idx]['tbd'] + xy_cor[n_idx]['tbd']
        if num_tbd_neighbor == 2:
            continue
        if num_tbd_neighbor == 1:
            if (not xy_cor[p_idx]['tbd'] and xy_cor[p_idx]['type'] == xy_cor[tbd]['type']) or \
                    (not xy_cor[n_idx]['tbd'] and xy_cor[n_idx]['type'] == xy_cor[tbd]['type']):
                if xy_cor[tbd]['score'] >= -1:
                    xy_cor[tbd]['tbd'] = True                 # :284-287 re-queue
                    xy_cor[tbd]['score'] -= 100
                    events.add('requeue')
                else:
                    if not xy_cor[p_idx]['tbd']:
                        insert_at = tbd
                        if xy_cor[p_idx]['type'] == 0:
                            new_val, new_type = np_x_u_solve_y(xy_cor[p_idx]['val'], xy_cor[p_idx]['u1']), 1
                        else:
                            new_val, new_type = np_y_u_solve_x(xy_cor[p_idx]['val'], xy_cor[p_idx]['u1']), 0
                    else:
                        insert_at = n_idx
                        if xy_cor[n_idx]['type'] == 0:
                            new_val, new_type = np_x_u_solve_y(xy_cor[n_idx]['val'], xy_cor[n_idx]['u0']), 1
                        else:
                            new_val, new_type = np_y_u_solve_x(xy_cor[n_idx]['val'], xy_cor[n_idx]['u0']), 0
                    xy_cor.insert(insert_at, {'type': new_type, 'val': new_val, 'score': 0, 'gpid': -1,
                                              'u0': -1, 'u1': -1, 'tbd': False})
                    events.add('forced_infer')
            continue
        if xy_cor[p_idx]['type'] == xy_cor[n_idx]['type']:
            if xy_cor[tbd]['type'] == xy_cor[p_idx]['type']:  # :313-317 forced change
                xy_cor[tbd]['type'] = (xy_cor[tbd]['type'] + 1) % 2
                xy_cor[tbd]['val'] = xy[gpid == xy_cor[tbd]['gpid'], xy_cor[tbd]['type']].mean()
                events.add('forced_change')
        else:                                                 # :318-332 two inferred walls replace this one
            tp0 = xy_cor[n_idx]['type']
            tp1 = xy_cor[p_idx]['type']
            if xy_cor[p_idx]['type'] == 0:
                val0 = np_x_u_solve_y(xy_cor[p_idx]['val'], xy_cor[p_idx]['u1'])
                val1 = np_y_u_solve_x(xy_cor[n_idx]['val'], xy_cor[n_idx]['u0'])
            else:
                val0 = np_y_u_solve_x(xy_cor[p_idx]['val'], xy_cor[p_idx]['u1'])
                val1 = np_x_u_solve_y(xy_cor[n_idx]['val'], xy_cor[n_idx]['u0'])
            new_add = [{'type': tp0, 'val': val0, 'score': 0, 'gpid': -1, 'u0': -1, 'u1': -1, 'tbd': False},
                       {'type': tp1, 'val': val1, 'score': 0, 'gpid': -1, 'u0': -1, 'u1': -1, 'tbd': False}]
            xy_cor = xy_cor[:tbd] + new_add + xy_cor[tbd + 1:]
            events.add('insert')
    return xy_cor


def gen_ww(init_coorx, coory, z=50, coorW=1024, coorH=512, floorW=1024, floorH=512, tol=3, force_cuboid=True,
           vote_fn=vote, events=None):
    gpid = get_gpid(init_coorx, coorW)
    coor = np.hstack([np.arange(coorW)[:, None], coory[:, None]])
    xy = np_coor2xy(coor, z, coorW, coorH, floorW, floorH)
    if force_cuboid:
        xy_cor = gen_ww_cuboid(xy, gpid, tol, vote_fn)
    else:
        xy_cor = gen_ww_general(init_coorx, xy, gpid, tol, vote_fn, events)
    cor = []
    for j in range(len(xy_cor)):
        next_j = (j + 1) % len(xy_cor)
        if xy_cor[j]['type'] == 1:
            cor.append((xy_cor[next_j]['val'], xy_cor[j]['val']))
        else:
            cor.append((xy_cor[j]['val'], xy_cor[next_j]['val']))
    cor = np_xy2coor(np.array(cor), z, coorW, coorH, floorW, floorH)
    cor = np.roll(cor, -2 * cor[::2, 0].argmin(), axis=0)
    return cor, xy_cor


# ------------------------------------------------------------------------------------------ validity (:114-120)
def wall_ring(xy_cor):
    """xy2d exactly as inference.py:116-119 builds it (float32; one coordinate stays 0 when two adjacent walls
    share a type)."""
    xy2d = np.zeros((len(xy_cor), 2), np.float32)
    for i in range(len(xy_cor)):
        xy2d[i, xy_cor[i]['type']] = xy_cor[i]['val']
        xy2d[i, xy_cor[i - 1]['type']] = xy_cor[i - 1]['val']
    return xy2d


def _orient(a, b, c):
    d = (b[0] - a[0]) * (c[1] - a[1]) - (b[1] - a[1]) * (c[0] - a[0])
    return (d > 0) - (d < 0)


def _on_segment(a, b, p):                                     # p collinear with a-b: inside the closed box?
    return min(a[0], b[0]) <= p[0] <= max(a[0], b[0]) and min(a[1], b[1]) <= p[1] <= max(a[1], b[1])


def _segments_touch(a, b, c, d):
    o1, o2, o3, o4 = _orient(a, b, c), _orient(a, b, d), _orient(c, d, a), _orient(c, d, b)
    if o1 != o2 and o3 != o4 and o1 * o2 <= 0 and o3 * o4 <= 0:
        if o1 != 0 or o2 != 0:
            return True
    return ((o1 == 0 and _on_segment(a, b, c)) or (o2 == 0 and _on_segment(a, b, d)) or
            (o3 == 0 and _on_segment(c, d, a)) or (o4 == 0 and _on_segment(c, d, b)))


def ring_is_valid(xy2d):
    """Exact simple-ring test on float32 vertices (rational arithmetic): repeated consecutive vertices are dropped,
    at least 3 distinct vertices are needed, non-adjacent edges must not meet at all and adjacent edges must not
    fold back onto each other (a spike).  Raises ValueError for fewer than 3 input vertices, as shapely's
    Polygon() does."""
    if len(xy2d) < 3:
        raise ValueError('A linearring requires at least 4 coordinates.')
    pts = [(Fraction(float(x)), Fraction(float(y))) for x, y in np.asarray(xy2d, np.float32)]
    ring = []
    for p in pts:
        if not ring or ring[-1] != p:
            ring.append(p)
    while len(ring) > 1 and ring[-1] == ring[0]:
        ring.pop()
    n = len(ring)
    if n < 3:
        return False
    edges = [(ring[i], ring[(i + 1) % n]) for i in range(n)]
    for i in range(n):
        for j in range(i + 1, n):
            a, b = edges[i]
            c, d = edges[j]
            if j == i + 1 or (i == 0 and j == n - 1):
                # shared vertex: b == c (j == i+1) or d == a (wrap); spike when the other ends fold back over it
                if j == i + 1:
                    p, q, r = a, b, d
                else:
                    p, q, r = b, a, c
                if _orient(p, q, r) == 0 and ((q[0] - p[0]) * (r[0] - q[0]) + (q[1] - p[1]) * (r[1] - q[1])) < 0:
                    return False
                if n == 3:
                    continue
                continue
            if _segments_touch(a, b, c, d):
                return False
    return True


# ------------------------------------------------------------------------------------------ inference.py:90-139
def decode(y_bon, H=512):
    """inference.py:90-92 on the merged boundary output [2, W] (radians) -> pixel rows, float32."""
    y_bon_ = (y_bon / np.pi + 0.5) * H - 0.5
    y_bon_[0] = np.clip(y_bon_[0], 1, H / 2 - 1)
    y_bon_[1] = np.clip(y_bon_[1], H / 2 + 1, H - 2)
    return y_bon_


def layout(y_bon_, y_cor_, force_cuboid=False, force_raw=False, min_v=None, r=0.05, H=512, W=1024,
           vote_fn=vote, ring_fn=ring_is_valid):
    """inference.py:95-139 on decoded signals (y_bon_ [2, W] float32 pixel rows, y_cor_ [W] float32).  Never
    raises for the reference's own exceptions: returns a dict with 'status' (0 ok, 1 AssertionError, 2 ValueError
    from the ring), 'fallback', 'peaks', 'types', 'vals', 'z1', 'cor_id' and 'events'."""
    y_bon_ = np.asarray(y_bon_, np.float32)
    y_cor_ = np.asarray(y_cor_, np.float32)
    z0 = 50
    _, z1 = np_refine_by_fix_z(*y_bon_, z0)
    out = {'status': STATUS_OK, 'fallback': False, 'peaks': np.zeros(0, np.int64), 'types': np.zeros(0, np.int64),
           'vals': np.zeros(0), 'z1': z1, 'cor_id': np.zeros((0, 2), np.float32), 'events': set()}
    try:
        if force_raw:
            cor = np.stack([np.arange(1024), y_bon_[0]], 1)
        else:
            if min_v is None:
                min_v = 0 if force_cuboid else 0.05
            r = int(round(W * r / 2))
            N = 4 if force_cuboid else None
            xs_ = find_n_peaks(y_cor_, r=r, min_v=min_v, N=N)[0]
            out['peaks'] = xs_
            tol = abs(0.16 * z1 / 1.6)
            cor, xy_cor = gen_ww(xs_, y_bon_[0], z0, tol=tol, force_cuboid=force_cuboid, vote_fn=vote_fn,
                                 events=out['events'])
            if not force_cuboid:
                out['types'] = np.array([c['type'] for c in xy_cor])
                if not ring_fn(wall_ring(xy_cor)):
                    out['fallback'] = True
                    xs_ = find_n_peaks(y_cor_, r=r, min_v=0, N=4)[0]
                    out['peaks'] = xs_
                    cor, xy_cor = gen_ww(xs_, y_bon_[0], z0, tol=tol, force_cuboid=True, vote_fn=vote_fn)
            out['types'] = np.array([c['type'] for c in xy_cor])
            out['vals'] = np.array([c['val'] for c in xy_cor], np.float64)
    except AssertionError:
        out['status'] = STATUS_ASSERT
        return out
    except ValueError:
        out['status'] = STATUS_RING
        return out
    cor = np.hstack([cor, infer_coory(cor[:, 1], z1 - z0, z0)[:, None]])
    cor_id = np.zeros((len(cor) * 2, 2), np.float32)
    for j in range(len(cor)):
        cor_id[j * 2] = cor[j, 0], cor[j, 1]
        cor_id[j * 2 + 1] = cor[j, 0], cor[j, 2]
    cor_id[:, 0] /= W
    cor_id[:, 1] /= H
    out['cor_id'] = cor_id
    return out


def near_tie(y_bon_, y_cor_, **kw):
    """True when the discrete result moves under tiny perturbations (tol by +-1e-5 relative, y_cor by +-1e-6):
    such cases pin rounding, not behaviour, and the corpora drop them."""
    base = layout(y_bon_, y_cor_, **kw)
    key = _discrete(base)
    if not kw.get('force_raw'):                               # top-4 cut between (nearly) equal peak values
        r_px = int(round(1024 * kw.get('r', 0.05) / 2))
        min_vs = [0] + ([kw['min_v']] if kw.get('min_v') is not None else [])
        for mv in min_vs:
            vals = np.sort(find_n_peaks(np.asarray(y_cor_, np.float32), r=r_px, min_v=mv)[1])[::-1]
            if len(vals) > 4 and vals[3] - vals[4] <= 1e-6:
                return True
    for s in (1 + 1e-5, 1 - 1e-5):
        if _discrete(_layout_tol_scaled(y_bon_, y_cor_, s, **kw)) != key:
            return True
    for d in (1e-6, -1e-6):
        if _discrete(layout(y_bon_, np.asarray(y_cor_, np.float32) + np.float32(d), **kw)) != key:
            return True
    return False


def _discrete(o):
    return (o['status'], o['fallback'], tuple(o['peaks'].tolist()), tuple(o['types'].tolist()), len(o['cor_id']))


def _layout_tol_scaled(y_bon_, y_cor_, s, **kw):
    global np_refine_by_fix_z
    orig = np_refine_by_fix_z

    def scaled(*a, **k):
        c, z = orig(*a, **k)
        return c, np.float32(z * s)
    np_refine_by_fix_z = scaled
    try:
        return layout(y_bon_, y_cor_, **kw)
    finally:
        np_refine_by_fix_z = orig
