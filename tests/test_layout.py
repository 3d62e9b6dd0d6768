"""CPU: the layout oracle (oracle/layout_ref.py) reproduces tests/golden/layout.npz, minted from the real reference's
inference(); the O(n) vote equals post_proc.vote's O(n^2) definition; the exact ring predicate equals shapely's
Polygon.is_valid where shapely imports."""
import os

import numpy as np
import pytest

from oracle import layout_ref


def golden_cases(golden_dir):
    """One dict per case of layout.npz (ragged arrays split by the n_* counts)."""
    g = np.load(os.path.join(golden_dir, 'layout.npz'))
    cases = []
    op = ow = oc = 0
    for i in range(len(g['sig'])):
        npk, nw, nc = int(g['n_peaks'][i]), int(g['n_walls'][i]), int(g['n_cor'][i])
        kw = dict(force_cuboid=bool(g['force_cuboid'][i]), force_raw=bool(g['force_raw'][i]), r=float(g['r'][i]),
                  min_v=None if np.isnan(g['min_v'][i]) else float(g['min_v'][i]))
        cases.append(dict(y_bon=g['y_bon'][g['sig'][i]], y_cor=g['y_cor'][g['sig'][i]], kw=kw,
                          status=int(g['status'][i]), fallback=bool(g['fallback'][i]), z1=float(g['z1'][i]),
                          peaks=g['peaks'][op:op + npk], types=g['types'][ow:ow + nw], cor_id=g['cor_id'][oc:oc + nc]))
        op, ow, oc = op + npk, ow + nw, oc + nc
    return cases


def test_golden_corpus_covers_every_branch(golden_dir):
    cases = golden_cases(golden_dir)
    assert len(cases) >= 120
    assert os.path.getsize(os.path.join(golden_dir, 'layout.npz')) < 1 << 20
    assert any(c['kw']['force_cuboid'] for c in cases) and any(c['kw']['force_raw'] for c in cases)
    assert any(c['fallback'] for c in cases)
    assert any(c['status'] == layout_ref.STATUS_ASSERT for c in cases)
    assert any(c['kw']['min_v'] is not None for c in cases)
    assert {int(round(1024 * c['kw']['r'] / 2)) % 2 for c in cases} == {0, 1}
    events = set()
    for c in cases:
        if not (c['kw']['force_cuboid'] or c['kw']['force_raw']):
            events |= layout_ref.layout(c['y_bon'], c['y_cor'], **c['kw'])['events']
    assert {'requeue', 'forced_infer', 'forced_change', 'insert'} <= events


@pytest.mark.parametrize('vote_fn', [layout_ref.vote, layout_ref.vote_fast], ids=['vote', 'vote_fast'])
def test_oracle_reproduces_golden(golden_dir, vote_fn):
    for i, c in enumerate(golden_cases(golden_dir)):
        o = layout_ref.layout(c['y_bon'], c['y_cor'], vote_fn=vote_fn, **c['kw'])
        assert o['status'] == c['status'] and o['fallback'] == c['fallback'], i
        assert abs(float(o['z1']) - c['z1']) <= 1e-6 * abs(c['z1']), i
        if c['status']:
            continue
        if not c['kw']['force_raw']:
            np.testing.assert_array_equal(o['peaks'], c['peaks'], err_msg=str(i))
            np.testing.assert_array_equal(o['types'], c['types'], err_msg=str(i))
        assert o['cor_id'].shape == c['cor_id'].shape, i
        assert np.abs(o['cor_id'] - c['cor_id']).max() <= 1e-6, i


def _tie_vectors():
    rs = np.random.RandomState(11)
    for k in range(400):
        n = int(rs.randint(1, 90))
        kind = k % 4
        if kind == 0:                                   # few distinct values: heavy ties
            v = rs.randint(0, 6, n).astype(np.float64) * rs.choice([0.5, 1.0, 3.0])
        elif kind == 1:                                 # values on a grid that meets tol (+1e-9) exactly
            v = np.round(rs.uniform(0, 20, n)) * 0.25
        elif kind == 2:
            v = rs.normal(100, 5, n)
        else:
            v = np.concatenate([np.full(n // 2 + 1, 7.0), rs.uniform(0, 30, n)])
        tol = float(np.float32(rs.choice([0.5, 1.0, 2.0, 3.0, 5.0, 8.0, 12.0, 40.0])))
        yield v, tol


def test_vote_fast_equals_quadratic_definition():
    checked = 0
    for v, tol in _tie_vectors():
        try:
            ref = layout_ref.vote(v, tol)
        except AssertionError:
            with pytest.raises(AssertionError):
                layout_ref.vote_fast(v, tol)
            continue
        got = layout_ref.vote_fast(v, tol)
        assert got[1] == ref[1]
        assert got[0] == ref[0] and got[2] == ref[2]
        checked += 1
    assert checked > 300


RINGS = {
    'square': ([[0, 0], [4, 0], [4, 4], [0, 4]], True),
    'L': ([[0, 0], [4, 0], [4, 2], [2, 2], [2, 4], [0, 4]], True),
    'bowtie': ([[0, 0], [4, 4], [4, 0], [0, 4]], False),
    'vertex_touch': ([[0, 0], [4, 0], [2, 2], [4, 4], [0, 4], [2, 2]], False),
    'spike': ([[0, 0], [4, 0], [4, 4], [4, 6], [4, 4], [0, 4]], False),
    'spike_back': ([[0, 0], [6, 0], [4, 0], [4, 4]], False),
    'duplicates': ([[0, 0], [0, 0], [4, 0], [4, 4], [4, 4], [0, 4], [0, 0]], True),
    'collinear': ([[0, 0], [2, 0], [4, 0], [4, 4], [0, 4]], True),
    'degenerate': ([[0, 0], [1, 1], [2, 2]], False),
    'two_distinct': ([[0, 0], [1, 1], [1, 1]], False),
    'edge_touch': ([[0, 0], [6, 0], [6, 4], [3, 4], [3, 0.0], [0, 4]], False),
}


def random_rings(n, seed):
    rs = np.random.RandomState(seed)
    out = []
    for _ in range(n):
        k = int(rs.randint(3, 12))
        pts = rs.randint(0, 5, (k, 2)).astype(np.float32) if rs.rand() < 0.5 else \
            rs.uniform(-300, 300, (k, 2)).astype(np.float32)
        out.append(pts)
    return out


def test_ring_predicate_on_constructed_rings():
    for name, (pts, valid) in RINGS.items():
        assert layout_ref.ring_is_valid(np.array(pts, np.float32)) == valid, name
    with pytest.raises(ValueError):
        layout_ref.ring_is_valid(np.zeros((2, 2), np.float32))


def test_ring_predicate_equals_shapely():
    shapely_geometry = pytest.importorskip('shapely.geometry')
    rings = [np.array(p, np.float32) for p, _ in RINGS.values()] + random_rings(300, 5)
    for pts in rings:
        assert layout_ref.ring_is_valid(pts) == shapely_geometry.Polygon(pts).is_valid, pts.tolist()
