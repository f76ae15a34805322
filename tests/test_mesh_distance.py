"""Stage-I surface term (SURVEY.md 8(f-2)): point-to-triangle-mesh distance with derivatives.

CPU: the oracle's restatement against the reference header itself (values of the UNMODIFIED
scan2mesh/mesh_distance/sample2meshdist.h compiled against an Eigen stand-in, stored in tests/golden/ref_s2m.npz by
tests/golden/make_reference_vectors.py) and against finite differences.  GPU: the CUDA kernel (C-ABI
mosh2_mesh_distance) against the oracle."""
import os

import numpy as np
import pytest

from oracle import mesh_distance as omd

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _random_case(rng):
    a, b, c = rng.normal(0, 0.3, (3, 3))
    x = (a + b + c) / 3 + rng.normal(0, 0.2, 3)
    return x, a, b, c


def test_oracle_tri_equals_reference_header():
    """Every part (plane, three edges, three vertices) under the three robustifiers: value and all four gradients."""
    g = np.load(os.path.join(ROOT, 'tests', 'golden', 'ref_s2m.npz'))
    assert g['xabc'].shape[0] == 40 and len(g['kinds']) == 4
    for trial, (x, a, b, c) in enumerate(g['xabc']):
        for k, (kind, sigma) in enumerate(g['kinds']):
            for part in range(7):
                ref = (g['value'][trial, k, part], *g['grad'][trial, k, part])
                got = omd.tri(part, x, a, b, c, int(kind), float(sigma))
                assert abs(got[0] - ref[0]) <= 1e-12 * max(1.0, abs(ref[0]))
                for gr, r in zip(got[1:], ref[1:]):
                    assert np.abs(gr - r).max() <= 1e-10 * max(1.0, np.abs(r).max()), (kind, part)


def test_oracle_gradients_are_derivatives():
    rng = np.random.default_rng(11)
    for trial in range(10):
        x, a, b, c = _random_case(rng)
        for kind, sigma in ((omd.KIND_SQUARED, 1.0), (omd.KIND_GM, 0.1)):
            for part in range(7):
                v, dx, da, db, dc = omd.tri(part, x, a, b, c, kind, sigma)
                for which, g in enumerate((dx, da, db, dc)):
                    num = np.zeros(3)
                    for k in range(3):
                        args = [x.copy(), a.copy(), b.copy(), c.copy()]
                        args[which][k] += 1e-6
                        vp = omd.tri(part, *args, kind, sigma)[0]
                        args[which][k] -= 2e-6
                        vm = omd.tri(part, *args, kind, sigma)[0]
                        num[k] = (vp - vm) / 2e-6
                    assert np.abs(num - g).max() < 1e-6 * max(1.0, np.abs(g).max())


def test_nearest_part_is_consistent_with_the_distance():
    """The brute-force query returns the triangle / part whose closed-form distance (of that part) is the minimum over all
    triangles -- what the AABB tree of the reference returns (mesh_distance_main.py:358-376)."""
    rng = np.random.default_rng(3)
    verts = rng.normal(0, 0.3, (60, 3))
    faces = rng.integers(0, 60, (150, 3))
    faces = faces[(faces[:, 0] != faces[:, 1]) & (faces[:, 1] != faces[:, 2]) & (faces[:, 0] != faces[:, 2])]
    # an isolated triangle far from the soup, with samples beyond its corners and edges: vertex and edge parts for sure
    verts = np.concatenate([verts, [[10, 0, 0], [11, 0, 0], [10, 1, 0]]])
    faces = np.concatenate([faces, [[60, 61, 62]]])
    corner = np.array([[9.5, -0.5, 0.2], [11.8, -0.3, 0.1], [9.7, 1.9, -0.2], [10.5, -0.7, 0.1], [11.0, 1.0, 0.3], [9.2, 0.5, 0.0]])
    samples = np.concatenate([rng.normal(0, 0.35, (50, 3)), corner])
    r, dsample, dref, t, p = omd.somedistance(samples, verts, faces, omd.KIND_DISTANCE)
    assert p[-6:].tolist() == [4, 5, 6, 1, 2, 3] and (t[-6:] == len(faces) - 1).all()
    parts = set(np.unique(p).tolist())
    assert 0 in parts and parts & {1, 2, 3} and parts & {4, 5, 6}      # interior, edge and vertex cases all occur
    for s in range(len(samples)):
        a, b, c = (verts[faces[t[s], k]] for k in range(3))
        assert abs(abs(r[s]) - abs(omd.tri(int(p[s]), samples[s], a, b, c)[0])) < 1e-12
        A, B, Cc = verts[faces[:, 0]], verts[faces[:, 1]], verts[faces[:, 2]]
        d2, _ = omd.closest_on_triangles(samples[s], A, B, Cc)
        assert abs(np.sqrt(d2.min()) - abs(r[s])) < 1e-9
        assert np.abs(dsample[s] + dref[s].reshape(3, 3).sum(0)).max() < 1e-9      # translation invariance


@pytest.mark.gpu
@pytest.mark.parametrize('kind,sigma', [(omd.KIND_DISTANCE, 1.0), (omd.KIND_SQUARED, 1.0), (omd.KIND_GM, 0.05)])
def test_cuda_mesh_distance_equals_oracle(kind, sigma):
    from moshpp_b200 import mesh_distance as md
    rng = np.random.default_rng(5)
    V, T, S = 700, 1300, 333
    verts = rng.normal(0, 0.3, (V, 3))
    faces = rng.integers(0, V, (T, 3)).astype(np.int32)
    faces = faces[(faces[:, 0] != faces[:, 1]) & (faces[:, 1] != faces[:, 2]) & (faces[:, 0] != faces[:, 2])]
    samples = np.concatenate([rng.normal(0, 0.35, (S - 20, 3)), verts[:10] + 1e-3, verts[faces[:10]].mean(1)])
    out = md.mesh_distance(samples, verts, faces, kind=kind, sigma=sigma)
    r, dsample, dref, t, p = omd.somedistance(samples, verts, faces, kind, sigma)
    # the search runs in float32: a different triangle may win a tie within round-off -- the value must still agree
    same = (out['tri'] == t) & (out['part'] == p)
    assert same.mean() > 0.97
    assert np.abs(np.abs(out['value']) - np.abs(r)).max() < 1e-5 * max(1.0, np.abs(r).max())
    assert np.abs(out['value'][same] - r[same]).max() < 1e-12 * max(1.0, np.abs(r).max())
    assert np.abs(out['d_sample'][same] - dsample[same]).max() < 1e-9 * max(1.0, np.abs(dsample).max())
    assert np.abs(out['d_tri'][same] - dref[same]).max() < 1e-9 * max(1.0, np.abs(dref).max())
    # with the nearest (triangle, part) given -- what the reference's somedistance takes -- everything is exact
    out2 = md.mesh_distance(samples, verts, faces, kind=kind, sigma=sigma, nearest_tri=t, nearest_part=p)
    assert np.abs(out2['value'] - r).max() < 1e-12 * max(1.0, np.abs(r).max())
    assert np.abs(out2['d_tri'] - dref).max() < 1e-9 * max(1.0, np.abs(dref).max())
    Dr_ref, Dr_sample = md.as_sparse(out2, faces, V)
    assert Dr_ref.shape == (len(samples), 3 * V) and Dr_sample.shape == (len(samples), 3 * len(samples))
    assert np.allclose(np.asarray(Dr_sample.sum(1)).ravel(), dsample.sum(1), atol=1e-9)
