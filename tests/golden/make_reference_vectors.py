"""Generates tests/golden/ref_*.npz from the parts of the UNMODIFIED reference that import in this container
(everything on the Stage-II path that needs chumpy / psbody / ezc3d does not, SURVEY.md 8(c)):

  * moshpp.rigid_transformations (numpy, scipy, cv2 only): `rigid_landmark_transform`, `perform_rigid_adjustment`
    -- the first-frame rigid adjustment, row a9 of SURVEY.md section 8, chmosh.py:634;
  * moshpp.tools.c3d: header / parameter parsing of a c3d file written by moshpp_b200.c3d_io (row f-1).  Its frame
    reader raises OverflowError under numpy 2 (`int32 & 0x80008000`), so only the metadata is pinned.

  * moshpp.prior.gmm_prior_ch and moshpp.transformed_lm (rows a5, a6, a7) need `chumpy` only as an array container with
    a calling convention: they import against the forward-only stand-in tests/golden/ref_shim (chumpy, plus the one helper
    of human_body_prior they use) and then run UNMODIFIED: `create_gmm_body_prior` (weights normalisation, Cholesky factors),
    `MaxMixtureComplete` (arg-min component, residual), `TransformedCoeffs` (8-NN attachment incl. the SMPL-X eyeball
    exclusion and the collinear-neighbour fallback) and `TransformedLms` (simulated markers on posed vertices)
    -> ref_prior.npz, ref_lms.npz.

  * scan2mesh/mesh_distance/sample2meshdist.h (row f-2), compiled unmodified by oracle/build_ref.py: the
    point-to-triangle distance and its gradients -> ref_s2m.npz.

The vectors travel with the repository; /root/reference is needed only to regenerate them:

    python tests/golden/make_reference_vectors.py
"""
import os
import sys
import tempfile
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = '/root/reference/src'
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)


def main():
    from moshpp import rigid_transformations as ref_rigid      # the reference, unmodified
    from moshpp.tools import c3d as ref_c3d
    from moshpp_b200 import c3d_io

    rng = np.random.default_rng(20240924)
    cases = []
    for k in range(12):
        m = int(rng.integers(3, 60))
        sim = rng.normal(0, 0.4, (m, 3)) + rng.normal(0, 1.0, 3)
        rv = rng.normal(0, 1.0, 3) * (3.0 if k % 4 == 0 else 0.7)        # some large rotations
        import cv2
        R = cv2.Rodrigues(rv)[0]
        obs = sim @ R.T + rng.normal(0, 1.0, 3) + rng.normal(0, 0.003, (m, 3))
        if k == 5:                      # reflection-prone: nearly planar, noisy
            sim[:, 2] *= 1e-3
            obs = sim @ R.T + rng.normal(0, 0.05, (m, 3))
        if k == 7:                      # NaN rows of the observation are replaced by the simulated ones (line 52)
            obs[1] = np.nan
        R_ref, T_ref = ref_rigid.rigid_landmark_transform(sim.T, obs.T)
        poses, trans = [np.zeros(9)], [np.zeros(3)]
        ref_rigid.perform_rigid_adjustment(poses, trans, [None], [np.where(np.isnan(obs), sim, obs)], [sim])
        cases.append(dict(sim=sim, obs=obs, R=R_ref, T=T_ref.ravel(), rv=poses[0][:3].copy(), trans=trans[0].copy()))
    np.savez_compressed(os.path.join(HERE, 'ref_rigid.npz'),
                        **{f'{k}_{i}': v for i, c in enumerate(cases) for k, v in c.items()}, n=np.array(len(cases)))
    print('ref_rigid.npz:', len(cases), 'cases')

    d = tempfile.mkdtemp(prefix='mosh_refc3d_')
    F, L = 9, 6
    data = rng.normal(0, 500, (F, L, 3))
    data[2, 1] = np.nan
    labels = ['LFHD', 'RFHD', 'C7', 'T10', '*12', 'EXTRA1']
    fn = os.path.join(d, 'written_by_c3d_io.c3d')
    c3d_io.write_c3d(fn, data, labels, frame_rate=120.0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        with open(fn, 'rb') as h:
            r = ref_c3d.Reader(h)
            meta = dict(point_rate=np.array(r.point_rate), point_scale=np.array(r.point_scale),
                        point_used=np.array(r.point_used), first_frame=np.array(r.first_frame),
                        last_frame=np.array(r.last_frame), labels=np.array([s.strip() for s in r.point_labels]))
    with open(fn, 'rb') as h:
        blob = np.frombuffer(h.read(), dtype=np.uint8)
    # the same content in the DEC and the SGI/MIPS processor formats: header and parameters as the reference's parser
    # reads them (tools/c3d.py:35-100,368-424), and the reference's own DEC -> IEEE conversion of random DEC numbers
    extra = {}
    for proc in ('dec', 'mips'):
        fnp = os.path.join(d, f'written_{proc}.c3d')
        c3d_io.write_c3d(fnp, data, labels, frame_rate=120.0, processor=proc)
        with warnings.catch_warnings():
            warnings.simplefilter('ignore')
            with open(fnp, 'rb') as h:
                r = ref_c3d.Reader(h)
                extra[f'{proc}_point_rate'] = np.array(r.point_rate)
                extra[f'{proc}_point_scale'] = np.array(r.point_scale)
                extra[f'{proc}_point_used'] = np.array(r.point_used)
                extra[f'{proc}_first_frame'] = np.array(r.first_frame)
                extra[f'{proc}_last_frame'] = np.array(r.last_frame)
                extra[f'{proc}_labels'] = np.array([s.strip() for s in r.point_labels])
        with open(fnp, 'rb') as h:
            extra[f'{proc}_file_bytes'] = np.frombuffer(h.read(), dtype=np.uint8)
    vals = np.concatenate([rng.normal(0, 800, 400), rng.normal(0, 1e-3, 50), [0.0, 1.0, -1.0, 0.5, 1234.5]]).astype(np.float32)
    dec_bytes = np.frombuffer(c3d_io.ieee_to_dec(vals), dtype=np.uint8)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        extra['dec_bytes'] = dec_bytes
        extra['dec_as_ieee_by_reference'] = np.array(ref_c3d.DEC_to_IEEE_BYTES(dec_bytes.tobytes()), dtype=np.float32)
        extra['dec_scalar_by_reference'] = np.array([ref_c3d.DEC_to_IEEE(int(u)) for u in dec_bytes.view('<u4')[:64]], dtype=np.float32)
    np.savez_compressed(os.path.join(HERE, 'ref_c3d.npz'), file_bytes=blob, data=data, in_labels=np.array(labels), **meta, **extra)
    print('ref_c3d.npz:', {k: (v.tolist() if v.size < 8 else v.shape) for k, v in {**meta, **extra}.items()})


def prior_and_marker_vectors():
    """Rows a5-a7 from the unmodified reference files over the chumpy stand-in."""
    import pickle
    sys.path.insert(0, os.path.join(HERE, 'ref_shim'))
    import chumpy as ch                                             # the stand-in
    assert 'ref_shim' in ch.__file__
    from moshpp.prior import gmm_prior_ch as ref_prior              # the reference, unmodified
    from moshpp import transformed_lm as ref_lm
    from moshpp_b200 import synth

    rng = np.random.default_rng(20240925)
    d = tempfile.mkdtemp(prefix='mosh_refprior_')
    fn = os.path.join(d, 'pose_body_prior.pkl')
    gmm = synth.make_body_prior()
    with open(fn, 'wb') as f:
        pickle.dump(gmm, f)
    out = dict(covars=gmm['covars'], means=gmm['means'], weights=gmm['weights'])
    for tag, excl in (('63', True), ('69', False)):
        wrap = ref_prior.create_gmm_body_prior(fn, exclude_hands=excl)
        D = 63 if excl else 69
        K = len(wrap.means)
        xs = np.concatenate([rng.normal(0, 0.25, (10, D)), wrap.means[:K] + rng.normal(0, 0.02, (K, D))])
        rs, ks = [], []
        for x in xs:
            mm = wrap(ch.Ch(x))                                     # MaxMixtureComplete(x=..., means, precs, weights)
            rs.append(np.asarray(mm.r))
            ks.append(int(mm.min_component_idx))
        out.update({f'x_{tag}': xs, f'r_{tag}': np.array(rs), f'k_{tag}': np.array(ks),
                    f'chols_{tag}': np.asarray(wrap.precs.r), f'weights_{tag}': np.asarray(wrap.weights.r),
                    f'means_{tag}': np.asarray(wrap.means)})
        assert len(set(ks)) > 2, 'the probe points should select several mixture components'
    np.savez_compressed(os.path.join(HERE, 'ref_prior.npz'), **out)
    print('ref_prior.npz: components picked', sorted(set(out['k_63'].tolist())), sorted(set(out['k_69'].tolist())))

    eyeballs = ref_lm.TransformedCoeffs.no_eye_ball_vids
    assert eyeballs == list(range(len(eyeballs))) and len(eyeballs) == 9383      # the eyeballs are the tail block
    cases = {}
    for tag, V in (('smplh', 6890), ('smplx', 10475), ('line', 400)):
        can = rng.normal(0, 0.35, (V, 3))
        M = 40
        vids = rng.choice(V if tag != 'smplx' else 9383, M, replace=False)
        mk = can[vids] + rng.normal(0, 0.01, (M, 3))
        if tag == 'smplx':          # eyeball vertices sitting right on top of some markers: they must be skipped
            can[9383:9383 + 20] = mk[:20] + 1e-4
        if tag == 'line':           # the three nearest vertices of marker 0 are collinear: the third neighbour is swapped
            p0 = mk[0] + np.array([0.002, 0.0, 0.0])
            far = np.linalg.norm(can - mk[0], axis=1) < 0.06
            can[far] += 1.0
            can[0], can[1], can[2], can[3] = p0, p0 + [0.001, 0, 0], p0 + [0.0021, 0, 0], p0 + [0.0, 0.004, 0.001]
        tc = ref_lm.TransformedCoeffs(can_body=can.copy(), markers_latent=mk.copy())
        coefs = np.asarray(tc.r)
        posed = can + rng.normal(0, 0.02, can.shape)               # any other vertex positions: the "posed" body
        lms = ref_lm.TransformedLms(transformed_coeffs=tc, can_body=ch.Ch(posed))
        cases.update({f'can_{tag}': can, f'markers_latent_{tag}': mk, f'closest_{tag}': np.asarray(tc.closest),
                      f'coefs_{tag}': coefs, f'posed_{tag}': posed, f'markers_{tag}': np.asarray(lms.r)})
        # canonical pose: the attachment reproduces the latent markers
        back = ref_lm.TransformedLms(transformed_coeffs=tc, can_body=ch.Ch(can))
        assert np.abs(np.asarray(back.r) - mk).max() < 1e-9
    assert (cases['closest_smplx'] < 9383).all()
    np.savez_compressed(os.path.join(HERE, 'ref_lms.npz'), **cases)
    print('ref_lms.npz:', {k: v.shape for k, v in cases.items() if k.startswith('closest')})


def mesh_distance_vectors():
    """Row f-2: the point-to-triangle distance of scan2mesh/mesh_distance/sample2meshdist.h, UNMODIFIED, compiled against
    the Eigen stand-in (oracle/build_ref.py): value and the four gradients of every part (plane, three edges, three
    vertices) under the three robustifiers on 40 random (sample, triangle) cases -> ref_s2m.npz."""
    import ctypes as C
    from oracle import build_ref
    from oracle import mesh_distance as omd

    lib = C.CDLL(build_ref.build(force=True))
    dp = C.POINTER(C.c_double)
    lib.s2m_tri.restype = C.c_double
    lib.s2m_tri.argtypes = [C.c_int, C.c_double, C.c_int, dp, dp, dp, dp, dp, dp, dp, dp]
    rng = np.random.default_rng(7)
    kinds = np.array([(omd.KIND_DISTANCE, 1.0), (omd.KIND_SQUARED, 1.0), (omd.KIND_GM, 0.05), (omd.KIND_GM, 0.5)])
    xabc = np.zeros((40, 4, 3))
    value, grad = np.zeros((40, len(kinds), 7)), np.zeros((40, len(kinds), 7, 4, 3))
    for t in range(40):
        a, b, c = rng.normal(0, 0.3, (3, 3))
        xabc[t] = (a + b + c) / 3 + rng.normal(0, 0.2, 3), a, b, c
        for k, (kind, sigma) in enumerate(kinds):
            for part in range(7):
                args = [np.ascontiguousarray(v) for v in xabc[t]]
                bufs = [np.zeros(3) for _ in range(4)]
                value[t, k, part] = lib.s2m_tri(int(kind), float(sigma), part, *[v.ctypes.data_as(dp) for v in args + bufs])
                grad[t, k, part] = bufs
    np.savez_compressed(os.path.join(HERE, 'ref_s2m.npz'), kinds=kinds, xabc=xabc, value=value, grad=grad)
    print('ref_s2m.npz:', value.shape, grad.shape)


if __name__ == '__main__':
    main()
    prior_and_marker_vectors()
    mesh_distance_vectors()
