"""Pins the oracle's patch-correlation restatement (A1, A11, and through A11 the A2 loop), its models and its
whole tracking step to the REFERENCE's own source: SceneLib2's improc/{improc,search_multiple_overlapping_ellipses}.cpp
compiled unmodified (oracle/_ref/libsl2ref.so, golden vectors of tests/golden/make_golden.py; bit-exact) and its
tracking core compiled against oracle/stubs_arith (oracle/_ref/libsl2refmodels.so).  The outputs of that code for
the inputs below are stored under tests/golden/ref_*.npz (the `ref` fixture, tests/refgolden.py)."""
import os

import numpy as np
import pytest

from refgolden import assert_cov_close, cov_sample, digest, pick

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_a1_matches_reference_golden(oracle):
    k = np.load(os.path.join(G, "a1_ref_kat.npz"))
    assert len(k["B"]) == 48
    for B, patch, image, xy, out in zip(k["B"], k["patch"], k["image"], k["xy"], k["out"]):
        c, s0, s1 = oracle.correlate2_warning(patch[:B, :B], image, xy[0], xy[1])
        # bit-exact, NaN-safe
        assert np.array([c, s0, s1]).tobytes() == out.tobytes()
    # the degenerate branches (improc.cpp:117-125) are present in the vectors
    assert (k["out"][:, 1] == 0).any() and (k["out"][:, 2] == 0).any()
    assert ((k["out"][:, 1] == 0) & (k["out"][:, 2] == 0) & (k["out"][:, 0] == 0)).any()


def test_a11_matches_reference_golden(oracle):
    k = np.load(os.path.join(G, "a11_ref_kat.npz"))
    ru, rv, rf, _ = oracle.smoe_search(k["image"], k["patch"], k["puinv3"], k["centres"])
    assert (ru == k["res_u"]).all() and (rv == k["res_v"]).all() and (rf == k["res_flag"]).all()
    assert rf.any() and not rf.all()


def test_a1_live_reference_random(oracle, ref):
    rng = np.random.default_rng(7)
    for B in (11, 15, 9):
        img = rng.integers(0, 256, (40, 50), dtype=np.uint8)
        for _ in range(200):
            patch = rng.integers(0, 256, (B, B), dtype=np.uint8)
            x1, y1 = int(rng.integers(0, 50 - B)), int(rng.integers(0, 40 - B))
            a = oracle.correlate2_warning(patch, img, x1, y1)
            b = ref.take("a1", lambda: oracle.correlate2_warning(patch, img, x1, y1, use_ref=True))
            assert np.array(a).tobytes() == np.array(b).tobytes()


def test_a11_live_reference_random(oracle, ref):
    from scenelib2_b200 import synth
    rng = np.random.default_rng(11)
    img = synth.make_texture(rng, 96, 128)
    img[20:50, 30:70] = 90
    for B in (11, 15):
        patch = img[60:60 + B, 80:80 + B].copy()
        K = 20
        centres = np.column_stack([rng.uniform(0, 128, K), rng.uniform(0, 96, K)])
        centres[:4] = [[80 + B // 2 + 0.4, 60 + B // 2 + 0.6]] * 4
        sx, sy = rng.uniform(1.5, 6, K), rng.uniform(1.5, 6, K)
        rho = rng.uniform(-0.8, 0.8, K)
        pu = []
        for a, b, r in zip(sx, sy, rho):
            Si = np.linalg.inv(np.array([[a * a, r * a * b], [r * a * b, b * b]]))
            pu.append([Si[0, 0], Si[0, 1], Si[1, 1]])
        pu = np.array(pu)
        a = oracle.smoe_search(img, patch, pu, centres)
        b = ref.take("a11", lambda: oracle.smoe_search(img, patch, pu, centres, use_ref=True))
        for x, y in zip(a[:3], b[:3]):
            assert (x == y).all()


def test_a2_equals_a11_where_they_coincide(oracle):
    """A2 (monoslam.cpp:401-477) and A11 share the scan; with integer+0.0 centres (rounding ==
    truncation), image sigma >= 10 everywhere and one ellipse they must agree exactly."""
    from scenelib2_b200 import synth
    rng = np.random.default_rng(5)
    img = synth.make_texture(rng, 100, 140)
    B = 11
    for _ in range(10):
        cx, cy = int(rng.integers(10, 130)), int(rng.integers(10, 90))
        patch = img[cy - 5:cy + 6, cx - 5:cx + 6].copy()
        c = np.array([[cx + int(rng.integers(-4, 5)), cy + int(rng.integers(-4, 5))]], float)
        a, b, r = rng.uniform(2, 7), rng.uniform(2, 7), rng.uniform(-0.7, 0.7)
        Si = np.linalg.inv(np.array([[a * a, r * a * b], [r * a * b, b * b]]))
        pu = np.array([[Si[0, 0], Si[0, 1], Si[1, 1]]])
        u, v, f, best = oracle.elliptical_search(img, patch[None], c, pu)
        ru, rv, rf, rbest = oracle.smoe_search(img, patch, pu, c)
        assert (u[0], v[0], f[0]) == (ru[0], rv[0], rf[0])
        assert best[0] == rbest[0]


# ---- closed-form models: the reference's OWN motion_model.cpp / camera.cpp / feature_model.cpp /
# full_feature_model.cpp / support/math_util.cpp, compiled unmodified against oracle/stubs_arith (a minimal
# matrix class with plain-loop arithmetic, NOT Eigen), vs the oracle's restatement.  Pins every formula
# (Jacobians, Q, projection + distortion, R_i, S_i, visibility); Eigen's summation order stays unpinned.

def _random_xv(rng, normalise=True):
    xv = np.zeros(13)
    xv[:3] = rng.normal(0, 0.3, 3)
    q = rng.normal(0, 1, 4)
    if normalise:
        q /= np.linalg.norm(q)
    xv[3:7] = q
    xv[7:10] = rng.normal(0, 0.2, 3)
    xv[10:13] = rng.normal(0, 0.3, 3)
    return xv


def test_motion_model_matches_reference_source(oracle, ref):
    rng = np.random.default_rng(31)
    worst = 0.0
    for k in range(200):
        xv = _random_xv(rng, normalise=(k % 3 != 0))        # the reference never renormalises q (Q1)
        if k % 10 == 0:
            xv[10:13] = [0.0, 0.0, 0.01]                    # the cfg's starting omega (data/SceneLib2.cfg:81-83)
        dt = [1 / 30.0, 0.05, 0.01][k % 3]
        u = rng.normal(0, 1, 3) if k % 4 == 0 else np.zeros(3)
        a = oracle.motion(xv, dt, u)
        b = ref.take("motion", lambda: [pick(v, k, 16) for v in oracle.motion(xv, dt, u, use_ref=True)])
        for x, y in zip(a, b):
            x = pick(x, k, 16)
            assert np.isfinite(y).all()
            worst = max(worst, np.abs(x - y).max() / max(1.0, np.abs(y).max()))
        J = oracle.dxvnorm_by_dxv(xv)
        Jr, xn = ref.take("dxvnorm", lambda: [digest(v) for v in oracle.dxvnorm_by_dxv(xv, use_ref=True)])
        assert (digest(J) == Jr).all()                       # scalar formulas only: bit-exact
        assert (digest(xv) == xn).all()                      # quirk Q1: xv comes back un-normalised
    assert worst < 1e-15, worst


def test_measurement_model_matches_reference_source(oracle, ref):
    rng = np.random.default_rng(32)
    cams = [np.array([320, 240, 195.0, 195.0, 162.0, 125.0, 9e-6, 1.0]),
            np.array([640, 480, 390.0, 392.0, 322.0, 247.0, 2e-6, 2.0])]
    worst = 0.0
    flags_seen = set()
    for k in range(300):
        cam8 = cams[k % 2]
        xv = _random_xv(rng)
        xv[:3] *= 0.2
        xv[3:7] = [1, 0, 0, 0] + rng.normal(0, 0.15 if k % 5 else 1.0, 4)
        y = np.array([rng.uniform(-0.6, 0.6), rng.uniform(-0.4, 0.4), rng.uniform(0.3, 3.0)])
        if k % 17 == 0:
            y[2] = -abs(y[2])                                # behind the camera
        A = rng.normal(0, 1, (16, 16))
        P = A @ A.T * 1e-4 + 1e-6 * np.eye(16)
        Pxx, Pxy, Pyy = P[:13, :13], P[:13, 13:], P[13:, 13:]
        a = oracle.predict_feature(cam8, xv, y, Pxx, Pxy, Pyy)
        b = ref.take("predict", lambda: [pick(v, k, 4) for v in
                                         oracle.predict_feature(cam8, xv, y, Pxx, Pxy, Pyy, use_ref=True)])
        for x, r in zip(a, b):
            x = pick(x, k, 4)
            if np.isfinite(r).all():
                worst = max(worst, np.abs(x - r).max() / max(1.0, np.abs(r).max()))
            else:
                assert not np.isfinite(x).all()
        xp_org = _random_xv(rng)[:7]
        xp_org[:3] *= 0.2
        xp_org[3:7] = [1, 0, 0, 0] + rng.normal(0, 0.3, 4)
        h = a[0] if np.isfinite(a[0]).all() else np.array([100.0, 100.0])
        va = oracle.visibility_test(cam8, xv[:7], y, xp_org, h)
        vb = ref.take("visibility", lambda: oracle.visibility_test(cam8, xv[:7], y, xp_org, h, use_ref=True))
        assert va == vb, (k, va, vb)
        flags_seen.add(vb)
    assert worst < 1e-13, worst
    assert 0 in flags_seen and len(flags_seen) >= 5          # visible and several distinct failure codes


def test_particle_prediction_matches_reference_source(oracle, ref):
    """N2 prediction (monoslam.cpp:1347-1400): the oracle's PartFeatureModel::predict_particle against the
    reference's own part_feature_model.cpp / feature_model.cpp / feature_init_info.cpp (compiled unmodified
    against oracle/stubs_arith): h, S, S^-1, det S per depth particle."""
    rng = np.random.default_rng(57)
    cams = [np.array([320, 240, 195.0, 195.0, 162.0, 125.0, 9e-6, 1.0]),
            np.array([640, 480, 390.0, 392.0, 322.0, 247.0, 2e-6, 2.0])]
    worst = 0.0
    for k in range(120):
        cam8 = cams[k % 2]
        xv = _random_xv(rng)
        xv[:3] *= 0.2
        xv[3:7] = [1, 0, 0, 0] + rng.normal(0, 0.15, 4)
        hh = np.array([rng.uniform(-0.5, 0.5), rng.uniform(-0.4, 0.4), 1.0])
        ypi = np.concatenate([xv[:3] + rng.normal(0, 0.05, 3), hh / np.linalg.norm(hh)])
        A = rng.normal(0, 1, (19, 19))
        P = A @ A.T * 1e-4 + 1e-6 * np.eye(19)
        lam = np.sort(rng.uniform(0.3, 6.0, 9))
        a = oracle.predict_particles(cam8, xv, ypi, lam, P[:13, :13], P[:13, 13:], P[13:, 13:])
        b = ref.take("particles", lambda: [pick(v, k, 4) for v in oracle.predict_particles(
            cam8, xv, ypi, lam, P[:13, :13], P[:13, 13:], P[13:, 13:], use_ref=True)])
        for x, r in zip(a, b):
            x = pick(x, k, 4)
            assert np.isfinite(r).all()
            worst = max(worst, np.abs(x - r).max() / max(1.0, np.abs(r).max()))
    assert worst < 1e-13, worst


def test_sinv_matches_reference_source(oracle, ref):
    """Particle::set_S (the reference's own feature_init_info.cpp:55-63, compiled against oracle/stubs_arith)
    runs the same LLT -> matrixL -> inverse -> L^-T L^-1 sequence as MonoSLAM::measure_feature
    (monoslam.cpp:371-374), i.e. the oracle's S -> PuInv (A3).  (The particle bookkeeping of that file is
    checked bit-exactly in test_particle_cycle_matches_reference_source.)"""
    rng = np.random.default_rng(33)
    for _ in range(300):
        a, b = rng.uniform(1, 400, 2)
        r = rng.uniform(-0.95, 0.95)
        S = np.array([[a, r * np.sqrt(a * b)], [r * np.sqrt(a * b), b]])
        Sinv_ref, det_ref = ref.take("set_S", lambda: oracle.particle_set_S_ref(S))
        pu = oracle.puinv_from_S(S)
        ref3 = np.array([Sinv_ref[0, 0], Sinv_ref[0, 1], Sinv_ref[1, 1]])
        np.testing.assert_allclose(pu, ref3, rtol=4e-15, atol=0)
        assert Sinv_ref[0, 1] == Sinv_ref[1, 0]
        np.testing.assert_allclose(det_ref, a * b * (1 - r * r), rtol=1e-12)


# ---- the whole tracking step: the reference's OWN monoslam.cpp / kalman.cpp / feature.cpp (+ models, improc)
# compiled unmodified against oracle/stubs_arith and driven through MonoSLAM::Init / AddNewKnownFeature /
# fill_* / GoOneStep (oracle/ref_slam_shim.cpp), vs the oracle.  Integer results must be identical; state and
# covariance agree up to summation order (the stand-in matrix class is not Eigen).

def ref_state(r):
    """What the comparisons use of the reference's state: x, and a cov_sample of P (keys P_*)."""
    x, P = r.get_state()
    return dict(x=x, num_features=r.num_features, n=r.n, **{"P_" + k: v for k, v in cov_sample(P).items()})


def ref_step(ref, key, r, frame):
    """One GoOneStep of the reference slam `r` (recording only) -> its features and ref_state."""
    def run():
        r.step(frame)
        return dict(r.features(), **ref_state(r))
    return ref.take(key, run)


def ref_cov(fr):
    return {k[2:]: v for k, v in fr.items() if k.startswith("P_")}


def _compare_step(fr, o, t, tol):
    fo = o.features()
    assert fr["num_features"] == o.num_features and fr["n"] == o.n
    assert (fr["label"] == fo["label"]).all()
    assert (fr["select_rank"] == fo["select_rank"]).all(), t
    assert ((fr["flags"] & 1) == (fo["flags"] & 1)).all(), t
    seen = fo["attempted"] > 0      # the reference leaves the success flag uninitialised until first measured
    assert ((fr["flags"] & 2)[seen] == (fo["flags"] & 2)[seen]).all(), t
    ok = (fo["flags"] & 2) > 0
    assert (fr["z"][ok] == fo["z"][ok]).all(), t                       # bit-exact match positions
    assert (fr["attempted"] == fo["attempted"]).all() and (fr["successful"] == fo["successful"]).all()
    sel = fo["select_rank"] >= 0
    np.testing.assert_allclose(fr["h"][sel], fo["h"][sel], rtol=tol, atol=tol)
    np.testing.assert_allclose(fr["S"][sel], fo["S"][sel], rtol=tol, atol=tol)
    xo, Po = o.get_state()
    d = np.sqrt(np.abs(np.diag(Po))) + 1e-300
    assert np.abs(fr["x"] - xo).max() <= tol * max(1.0, np.abs(xo).max())
    assert_cov_close(Po, ref_cov(fr), tol, d)
    assert fr["P_asym"] == 0.0


def test_whole_step_matches_reference_source(oracle, ref, tmp_path):
    from scenelib2_b200 import synth
    from test_oracle_slam import make_oracle_slam
    kp = np.load(os.path.join(G, "known_patches.npy"))
    # C1: 20 features, 10 selected per frame by trace(S), ellipses from the EKF's own S_i
    sc = synth.make_scene("C1", n_frames=12, known_patches=kp)
    r = oracle.RefSlam(sc, str(tmp_path / "c1")) if ref.recording else None
    o = make_oracle_slam(oracle, sc)
    fr = ref.take("c1_init", lambda: ref_state(r))
    xo, Po = o.get_state()
    assert (fr["x"] == xo).all()                          # Init + AddNewKnownFeature + fill_* round trip
    assert_cov_close(Po, ref_cov(fr), 0.0, np.ones(len(xo)))
    for t in range(12):
        fr = ref_step(ref, "c1", r, sc.frames[t])
        o.step(sc.frames[t])
        _compare_step(fr, o, t, 1e-12)
    # C2-like without the benchmark's ellipse override: every feature selected (m = 2N), bigger update
    sc = synth.make_scene("C2", n_frames=4, n_features=24, override=False)
    r = oracle.RefSlam(sc, str(tmp_path / "c2")) if ref.recording else None
    o = make_oracle_slam(oracle, sc)
    for t in range(4):
        fr = ref_step(ref, "c2", r, sc.frames[t])
        o.step(sc.frames[t])
        _compare_step(fr, o, t, 1e-11)
    assert (o.features()["select_rank"] >= 0).sum() == 24


def test_bad_feature_deletion_matches_reference_source(oracle, ref, tmp_path):
    """delete_bad_features / delete_feature (monoslam.cpp:644-703, 770-812): a template that never matches is
    culled after 10 attempts; the compaction of state, covariance blocks and lists is the reference's own."""
    from scenelib2_b200 import synth
    from test_oracle_slam import make_oracle_slam
    sc = synth.make_scene("C2", n_frames=2, n_features=12, override=False)
    bad = sc.patches.copy()
    bad[3] = np.random.default_rng(0).integers(0, 256, bad[3].shape, dtype=np.uint8)
    sc.patches = bad
    r = oracle.RefSlam(sc, str(tmp_path)) if ref.recording else None
    o = make_oracle_slam(oracle, sc)
    n0 = o.n
    for t in range(12):
        fr = ref_step(ref, "step", r, sc.frames[t % 2])
        o.step(sc.frames[t % 2])
        _compare_step(fr, o, t, 1e-11)
    assert fr["num_features"] == 11 and fr["n"] == n0 - 3


def test_c1_trajectory_1000_steps_reproduced_by_reference_source(oracle, refmodels, tmp_path):
    """tests/golden/c1_trajectory_1000.npz is an output of the reference's own code (make_c1_trajectory.py);
    re-running it live must reproduce the fixture: identical hash of the selection ranks / flags / match
    positions of all 1 000 steps (10 000 measurements), identical counters, camera state within 1e-11.
    (The oracle and the CUDA path are tested against the same fixture.)"""
    import hashlib
    import sys
    from scenelib2_b200 import synth
    sys.path.insert(0, G)
    import make_c1_trajectory as gen
    k = np.load(os.path.join(G, "c1_trajectory_1000.npz"))
    kp = np.load(os.path.join(G, "known_patches.npy"))
    sc = synth.make_scene("C1", n_frames=gen.RING, known_patches=kp)
    r = oracle.RefSlam(sc, str(tmp_path))
    hz = hashlib.sha256()
    for t in range(gen.STEPS):
        r.step(sc.frames[gen.frame_index(t)])
        f = r.features()
        hz.update(np.ascontiguousarray(f["select_rank"], np.int32).tobytes())
        hz.update(np.ascontiguousarray(f["flags"], np.uint8).tobytes())
        hz.update(np.ascontiguousarray(f["z"][(f["flags"] & 2) > 0], np.float64).tobytes())
        if (t + 1) % gen.EVERY == 0:
            x, P = r.get_state()
            i = (t + 1) // gen.EVERY - 1
            np.testing.assert_allclose(x[:13], k["xv"][i], rtol=1e-11, atol=1e-12)
            np.testing.assert_allclose(np.diag(P)[:13], k["Pxx_diag"][i], rtol=1e-10)
    f = r.features()
    assert (np.frombuffer(hz.digest(), np.uint8) == k["integer_hash"]).all()
    assert (f["attempted"] == k["attempted"]).all() and (f["successful"] == k["successful"]).all()


def test_elliptical_search_and_detector_match_reference_source(oracle, ref):
    """A2 / A3 / N3 one by one against the reference's own monoslam.cpp: MonoSLAM::elliptical_search (rotated and
    border-clamped ellipses, plateaus, 11x11 and 15x15), measure_feature (S -> PuInv -> search) and
    find_best_patch_inside_region (positions and FP64 eigenvalue bits)."""
    from scenelib2_b200 import synth
    rng = np.random.default_rng(41)
    img = synth.make_texture(rng, 120, 160)
    img[30:60, 40:90] = 128                                   # plateau: low sigma, ties
    n_found = 0
    for B in (11, 15):
        h = (B - 1) // 2
        for k in range(120):
            cu, cv = int(rng.integers(h, 160 - h)), int(rng.integers(h, 120 - h))
            patch = img[cv - h:cv + h + 1, cu - h:cu + h + 1].copy()
            if k % 4 == 0:
                patch = rng.integers(0, 256, (B, B), dtype=np.uint8)      # no good match anywhere
            a, b = rng.uniform(2, 14, 2)
            th = rng.uniform(0, np.pi)
            R = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
            Si = np.linalg.inv(R @ np.diag([a * a / 9, b * b / 9]) @ R.T)
            pu = np.array([Si[0, 0], Si[0, 1], Si[1, 1]])
            centre = np.array([cu + rng.uniform(-4, 4), cv + rng.uniform(-4, 4)])
            if k % 7 == 0:
                centre = np.array([rng.choice([1.5, 158.2]), rng.choice([2.4, 117.9])])   # clamped at a corner
            ok, ru, rv = ref.take("search", lambda: oracle.elliptical_search_ref(img, patch, centre, pu))
            ou, ov, of, _ = oracle.elliptical_search(img, patch[None], centre[None], pu[None])
            assert bool(of[0]) == bool(ok), (B, k)
            if ok:
                assert (ou[0], ov[0]) == (ru, rv), (B, k)
                n_found += 1
    assert n_found > 60
    for k in range(100):                                       # A3: S -> PuInv -> search, 11x11
        cu, cv = int(rng.integers(10, 150)), int(rng.integers(10, 110))
        patch = img[cv - 5:cv + 6, cu - 5:cu + 6].copy()
        a, b = rng.uniform(4, 60, 2)
        r = rng.uniform(-0.8, 0.8)
        S = np.array([[a, r * np.sqrt(a * b)], [r * np.sqrt(a * b), b]])
        hh = np.array([cu + rng.uniform(-3, 3), cv + rng.uniform(-3, 3)])
        ok, z = ref.take("measure", lambda: oracle.measure_feature_ref(img, patch, hh, S))
        pu = oracle.puinv_from_S(S)
        ou, ov, of, _ = oracle.elliptical_search(img, patch[None], hh[None], pu[None])
        assert bool(of[0]) == bool(ok), k
        if ok:
            assert (z == [ou[0], ov[0]]).all(), k
    regions = np.array([[40, 30, 120, 90], [-5, -7, 60, 40], [100, 70, 400, 300], [0, 0, 160, 120],
                        [50, 50, 50, 80], [3, 3, 40, 30], [90, 20, 91, 21], [10, 10, 30, 25]], np.int32)
    for B in (11, 15):
        for reg in regions:
            a = oracle.find_best_patch(img, B, reg, ubest=-7, vbest=-9)
            b = ref.take("best_patch", lambda: oracle.find_best_patch(img, B, reg, ubest=-7, vbest=-9, use_ref=True))
            assert a[:2] == b[:2] and np.float64(a[2]).tobytes() == np.float64(b[2]).tobytes(), (B, reg)


def test_particle_cycle_matches_reference_source(oracle, ref, tmp_path):
    """N2 end to end on the reference's own code: InitialiseFeature creates a partially-initialised feature with
    100 depth particles; after the camera has moved, predict_partially_initialised_feature_measurements
    (part_feature_model.cpp), measure_feature_with_multiple_priors (SMOE) and
    update_partially_initialised_feature_probabilities run as in MatchPartiallyInitialisedFeatures
    (monoslam.cpp:1299-1340).  Fed with the same particle inputs, the oracle's SMOE search and particle update
    give identical matches, survivors, probabilities (bit-exact), mean and variance."""
    from scenelib2_b200 import synth
    kp = np.load(os.path.join(G, "known_patches.npy"))
    sc = synth.make_scene("C1", n_frames=6, known_patches=kp)
    cycles = 0
    for (u, v, dx) in ((150, 110, (0.03, -0.01, 0.0)), (90, 70, (-0.02, 0.02, 0.01)), (200, 150, (0.0, 0.04, 0.0))):
        r = oracle.RefSlam(sc, str(tmp_path / ("p%d_%d" % (u, v)))) if ref.recording else None

        def init():
            r.init_partial_feature(sc.frames[0], u, v)
            return r.num_features, r.n
        nf, n = ref.take("init", init)
        assert nf == sc.n_features + 1 and n == 13 + 3 * sc.n_features + 6
        # no match attempt right after initialisation
        assert ref.take("cycle", lambda: r.particle_cycle(sc.frames[0])) is None
        patch = sc.frames[0][v - 5:v + 6, u - 5:u + 6]
        for t in (1, 2, 3):
            def cycle():
                x, P = r.get_state()
                x[:3] += dx                                    # the camera moves: the depth line spreads out
                r.set_state(x, P)
                return r.particle_cycle(sc.frames[t])
            c = ref.take("cycle", cycle)
            if c is None:
                break
            ou, ov, of, _ = oracle.smoe_search(sc.frames[t], patch, c["sinv3"], c["h"])
            assert (of == c["found"]).all()
            assert (ou[of > 0] == c["z"][of > 0, 0]).all() and (ov[of > 0] == c["z"][of > 0, 1]).all()
            o = oracle.particle_update(c["h"], c["sinv3"], c["detS"], c["lam"], c["z"], c["found"], 0.05,
                                       c["prob_before"])
            assert o[0] == c["K_after"] and (o[2] == c["keep"]).all()
            kk = c["keep"] > 0
            assert o[1][kk].tobytes() == c["prob_after"][kk].tobytes()
            assert o[3][kk].tobytes() == c["cum"][kk].tobytes()
            assert o[4].tobytes() == c["mean_var"].tobytes()
            cycles += 1
            if c["K_after"] == 0:
                break
    assert cycles >= 4


def test_c4_size_step_matches_reference_source(oracle, ref, tmp_path):
    """Full-size update (n = 313, all 100 features measured, m = 200; ellipses from the EKF's own S_i since the
    reference has no fixed-ellipse switch): Kalman::KalmanFilterUpdate as written (kalman.cpp:72-119) with its
    gather / scatter, on the reference's own code vs the oracle."""
    from scenelib2_b200 import synth
    from test_oracle_slam import make_oracle_slam
    sc = synth.make_scene("C4", n_frames=3, override=False)
    r = oracle.RefSlam(sc, str(tmp_path)) if ref.recording else None
    o = make_oracle_slam(oracle, sc)
    for t in range(3):
        fr = ref_step(ref, "step", r, sc.frames[t])
        o.step(sc.frames[t])
        _compare_step(fr, o, t, 1e-11)
    f = o.features()
    assert ((f["flags"] & 2) > 0).sum() == 100 and o.n == 313
