"""GPU parity, EKF: predict / measurement prediction + selection / update / normalise / delete
through the C ABI vs the CPU oracle.  Tolerance: the north star's 1e-5 relative, tested at 1e-8
(gpu_util.RTOL_TEST) relative to the natural covariance scale sqrt(P_ii P_jj)."""
import numpy as np
import pytest

from gpu_util import (RTOL_TEST, assert_state_close, ctx_from_scenes, oracle_slam_from_scene, random_measurements,
                      state_err, synth)

pytestmark = pytest.mark.gpu


def test_predict_matches_oracle(oracle):
    sc = synth.make_scene("C2", n_frames=1, n_features=30)
    ctx = ctx_from_scenes([sc])
    o = oracle_slam_from_scene(oracle, sc)
    for _ in range(3):
        ctx.ekf_predict(0)
        o.predict()
        xg, Pg = ctx.get_state(0)
        xo, Po = o.get_state()
        assert_state_close(xg, Pg, xo, Po, rtol=1e-12)    # same op order; only sin/cos ulps differ
        assert np.abs(Pg - Pg.T)[13:, :].max() == 0.0      # Pxy mirrored exactly
    ctx.close()


def test_measurement_prediction_and_selection(oracle):
    for name, kw in (("C1", dict()), ("C2", dict(n_features=40, override=False))):
        sc = synth.make_scene(name, n_frames=1, **kw)
        ctx = ctx_from_scenes([sc])
        o = oracle_slam_from_scene(oracle, sc)
        ctx.ekf_predict(0)
        o.predict()
        nv = ctx.predict_measurements(0)
        assert nv == o.select()
        fg, fo = ctx.features(0), o.features()
        assert np.allclose(fg["h"], fo["h"], rtol=0, atol=1e-9)
        assert np.allclose(fg["S"], fo["S"], rtol=1e-10, atol=0)
        assert (fg["select_rank"] == fo["select_rank"]).all()
        assert (fg["select_rank"] >= 0).sum() == min(sc.n_select, nv)
        ctx.close()


@pytest.mark.parametrize("nf,K", [(20, 4), (20, 20), (50, 50), (100, 100), (37, 13), (128, 128), (128, 77),
                                  (5, 1), (9, 9)])
def test_update_with_host_rows_matches_dense_oracle(oracle, nf, K):
    """kalman.cpp:72-119 as written (dense, explicit S^-1) vs the structured CUDA update."""
    sc = synth.make_scene("C4", n_frames=1, n_features=nf)
    ctx = ctx_from_scenes([sc])
    rng = np.random.default_rng(nf * 1000 + K)
    n = sc.n
    feats, Hxv, Hy, R, nu, H, Rfull = random_measurements(rng, n, nf, K)
    ctx.ekf_update(0, feats, Hxv, Hy, R, nu)
    xg, Pg = ctx.get_state(0)
    xo, Po = oracle.kalman_update_dense(sc.x0, sc.P0, H, Rfull, nu)
    # normalise + symmetrise as GoOneStep does after the update (monoslam.cpp:137,143-150)
    J = np.eye(n)
    J[:13, :13] = oracle.dxvnorm_by_dxv(xo[:13])
    Po = J @ Po @ J.T
    Po = 0.5 * (Po + Po.T)
    ex, eP = assert_state_close(xg, Pg, xo, Po)
    assert np.abs(Pg - Pg.T).max() == 0.0
    print("update nf=%d K=%d: state err %.2e cov err %.2e" % (nf, K, ex, eP))
    ctx.close()


def test_staged_pipeline_matches_oracle(oracle):
    sc = synth.make_scene("C2", n_frames=3, n_features=32, override=False)
    ctx = ctx_from_scenes([sc])
    o = oracle_slam_from_scene(oracle, sc)
    for t in range(3):
        ctx.set_frame(0, 0, sc.frames[t])
        ctx.ekf_predict(0)
        ctx.predict_measurements(0)
        cnt = ctx.make_measurements(0, 0)
        ctx.ekf_update_measured(0)
        o.predict()
        o.select()
        assert cnt == o.measure(sc.frames[t])
        o.update()
        o.normalise()
        o.finish()
        fg, fo = ctx.features(0), o.features()
        assert (fg["z"] == fo["z"]).all() and (fg["flags"] == fo["flags"]).all()
        assert (fg["attempted"] == fo["attempted"]).all() and (fg["successful"] == fo["successful"]).all()
        assert_state_close(*ctx.get_state(0), *o.get_state())
    ctx.close()


def test_normalise_only(oracle):
    sc = synth.make_scene("C2", n_frames=1, n_features=10)
    sc.x0[3:7] = [0.9, 0.1, -0.2, 0.15]
    ctx = ctx_from_scenes([sc])
    o = oracle_slam_from_scene(oracle, sc)
    ctx.normalise_state(0)
    o.normalise()
    o.finish()
    assert_state_close(*ctx.get_state(0), *o.get_state(), rtol=1e-13)
    ctx.close()


def test_delete_feature(oracle):
    sc = synth.make_scene("C2", n_frames=1, n_features=9)
    ctx = ctx_from_scenes([sc])
    ctx.delete_feature(0, 3)
    ctx.delete_feature(0, 7)           # last one after the shift
    keep = np.r_[0:13, [13 + 3 * f + c for f in (0, 1, 2, 4, 5, 6, 7) for c in range(3)]]
    x, P = ctx.get_state(0)
    assert ctx.num_features(0) == 7
    assert (x == sc.x0[keep]).all() and (P == sc.P0[np.ix_(keep, keep)]).all()
    # the templates moved with their features: search still finds feature 4 (now index 3)
    ctx.set_frame(0, 0, sc.frames[0])
    u, v, f, _ = ctx.patch_search(0, 0, np.array([3], np.int32), sc.pix[4:5].astype(float),
                                  np.array([[0.0225, 0, 0.0225]]))
    assert f[0] == 1 and (u[0], v[0]) == tuple(sc.pix[4])
    ctx.close()


def test_update_honours_full_2x2_R_and_rejects_asymmetric(oracle):
    """kalman.cpp:101 adds the whole block-diagonal R; the ABI takes R as K x (2x2 column-major)."""
    nf, K = 24, 10
    sc = synth.make_scene("C4", n_frames=1, n_features=nf)
    ctx = ctx_from_scenes([sc])
    rng = np.random.default_rng(77)
    n = sc.n
    feats, Hxv, Hy, R, nu, H, _ = random_measurements(rng, n, nf, K)
    Hxv[:, 7:] = rng.standard_normal((2 * K, 6)) * 20      # all 13 dh/dxv columns, not only [dh/dxp | 0]
    H[:, :13] = Hxv
    for k in range(K):                                     # anisotropic, correlated measurement noise
        a = rng.standard_normal((2, 2))
        R[k] = a @ a.T + 0.5 * np.eye(2)
    Rfull = np.zeros((2 * K, 2 * K))
    for k in range(K):
        Rfull[2 * k:2 * k + 2, 2 * k:2 * k + 2] = R[k]
    ctx.ekf_update(0, feats, Hxv, Hy, R, nu)
    xg, Pg = ctx.get_state(0)
    xo, Po = oracle.kalman_update_dense(sc.x0, sc.P0, H, Rfull, nu)
    J = np.eye(n)
    J[:13, :13] = oracle.dxvnorm_by_dxv(xo[:13])
    Po = J @ Po @ J.T
    Po = 0.5 * (Po + Po.T)
    assert_state_close(xg, Pg, xo, Po)
    bad = R.copy()
    bad[3, 0, 1] += 1e-3                                   # R01 != R10: not a covariance block
    with pytest.raises(Exception) as e:
        ctx.ekf_update(0, feats, Hxv, Hy, bad, nu)
    assert "symmetric" in str(e.value)
    ctx.close()


def test_make_measurements_counts_only_this_frames_selection(oracle):
    """ADVICE r1: found[] keeps the flag of features that are not selected this frame (like
    Feature::successful_measurement_flag_); the returned count must cover the selected ones only
    (monoslam.cpp:336-359).  n_select = 4 of 20 and a camera that turns: the selection changes."""
    sc = synth.make_scene("C2", n_frames=6, n_features=20, override=False)
    sc.n_select = 4
    ctx = ctx_from_scenes([sc])
    o = oracle_slam_from_scene(oracle, sc)
    sels = []
    for t in range(6):
        ctx.set_frame(0, 0, sc.frames[t])
        ctx.ekf_predict(0)
        ctx.predict_measurements(0)
        cnt = ctx.make_measurements(0, 0)
        ctx.ekf_update_measured(0)
        o.predict()
        o.select()
        assert cnt == o.measure(sc.frames[t]), t
        o.update()
        o.normalise()
        o.finish()
        fg = ctx.features(0)
        sel = fg["select_rank"] >= 0
        assert cnt == int(((fg["flags"] & 2) > 0)[sel].sum()) and cnt <= 4
        sels.append(tuple(np.nonzero(sel)[0]))
    assert len(set(sels)) > 1, "the scenario must change the selection between frames"
    ctx.close()


def test_delete_feature_moves_jacobians_with_the_feature(oracle):
    """ADVICE r1: Feature::dh_by_dxv_ / dh_by_dy_ / R_ belong to the Feature object (feature.h:104-112);
    after a deletion the records of the later features must move down with them."""
    sc = synth.make_scene("C2", n_frames=1, n_features=12, override=False)
    ctx = ctx_from_scenes([sc])
    ctx.ekf_predict(0)
    ctx.predict_measurements(0)
    J0, Jy0, R0, _ = ctx.feature_jacobians(0)
    ctx.delete_feature(0, 4)
    J1, Jy1, R1, _ = ctx.feature_jacobians(0)
    keep = [i for i in range(12) if i != 4]
    assert J1.shape[0] == 11
    assert (J1 == J0[keep]).all() and (Jy1 == Jy0[keep]).all() and (R1 == R0[keep]).all()
    ctx.close()


def test_append_feature_grows_the_map_in_place(oracle):
    """MonoSLAM::AddNewKnownFeature on the device (monoslam.cpp:1278-1289, feature.cpp:108-149): x and P grow by the
    new feature (zero covariance blocks for a known feature, or the caller's column block), nothing else moves, and a
    fused step on the grown map equals a step on a map that was uploaded whole."""
    import scenelib2_b200 as sl2
    full = synth.make_scene("C2", n_frames=2, n_features=12, override=False)
    n10 = 13 + 3 * 10
    # context A: 10 features uploaded, 2 appended; context B: the 12-feature map uploaded whole
    cfg = sl2.config_for_scene(full, num_streams=1, frame_slots=1, max_features=12)
    a, b = sl2.Context(cfg), sl2.Context(cfg)
    a.set_features(0, full.x0[13:n10].reshape(10, 3), full.xp_org[:10], full.patches[:10])
    a.set_state(0, full.x0[:n10], full.P0[:n10, :n10])
    Pcol10 = np.asfortranarray(full.P0[:n10 + 3, n10:n10 + 3])
    assert a.append_feature(0, full.x0[n10:n10 + 3], full.xp_org[10], full.patches[10], Pcol10) == 10
    n11 = n10 + 3
    assert a.append_feature(0, full.x0[n11:n11 + 3], full.xp_org[11], full.patches[11],
                            full.P0[:n11 + 3, n11:n11 + 3]) == 11
    with pytest.raises(Exception):                       # the map is full
        a.append_feature(0, full.x0[n11:n11 + 3], full.xp_org[11], full.patches[11])
    sl2.load_scene(b, 0, full)
    xa, Pa = a.get_state(0)
    xb, Pb = b.get_state(0)
    assert a.num_features(0) == 12 and (xa == xb).all() and (Pa == Pb).all()
    for t in range(2):
        for c in (a, b):
            c.set_frames(0, full.frames[t][None])
            c.step(0)
        (xa, Pa), (xb, Pb) = a.get_state(0), b.get_state(0)
        assert (xa == xb).all() and (Pa == Pb).all()
        fa, fb = a.features(0), b.features(0)
        assert all((fa[k] == fb[k]).all() for k in ("z", "flags", "attempted", "successful", "select_rank"))
    # a known feature (Pcol = NULL): zero blocks like Feature::Pxy_ / Pyy_ / matrix_block_list_ of the reference
    c = sl2.Context(cfg)
    c.set_features(0, full.x0[13:n10].reshape(10, 3), full.xp_org[:10], full.patches[:10])
    c.set_state(0, full.x0[:n10], full.P0[:n10, :n10])
    c.append_feature(0, full.x0[n10:n10 + 3], full.xp_org[10], full.patches[10])
    xc, Pc = c.get_state(0)
    assert Pc.shape == (n10 + 3, n10 + 3) and (Pc[:n10, :n10] == full.P0[:n10, :n10]).all()
    assert (Pc[n10:, :] == 0).all() and (Pc[:, n10:] == 0).all() and (xc[n10:] == full.x0[n10:n10 + 3]).all()
    for ctx in (a, b, c):
        ctx.close()
