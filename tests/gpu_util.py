"""Helpers shared by the GPU parity tests (CUDA path through the C ABI vs the CPU oracle)."""
import numpy as np

import scenelib2_b200 as sl2
from scenelib2_b200 import synth

# north star: "FP state/covariance within 1e-5 relative".  The tests hold the CUDA path to a
# much tighter bound (different summation order only) so that real bugs cannot hide.
RTOL_NORTH_STAR = 1e-5
RTOL_TEST = 1e-8


def oracle_slam_from_scene(oracle, sc):
    cfg = oracle.make_config(width=sc.width, height=sc.height, fku=sc.cam8[2], fkv=sc.cam8[3],
                             u0=sc.cam8[4], v0=sc.cam8[5], kd1=sc.cam8[6], sd=sc.cam8[7],
                             delta_t=sc.delta_t, n_select=sc.n_select, boxsize=sc.boxsize,
                             search_override=sc.search_override)
    s = oracle.Slam(cfg)
    for i in range(sc.n_features):
        s.add_feature(sc.x0[13 + 3 * i:16 + 3 * i], sc.xp_org[i], sc.patches[i])
    s.set_state(sc.x0, sc.P0)
    return s


def ctx_from_scenes(scenes, frame_slots=1, **kw):
    cfg = sl2.config_for_scene(scenes[0], num_streams=len(scenes), frame_slots=frame_slots, **kw)
    ctx = sl2.Context(cfg)
    for s, sc in enumerate(scenes):
        sl2.load_scene(ctx, s, sc)
    return ctx


def ctx_for_image(image, patches, radius=20, boxsize=None):
    """Context with one stream whose frame is `image` and whose templates are `patches`."""
    patches = np.ascontiguousarray(patches, np.uint8)
    n, B = patches.shape[0], patches.shape[1]
    cfg = sl2.default_config()
    cfg.width, cfg.height = image.shape[1], image.shape[0]
    cfg.boxsize = B
    cfg.max_features = max(n, 1)
    cfg.search_tile_radius = radius
    ctx = sl2.Context(cfg)
    ctx.set_features(0, np.zeros((n, 3)), np.tile([0, 0, 0, 1, 0, 0, 0.0], (n, 1)), patches)
    ctx.set_frame(0, 0, image)
    return ctx


def state_err(xg, Pg, xo, Po):
    """Largest error relative to the natural scale sqrt(P_ii P_jj) (covariance) / sigma_i (state)."""
    d = np.sqrt(np.abs(np.diag(Po))) + 1e-300
    eP = np.abs(Pg - Po) / (d[:, None] * d[None, :])
    ex = np.abs(xg - xo) / np.maximum(np.abs(xo), d)
    return float(ex.max()), float(eP.max())


def assert_state_close(xg, Pg, xo, Po, rtol=RTOL_TEST):
    ex, eP = state_err(xg, Pg, xo, Po)
    assert ex <= rtol, "state error %.3e" % ex
    assert eP <= rtol, "covariance error %.3e" % eP
    return ex, eP


def random_measurements(rng, n, nf, K):
    """K distinct measured features of an nf-feature map (state size n): their rows of H (dense dh/dxv in the first 7
    columns, dh/dy on the feature's 3 columns), isotropic R blocks and an innovation nu.  Returns the ABI's pieces
    (feats, Hxv, Hy, R as K x 2 x 2) and the dense H and R of the same update."""
    feats = rng.permutation(nf)[:K].astype(np.int32)
    Hxv = np.zeros((2 * K, 13))
    Hxv[:, :7] = rng.standard_normal((2 * K, 7)) * 60
    Hy = rng.standard_normal((2 * K, 3)) * 300
    var = rng.uniform(1, 4, K)
    R = np.zeros((K, 2, 2))
    R[:, 0, 0] = R[:, 1, 1] = var
    nu = rng.standard_normal(2 * K) * 2
    H = np.zeros((2 * K, n))
    H[:, :13] = Hxv
    for k, f in enumerate(feats):
        H[2 * k:2 * k + 2, 13 + 3 * f:16 + 3 * f] = Hy[2 * k:2 * k + 2]
    return feats, Hxv, Hy, R, nu, H, np.kron(np.diag(var), np.eye(2))


def check_streams_against_oracle(ctx, oracles, picks, scenes_of, frame):
    """Step the oracles of `picks` on `frame` and compare them with the context's streams after its step: map size,
    selection, flags, match positions and counters exactly, state within RTOL_TEST, P exactly symmetric."""
    for s in picks:
        o = oracles[s]
        o.step(scenes_of(s).frames[frame])
        fg, fo = ctx.features(s), o.features()
        assert ctx.num_features(s) == o.num_features, s
        assert (fg["select_rank"] == fo["select_rank"]).all() and (fg["flags"] == fo["flags"]).all(), s
        ok = (fo["flags"] & 2) > 0
        assert (fg["z"][ok] == fo["z"][ok]).all(), s
        assert (fg["attempted"] == fo["attempted"]).all() and (fg["successful"] == fo["successful"]).all(), s
        xg, Pg = ctx.get_state(s)
        assert_state_close(xg, Pg, *o.get_state())
        assert np.abs(Pg - Pg.T).max() == 0.0


def recipe_scene(cap, nf, n_bad, n_out, stream_id=0, n_frames=3):
    """A C4 scene (fixed +-20 px search) with nf features that selects up to `cap` per frame, n_bad of them with a
    template of noise (selected, never found) and n_out moved 3 m sideways (never visible, never selected): every
    frame measures m = 2 (nf - n_bad - n_out) rows.  Which features are spoiled is drawn from a seeded permutation."""
    sc = synth.make_scene("C4", stream_id=stream_id, n_frames=n_frames, n_features=nf)
    sc.n_select = cap
    rng = np.random.default_rng(1000 * cap + 7 * nf + stream_id)
    perm = rng.permutation(nf)
    sc.x0 = sc.x0.copy()
    for i in perm[:n_out]:
        sc.x0[13 + 3 * i] += 3.0
    sc.patches = sc.patches.copy()
    for i in perm[n_out:n_out + n_bad]:
        sc.patches[i] = rng.integers(0, 256, sc.patches[i].shape, dtype=np.uint8)
    return sc


def random_puinv(rng, n, lo, hi, iso_fraction=0.5):
    out = np.zeros((n, 3))
    for i in range(n):
        a, b = rng.uniform(lo, hi, 2)
        r = 0.0 if rng.random() < iso_fraction else rng.uniform(-0.8, 0.8)
        if rng.random() < iso_fraction:
            b = a
        Si = np.linalg.inv(np.array([[a * a / 9, r * a * b / 9], [r * a * b / 9, b * b / 9]]))
        out[i] = [Si[0, 0], Si[0, 1], Si[1, 1]]
    return out


__all__ = ["sl2", "synth", "np"]
