"""The EKF update (csrc/update.cu) in every launch shape it can take.

Which code runs is decided by the map capacity Nmax, the number of streams in the launch and the measurement count m of
each stream (the rules are restated, with their lines in update.cu, in `launch_shape` below):
* staged single-stream updates with host rows at the boundaries of every `upd_solve_kernel<NP>` instantiation, below
  capacity, at K = 1 and over a conditioning sweep, against an extended-precision (80-bit long double) Cholesky update;
* batched fused steps whose streams have different m and n in one launch, in the four launch shapes a context uses,
  each stream bit-identical to its twin in an 8-stream context, which is checked against the oracle;
* a CPU test that enumerates the reachable shape combinations and fails if the case lists stop covering one.
"""
import os
import re
import time

import numpy as np
import pytest

from gpu_util import (check_streams_against_oracle, ctx_from_scenes, oracle_slam_from_scene,
                      random_measurements, recipe_scene, state_err, synth)

UPDATE_CU = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scenelib2_b200", "csrc",
                         "update.cu")

# Accuracy of a staged update: err_gpu <= max(4 * min(err_oracle, err_fp64_cholesky), FLOOR), every error against the
# extended-precision reference in gpu_util.state_err's scale (relative to sqrt(P_ii P_jj), sigma_i for x).
# Measured on a B200 over STAGED_CASES: worst err_gpu 2.6e-13 (covariance, capacity 104, m = 208) outside the
# conditioning sweep, where the state error is at most 9e-15; 2.4e-13 at cond(S) = 1e4.  FLOOR is 10x the worst.
# (With one Newton step instead of two in upd_chol's pivot rsqrt the covariance error rises to 1e-11 - 1e-10 and every
# staged case fails.)
FLOOR = 2.5e-12


# ---- launch shape rules (csrc/update.cu) ---------------------------------------------------------------------------
def keven(nmax):                      # update.cu:54 upd_keven
    return (nmax + 1) & ~1


def solve_np(nmax):                   # update.cu:1443-1447 solve_panels / solve_np
    p = (2 * keven(nmax) + 15) // 16
    return 4 if p <= 4 else 7 if p <= 7 else 10 if p <= 10 else 13 if p <= 13 else 16


def launch_shape(nmax, stream_cnt, m):
    """(NP, FULL or guarded, upd_hp form, solve grid) of one stream's update in a launch of stream_cnt streams."""
    np_ = solve_np(nmax)
    one_cta = stream_cnt >= 2 * 148                          # update.cu:1515-1516 hp_blocks
    piped = one_cta and 13 + 3 * nmax <= 320                  # update.cu:1521 (SL2_TUNE_HP_PIPELINED on by default)
    hp = "hp2" if piped else ("hp-1cta" if one_cta else "hp-spread")
    walk = np_ <= 13 and stream_cnt >= 148                    # update.cu:1545
    m8 = (m + 7) & ~7
    full = np_ <= 13 and m8 >= 16 * np_ - 8                   # update.cu:1016-1017 (SPLIT == NP iff NP <= 13, :965)
    return np_, "full" if full else "guarded", hp, "walk" if walk else "slab"


# the lines launch_shape restates; if one of them changes, the rules above (and with them the case lists) must follow
RULE_LINES = [
    r"inline int solve_panels\(int Nmax\) \{ return \(2 \* upd_keven\(Nmax\) \+ 15\) / 16; \}",
    r"return p <= 4 \? 4 : \(p <= 7 \? 7 : \(p <= 10 \? 10 : \(p <= 13 \? 13 : 16\)\)\);",
    r"const int hp_blocks = stream_cnt >= 2 \* 148 \? 1 : hp_all;",
    r"const bool piped = d\.tune\[SL2_TUNE_HP_PIPELINED\] != 0 && hp_blocks == 1 && SL2_NXV \+ 3 \* d\.Nmax <= HP_THREADS;",
    r"constexpr int HP_THREADS = 320;",
    r"const bool walk = np <= 13 && stream_cnt >= 148;",
    r"const int m8 = \(m \+ 7\) & ~7;",
    r"const bool full = L::SPLIT == NP && m8 >= 16 \* NP - 8;",
    r"static constexpr int SPLIT = NP > 13 \? 6 : NP;",
    r"__host__ __device__ inline int upd_keven\(int Nmax\) \{ return \(Nmax \+ 1\) & ~1; \}",
]


# ---- case lists ----------------------------------------------------------------------------------------------------
# staged: (capacity, map features, measured features K, target cond(S) or None); m = 2 K
STAGED_CASES = []
for _cap, _np in ((32, 4), (56, 7), (80, 10), (104, 13)):
    for _m in (16 * _np - 16, 16 * _np - 14, 16 * _np, 16 * _np - 30):   # last guarded, first FULL, all panels, 2 mod 16
        STAGED_CASES.append((_cap, _cap, _m // 2, None))
STAGED_CASES += [(128, 128, 32, None),      # NP = 16, m = 64: the REUSE barrier is not reached
                 (128, 128, 33, None),      # m = 66: reached, no second-generation panel has rows
                 (128, 128, 49, None),      # m = 98: the first second-generation panel is staged
                 (128, 128, 128, None),     # m = 256
                 (128, 30, 30, None),       # map well below capacity
                 (80, 61, 61, None),        # odd n + 1 = 197: the one-column tail of the last column group
                 (128, 128, 1, None)]       # K = 1
COND_CASES = [(56, 56, 49, c) for c in (1e4, 1e8, 1e11)]
STAGED_CASES += COND_CASES

# batched: per capacity, 8 stream recipes (map features, failing templates, features out of view) and the m each one
# measures every frame.  NP <= 13: m = 0, 2, the last guarded m (16 NP - 16), the first FULL m (16 NP - 14), the full
# map, a FULL m inside the range, a guarded map well below capacity and a guarded m = 2 (mod 16).  NP = 16: the same
# with the REUSE boundaries of the staged list (66, 98, 64) in place of the FULL ones.
BATCH_CAPS = (32, 56, 80, 100, 104, 128)
CULL_CAPS = (80, 128)
BATCH_STREAMS = (160, 296)          # besides the 8-stream twin; 296 also runs as two groups of 148


def _batch_recipes(cap):
    np_ = solve_np(cap)
    kg, kf = (8 * np_ - 8, 8 * np_ - 7) if np_ <= 13 else (33, 49)
    small = cap // 3 | 1
    half = cap // 2
    k6 = max(k for k in range(1, half - 3) if k % 8 == 1)      # 2 k6 = 2 (mod 16)
    return [(cap, 0, 0),                          # every feature measured: the largest m
            (cap, 0, cap),                        # nothing in view: m = 0
            (cap - 1, 0, cap - 2),                # odd map, one feature in view: m = 2
            (cap, min(cap - kf, 10), max(cap - kf - 10, 0)),  # m = 2 kf: failing templates (beyond 10: out of view)
            (cap - 3, 0, cap - 3 - kg),           # odd map, m = 2 kg, out of view
            (small, 0, 0),                        # map well below capacity, all measured
            (half, (half - k6) // 2, half - k6 - (half - k6) // 2),
            (cap, 1, 1) if np_ <= 13 else (cap, 32, 64)]      # FULL inside the range / NP = 16: m = 64


BATCH_RECIPES = {cap: _batch_recipes(cap) for cap in BATCH_CAPS}


def recipe_m(recipe):
    nf, bad, out = recipe
    return 2 * (nf - bad - out)


def _covered():
    got = set()
    for cap, nf, K, _ in STAGED_CASES:
        got.add(launch_shape(cap, 1, 2 * K))
    for cap, recipes in BATCH_RECIPES.items():
        for cnt in (8,) + BATCH_STREAMS + (148,):             # 148: one group of a two-group 296-stream step
            for r in recipes:
                if recipe_m(r) > 0:
                    got.add(launch_shape(cap, cnt, recipe_m(r)))
    return got


def _reachable():
    out = set()
    for nmax in range(1, 129):
        for cnt in (1, 147, 148, 295, 296, 1000):
            for m in range(2, 2 * keven(nmax) + 1, 2):
                out.add(launch_shape(nmax, cnt, m))
    return out


def test_rules_match_update_cu():
    src = open(UPDATE_CU).read()
    missing = [r for r in RULE_LINES if not re.search(r, src)]
    assert not missing, "update.cu no longer has these launch-shape rules; update launch_shape and the case lists: %s" \
        % missing


def test_case_lists_cover_every_reachable_launch_shape():
    reach, got = _reachable(), _covered()
    assert len(reach) == 28                   # NP 4/7/10: 3 grids x 2, NP 13: 4 x 2, NP 16: 2
    assert reach - got == set(), sorted(reach - got)
    # and the other per-stream branches: m = 0 beside m > 0, maps below capacity (odd and even), two column chunks in
    # upd_hp (n > 320) in every hp form, m = 2 in one launch with the largest m
    for cap, recipes in BATCH_RECIPES.items():
        ms = [recipe_m(r) for r in recipes]
        assert 0 in ms and 2 in ms and max(ms) == 2 * cap, cap
        assert any(r[0] < cap and r[0] % 2 for r in recipes) and any(r[0] < cap and r[0] % 2 == 0 for r in recipes)
        assert len(set(ms)) == 8, (cap, ms)
        np_ = solve_np(cap)
        kinds = {launch_shape(cap, 8, m)[1] for m in ms if m > 0}
        assert kinds == ({"full", "guarded"} if np_ <= 13 else {"guarded"}), cap
    assert any(13 + 3 * r[0] > 320 for cap in BATCH_CAPS for r in BATCH_RECIPES[cap]
               if launch_shape(cap, 296, 2)[2] == "hp-1cta")
    assert any(13 + 3 * nf > 320 for _, nf, _, _ in STAGED_CASES)
    assert {solve_np(c) for c in BATCH_CAPS} == {4, 7, 10, 13, 16}


# ---- extended-precision reference ----------------------------------------------------------------------------------
def _need_longdouble():
    if np.finfo(np.longdouble).nmant < 63:
        pytest.skip("np.longdouble has %d mantissa bits here (needs the 64-bit significand of x86-64's 80-bit format)"
                    % np.finfo(np.longdouble).nmant)


def kalman_update_ext(oracle, x, P, H, R, nu):
    """The update in the Cholesky form of the kernels, in np.longdouble: S = H P H^T + R = U^T U, Y = U^-T [H P | nu],
    P - Y^T Y, x + Y^T w; then normalise_state's Jacobian (of the updated x) and the symmetrisation of GoOneStep
    (monoslam.cpp:137,143-150).  Returns long double x, P."""
    L = np.longdouble
    x, P, H, R, nu = (np.asarray(a, np.float64).astype(L) for a in (x, P, H, R, nu))
    n, m = x.size, nu.size
    HP = H @ P
    S = HP @ H.T + R
    S = 0.5 * (S + S.T)
    U = np.zeros((m, m), L)
    for k in range(m):                         # S = U^T U, one row of U per step
        d = S[k, k] - U[:k, k] @ U[:k, k]
        if d <= 0:
            raise np.linalg.LinAlgError("S is not positive definite")
        U[k, k] = np.sqrt(d)
        U[k, k + 1:] = (S[k, k + 1:] - U[:k, k] @ U[:k, k + 1:]) / U[k, k]
    B = np.concatenate([HP, nu[:, None]], axis=1)
    Y = np.zeros_like(B)
    for k in range(m):                         # U^T Y = B, forward substitution
        Y[k] = (B[k] - U[:k, k] @ Y[:k]) / U[k, k]
    Yp, w = Y[:, :n], Y[:, n]
    x = x + Yp.T @ w
    P = P - Yp.T @ Yp
    J = np.asarray(oracle.dxvnorm_by_dxv(np.asarray(x[:13], np.float64)), np.float64).astype(L)
    P[:13] = J @ P[:13]                        # J P J^T with J = diag(J13, I)
    P[:, :13] = P[:, :13] @ J.T
    return x, 0.5 * (P + P.T)


def _oracle_update(oracle, x, P, H, Rfull, nu):
    """The reference's own algorithm (kalman.cpp:100-115, explicit S^-1) in FP64, normalised and symmetrised."""
    xo, Po = oracle.kalman_update_dense(x, P, H, Rfull, nu)
    J = np.eye(x.size)
    J[:13, :13] = oracle.dxvnorm_by_dxv(xo[:13])
    Po = J @ Po @ J.T
    return xo, 0.5 * (Po + Po.T)


def _cholesky_update_fp64(oracle, x, P, H, Rfull, nu):
    """The kernels' Cholesky form in FP64 through LAPACK (scipy), normalised and symmetrised.  Far more accurate than
    the explicit inverse when S is ill-conditioned, so it is the yardstick that stays meaningful there."""
    import scipy.linalg as sl
    U = sl.cholesky(H @ P @ H.T + Rfull)
    Y = sl.solve_triangular(U, np.c_[H @ P, nu], trans="T")
    x = x + Y[:, :-1].T @ Y[:, -1]
    P = P - Y[:, :-1].T @ Y[:, :-1]
    J = np.eye(x.size)
    J[:13, :13] = oracle.dxvnorm_by_dxv(x[:13])
    P = J @ P @ J.T
    return x, 0.5 * (P + P.T)


def _condition(rng, sc, nf, K, target):
    """Measurements whose S has cond(S) ~ target: the 13 camera columns give S a part of rank <= 7; scaling them up
    (and R down with them) against the feature part raises cond(S).  The scale is found by bisection on log cond."""
    base = random_measurements(rng, sc.n, nf, K)
    if target is None:
        return base, None

    def scaled(a):
        feats, Hxv, Hy, R, nu, H, Rfull = (np.array(v) for v in base)
        Hxv[:, :7] *= a
        H[:, :13] = Hxv
        R /= a
        Rfull /= a
        return feats, Hxv, Hy, R, nu, H, Rfull

    def cond(a):
        H, Rfull = scaled(a)[5], scaled(a)[6]
        return np.linalg.cond(H @ sc.P0 @ H.T + Rfull)

    lo, hi = 0.0, 8.0                         # log10 of the scale
    for _ in range(40):
        mid = 0.5 * (lo + hi)
        lo, hi = (mid, hi) if cond(10 ** mid) < target else (lo, mid)
    a = 10 ** (0.5 * (lo + hi))
    return scaled(a), cond(a)


def test_extended_reference_matches_oracle_dense(oracle):
    """The long double Cholesky update agrees with the oracle's FP64 dense update (explicit S^-1) and with an FP64
    Cholesky update through LAPACK to FP64 rounding on small well-conditioned cases, so it computes the same operation.
    (The explicit inverse loses about two more digits in P where a measurement shrinks a variance by 10^2 - 10^3.)"""
    _need_longdouble()
    worst_o = worst_c = 0.0
    for nf, K in ((3, 1), (5, 5), (12, 7), (20, 20)):
        sc = synth.make_scene("C4", n_frames=1, n_features=nf)
        rng = np.random.default_rng(31 * nf + K)
        feats, Hxv, Hy, R, nu, H, Rfull = random_measurements(rng, sc.n, nf, K)
        xe, Pe = kalman_update_ext(oracle, sc.x0, sc.P0, H, Rfull, nu)
        eo = max(state_err(*_oracle_update(oracle, sc.x0, sc.P0, H, Rfull, nu), xe, Pe))
        ec = max(state_err(*_cholesky_update_fp64(oracle, sc.x0, sc.P0, H, Rfull, nu), xe, Pe))
        print("nf=%d K=%d: vs extended: oracle %.2e, FP64 Cholesky %.2e" % (nf, K, eo, ec))
        worst_o, worst_c = max(worst_o, eo), max(worst_c, ec)
    assert worst_o <= 1e-12 and worst_c <= 1e-13, (worst_o, worst_c)


# ---- staged update matrix ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("cap,nf,K,cond", STAGED_CASES)
def test_staged_update_shape_against_extended_reference(oracle, cap, nf, K, cond):
    """One stream, host rows (sl2_ekf_update) at capacity `cap`, an nf-feature map, K measured features: the CUDA
    update is as accurate as the better of the reference's algorithm and LAPACK's Cholesky form in FP64, both
    measured against the long double reference (or within FLOOR of it)."""
    _need_longdouble()
    sc = synth.make_scene("C4", n_frames=1, n_features=nf)
    ctx = ctx_from_scenes([sc], max_features=cap)
    rng = np.random.default_rng(cap * 100003 + nf * 1000 + K)
    (feats, Hxv, Hy, R, nu, H, Rfull), cS = _condition(rng, sc, nf, K, cond)
    ctx.ekf_update(0, feats, Hxv, Hy, R, nu)
    xg, Pg = ctx.get_state(0)
    ctx.close()
    assert np.abs(Pg - Pg.T).max() == 0.0
    xe, Pe = kalman_update_ext(oracle, sc.x0, sc.P0, H, Rfull, nu)
    xo, Po = _oracle_update(oracle, sc.x0, sc.P0, H, Rfull, nu)
    xc, Pc = _cholesky_update_fp64(oracle, sc.x0, sc.P0, H, Rfull, nu)
    eg, eo, ec = state_err(xg, Pg, xe, Pe), state_err(xo, Po, xe, Pe), state_err(xc, Pc, xe, Pe)
    cS = cS if cS is not None else np.linalg.cond(H @ sc.P0 @ H.T + Rfull)
    print("cap=%d nf=%d m=%d NP=%d %s cond(S)=%.1e: err x / P: gpu %.2e %.2e | oracle %.2e %.2e | FP64 Cholesky "
          "%.2e %.2e" % (cap, nf, 2 * K, solve_np(cap), launch_shape(cap, 1, 2 * K)[1], cS, *eg, *eo, *ec))
    for g, o, c, what in zip(eg, eo, ec, ("state", "covariance")):
        assert g <= max(4 * min(o, c), FLOOR), "%s error %.3e (oracle %.3e, FP64 Cholesky %.3e)" % (what, g, o, c)


# ---- batched fused-step matrix -------------------------------------------------------------------------------------
def _snapshot(ctx, s):
    x, P = ctx.get_state(s)
    f = ctx.features(s)
    return ctx.num_features(s), x, P, {k: f[k].copy() for k in ("z", "flags", "attempted", "successful",
                                                                "select_rank")}


def _assert_same(a, b, what):
    assert a[0] == b[0], ("map size", what)
    assert a[1].shape == b[1].shape and (a[1] == b[1]).all(), ("x", what)
    assert (a[2] == b[2]).all(), ("P", what)
    for k in a[3]:
        assert (a[3][k] == b[3][k]).all(), (k, what)


def _run_twin(oracle, cap, recipes, scenes, steps):
    """8 streams, one per recipe, every stream against its oracle at every step.  Returns the snapshots per step."""
    ctx = ctx_from_scenes(scenes, max_features=cap)
    oracles = [oracle_slam_from_scene(oracle, sc) for sc in scenes]
    snaps = []
    for t in range(steps):
        k = t % scenes[0].frames.shape[0]
        ctx.set_frames(0, np.stack([sc.frames[k] for sc in scenes]))
        ctx.step(0)
        ctx.sync()
        check_streams_against_oracle(ctx, oracles, range(len(scenes)), lambda s: scenes[s], k)
        snap = [_snapshot(ctx, s) for s in range(len(scenes))]
        if t < 3:   # before any failing feature can be culled, every recipe measures the m it was built for
            for r, (rec, sn) in enumerate(zip(recipes, snap)):
                fl = sn[3]["flags"]
                m = 2 * int(((fl & 3) == 3).sum())
                assert m == recipe_m(rec), (cap, r, t, m, recipe_m(rec))
        snaps.append(snap)
    ctx.close()
    return snaps


def _run_batch(cap, scenes, B, groups, steps, twin):
    recipe_of = lambda s: (5 * s) % len(scenes)
    ctx = ctx_from_scenes([scenes[recipe_of(s)] for s in range(B)], max_features=cap)
    ctx.set_step_groups(groups)
    picks = sorted({0, 1, 2, 7, B // 2 - 1, B // 2, B - 1})
    for t in range(steps):
        k = t % scenes[0].frames.shape[0]
        ctx.set_frames(0, np.stack([scenes[recipe_of(s)].frames[k] for s in range(B)]))
        ctx.step(0)
        ctx.sync()
        every = range(B) if t == steps - 1 else picks
        for s in every:
            _assert_same(_snapshot(ctx, s), twin[t][recipe_of(s)], (cap, B, groups, t, s))
    ctx.close()


def _scenes(cap, n_frames=3):
    return [recipe_scene(cap, *r, stream_id=i, n_frames=n_frames) for i, r in enumerate(BATCH_RECIPES[cap])]


@pytest.mark.gpu
@pytest.mark.parametrize("cap", BATCH_CAPS)
def test_batched_step_shapes_bit_identical_to_twin(oracle, cap):
    """Fused steps whose streams measure m = 0, 2, guarded, FULL and the largest m in one launch, at capacity `cap`:
    the 8-stream twin (upd_hp rows spread over CTAs, slab solve) against the oracle, and 160 streams (spread, walk),
    296 streams (one upd_hp CTA per stream, walk or slab by NP) and 296 streams as two groups of 148 (the second one
    at stream_lo = 148) bit-identical to the twin, stream by stream: the launch shape never changes a bit."""
    t0 = time.time()
    scenes = _scenes(cap)
    twin = _run_twin(oracle, cap, BATCH_RECIPES[cap], scenes, 3)
    for B in BATCH_STREAMS:
        _run_batch(cap, scenes, B, 1, 3, twin)
    _run_batch(cap, scenes, 296, 2, 3, twin)
    print("cap=%d NP=%d m per recipe %s: %.1f s" % (cap, solve_np(cap), [recipe_m(r) for r in BATCH_RECIPES[cap]],
                                                  time.time() - t0))


@pytest.mark.gpu
@pytest.mark.parametrize("cap", CULL_CAPS)
def test_batched_culling_inside_a_batch(oracle, cap):
    """12 steps: the failing templates reach the deletion rule, so some streams shrink below capacity while others
    keep their map, and the later steps run with different n in one launch.  Twin against the oracle at every step;
    296 streams bit-identical to the twin."""
    scenes = _scenes(cap)
    twin = _run_twin(oracle, cap, BATCH_RECIPES[cap], scenes, 12)
    sizes = [sn[0] for sn in twin[-1]]
    assert any(sz < r[0] for sz, r in zip(sizes, BATCH_RECIPES[cap])), sizes      # something was culled
    assert any(sz == r[0] == cap for sz, r in zip(sizes, BATCH_RECIPES[cap])), sizes
    _run_batch(cap, scenes, 296, 1, 12, twin)
    print("cap=%d map sizes after 12 steps: %s" % (cap, sizes))
