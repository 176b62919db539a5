"""ORACLE — TEST INFRASTRUCTURE ONLY.

ctypes binding of oracle/liboracle.so (the CPU restatement) and, when present, of
oracle/_ref/libsl2ref.so (the reference's own improc sources compiled unmodified).
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs
may import this module; nothing under scenelib2_b200/ does.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = os.path.join(_HERE, "liboracle.so")
_REF = os.path.join(_HERE, "_ref", "libsl2ref.so")
SCENELIB2_SRC_FILE = os.path.join(_HERE, "_ref", "scenelib2_src")   # the SceneLib2 tree _ref was built from

u8p = C.POINTER(C.c_uint8)
i32p = C.POINTER(C.c_int32)
f64p = C.POINTER(C.c_double)


class OrcConfig(C.Structure):
    _fields_ = [
        ("width", C.c_int32), ("height", C.c_int32),
        ("fku", C.c_double), ("fkv", C.c_double), ("u0", C.c_double), ("v0", C.c_double),
        ("kd1", C.c_double), ("sd", C.c_double),
        ("delta_t", C.c_double),
        ("number_of_features_to_select", C.c_int32),
        ("boxsize", C.c_int32),
        ("search_override", C.c_double * 3),
        ("minimum_attempted_measurements_of_feature", C.c_int32),
        ("successful_match_fraction", C.c_double),
    ]


def build(force=False):
    """Compile liboracle.so (and _ref when /root/reference exists).  Building is not using."""
    have_ref = os.path.isdir("/root/reference/scenelib2/improc")
    refm = os.path.join(_HERE, "_ref", "libsl2refmodels.so")
    libs = [_LIB] + ([_REF, refm, SCENELIB2_SRC_FILE] if have_ref else [])
    stale = force or any(not os.path.exists(p) for p in libs)
    if not stale:
        newest_src = 0.0
        for root, _dirs, files in os.walk(_HERE):
            if os.sep + "_ref" in root or "__pycache__" in root:
                continue
            for f in files:
                if f.endswith((".cpp", ".hpp", ".h")) or f in ("Makefile", "Eigen", "StdVector"):
                    newest_src = max(newest_src, os.path.getmtime(os.path.join(root, f)))
        stale = newest_src > min(os.path.getmtime(p) for p in libs)
    if stale:
        if not force and os.path.exists(_LIB):
            os.utime(os.path.join(_HERE, "capi.cpp"))  # make only tracks liboracle.so's own sources
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(t)


def _u8(a):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    return a, _p(a, u8p)


def _f64(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, _p(a, f64p)


_lib = None
_ref = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB)
        L.orc_correlate2_warning.restype = C.c_double
        L.orc_slam_create.restype = C.c_void_p
        L.orc_slam_run.restype = C.c_double
        L.orc_slam_run_pinned.restype = C.c_double
        for name in ("orc_slam_destroy", "orc_slam_add_feature", "orc_slam_set_state",
                     "orc_slam_get_state", "orc_slam_step", "orc_slam_predict",
                     "orc_slam_update", "orc_slam_normalise", "orc_slam_finish",
                     "orc_slam_get_features"):
            getattr(L, name).restype = None
        _lib = L
    return _lib


def scenelib2_src():
    """The SceneLib2 source tree oracle/_ref was built from, or None when _ref was not built here."""
    if not os.path.exists(SCENELIB2_SRC_FILE):
        return None
    d = open(SCENELIB2_SRC_FILE).read().strip()
    return d if os.path.isdir(d) else None


def ref():
    """The reference's own improc code (None when the prebuilt .so is absent)."""
    global _ref
    if _ref is None and os.path.exists(_REF):
        R = C.CDLL(_REF)
        R.ref_correlate2_warning.restype = C.c_double
        _ref = R
    return _ref


_REFM = os.path.join(_HERE, "_ref", "libsl2refmodels.so")
_refm = None


def ref_models():
    """The reference's own MotionModel / Camera / FullFeatureModel code compiled against the arithmetic
    stand-in of oracle/stubs_arith (None when the prebuilt .so is absent)."""
    global _refm
    if _refm is None and os.path.exists(_REFM):
        _refm = C.CDLL(_REFM)
    return _refm


def make_config(width=320, height=240, fku=195.0, fkv=195.0, u0=162.0, v0=125.0, kd1=9e-6, sd=1.0,
                delta_t=0.033333333, n_select=10, boxsize=11, search_override=(0.0, 0.0, 0.0),
                min_attempts=10, match_fraction=0.5):
    c = OrcConfig()
    c.width, c.height = width, height
    c.fku, c.fkv, c.u0, c.v0, c.kd1, c.sd = fku, fkv, u0, v0, kd1, sd
    c.delta_t = delta_t
    c.number_of_features_to_select = n_select
    c.boxsize = boxsize
    for i in range(3):
        c.search_override[i] = search_override[i]
    c.minimum_attempted_measurements_of_feature = min_attempts
    c.successful_match_fraction = match_fraction
    return c


# ---- primitives -------------------------------------------------------------------------------
def correlate2_warning(patch, image, x1, y1, use_ref=False):
    """A1.  patch (B,B) u8, image (H,W) u8 -> (corr, sd_patch, sd_image)."""
    patch, pp = _u8(patch)
    image, ip = _u8(image)
    sd0, sd1 = C.c_double(), C.c_double()
    if use_ref:
        r = ref().ref_correlate2_warning(pp, patch.shape[1], patch.shape[0], patch.shape[1],
                                         patch.shape[0], ip, image.shape[1], image.shape[0],
                                         int(x1), int(y1), C.byref(sd0), C.byref(sd1))
    else:
        r = lib().orc_correlate2_warning(pp, patch.shape[1], patch.shape[1], patch.shape[0], ip,
                                         image.shape[1], int(x1), int(y1), C.byref(sd0),
                                         C.byref(sd1))
    return r, sd0.value, sd1.value


def elliptical_search(image, patches, centres, puinv3):
    """A2 batched.  patches (n,B,B), centres (n,2), puinv3 (n,3) -> u,v (int32), found (u8), best."""
    image, ip = _u8(image)
    patches, pp = _u8(patches)
    centres, cp = _f64(centres)
    puinv3, qp = _f64(puinv3)
    n, B = patches.shape[0], patches.shape[1]
    u = np.zeros(n, np.int32)
    v = np.zeros(n, np.int32)
    found = np.zeros(n, np.uint8)
    best = np.zeros(n, np.float64)
    lib().orc_elliptical_search_batch(ip, image.shape[1], image.shape[0], pp, B, n, cp, qp,
                                      _p(u, i32p), _p(v, i32p), _p(found, u8p), _p(best, f64p))
    return u, v, found, best


def search_box(width, height, B, centre, puinv3):
    centre, cp = _f64(centre)
    puinv3, qp = _f64(puinv3)
    box = np.zeros(6, np.int32)
    lib().orc_search_box(width, height, B, cp, qp, _p(box, i32p))
    return box


def score_map(image, patch, centre, puinv3):
    """Scores of one feature over its clamped bounding box, urel-major."""
    image, ip = _u8(image)
    patch, pp = _u8(patch)
    centre, cp = _f64(centre)
    puinv3, qp = _f64(puinv3)
    B = patch.shape[0]
    box = search_box(image.shape[1], image.shape[0], B, centre, puinv3)
    nu, nv = max(0, box[1] - box[0] + 1), max(0, box[3] - box[2] + 1)
    corr = np.zeros((nu, nv), np.float64)
    sd = np.zeros((nu, nv), np.float64)
    inside = np.zeros((nu, nv), np.uint8)
    if nu and nv:
        lib().orc_score_map(ip, image.shape[1], image.shape[0], pp, B, cp, qp, _p(corr, f64p),
                            _p(sd, f64p), _p(inside, u8p))
    return box, corr, sd, inside


def puinv_from_S(S):
    S, sp = _f64(np.asarray(S, np.float64).reshape(2, 2).T)  # col-major
    out = np.zeros(3)
    lib().orc_puinv_from_S(sp, _p(out, f64p))
    return out


def smoe_search(image, patch, puinv3, centres, use_ref=False):
    """A11.  K ellipses sharing one template."""
    image, ip = _u8(image)
    patch, pp = _u8(patch)
    puinv3, qp = _f64(puinv3)
    centres, cp = _f64(centres)
    K = puinv3.shape[0]
    ru = np.zeros(K, np.int32)
    rv = np.zeros(K, np.int32)
    rf = np.zeros(K, np.uint8)
    best = np.zeros(K, np.float64)
    if use_ref:
        ref().ref_smoe_search(ip, image.shape[1], image.shape[0], pp, patch.shape[0], K, qp, cp,
                              _p(ru, i32p), _p(rv, i32p), _p(rf, u8p))
    else:
        lib().orc_smoe_search(ip, image.shape[1], image.shape[0], pp, patch.shape[0], K, qp, cp,
                              _p(ru, i32p), _p(rv, i32p), _p(rf, u8p), _p(best, f64p))
    return ru, rv, rf, best


def find_best_patch(image, boxsize, region, ubest=-1, vbest=-1, use_ref=False):
    """N3.  Shi-Tomasi best patch in region = (ustart, vstart, ufinish, vfinish)."""
    image, ip = _u8(image)
    region = np.ascontiguousarray(region, np.int32)
    u, v, ev = C.c_int32(ubest), C.c_int32(vbest), C.c_double(0.0)
    f = ref_models().ref_find_best_patch if use_ref else lib().orc_find_best_patch
    f(ip, image.shape[1], image.shape[0], boxsize, _p(region, i32p), C.byref(u), C.byref(v), C.byref(ev))
    return u.value, v.value, ev.value


def elliptical_search_ref(image, patch, centre, puinv3, u0=-7, v0=-9):
    """The reference's own MonoSLAM::elliptical_search (monoslam.cpp:401-477) -> found, u, v (u, v keep their
    input values on failure: quirk Q6)."""
    image, ip = _u8(image)
    patch, pp = _u8(patch)
    centre, cp = _f64(centre)
    puinv3, qp = _f64(puinv3)
    u, v = C.c_int32(u0), C.c_int32(v0)
    ok = ref_models().ref_elliptical_search(ip, image.shape[1], image.shape[0], pp, patch.shape[0], cp, qp,
                                            C.byref(u), C.byref(v))
    return ok, u.value, v.value


def measure_feature_ref(image, patch, h, S):
    """The reference's own MonoSLAM::measure_feature (monoslam.cpp:368-386), 11x11 patch -> found, z (2)."""
    image, ip = _u8(image)
    patch, pp = _u8(patch)
    h, hp = _f64(h)
    S, sp = _colmajor(S)
    z = np.full(2, -1.0)
    ok = ref_models().ref_measure_feature(ip, image.shape[1], image.shape[0], pp, hp, sp, _p(z, f64p))
    return ok, z


def particle_set_S_ref(S):
    """The reference's own Particle::set_S (feature_init_info.cpp:55-63): S (2,2) -> Sinv (2,2), det S."""
    S, sp = _colmajor(S)
    Sinv = np.zeros((2, 2), order="F")
    det = C.c_double(0.0)
    ref_models().ref_particle_set_S(sp, _p(Sinv, f64p), C.byref(det))
    return Sinv, det.value


def particle_update(h, Sinv3, detS, lam, z_uv, found, prune_threshold, prob):
    """N2.  -> survivors, prob (normalised), keep, cumulative, (mean, variance)."""
    h, hp = _f64(h)
    Sinv3, sp = _f64(Sinv3)
    detS, dp = _f64(detS)
    lam, lp = _f64(lam)
    z_uv = np.ascontiguousarray(z_uv, np.int32)
    found = np.ascontiguousarray(found, np.uint8)
    prob = np.array(prob, np.float64)
    K = prob.shape[0]
    keep = np.zeros(K, np.uint8)
    cum = np.zeros(K)
    mv = np.zeros(2)
    f = lib().orc_particle_update
    f.restype = C.c_int32
    left = f(K, hp, sp, dp, lp, _p(z_uv, i32p), _p(found, u8p), C.c_double(prune_threshold), _p(prob, f64p),
             _p(keep, u8p), _p(cum, f64p), _p(mv, f64p))
    return left, prob, keep, cum, mv


def motion(xv, dt, u=(0.0, 0.0, 0.0), use_ref=False):
    """A5.  -> fv (13), F (13,13), Q (13,13) as numpy (row/col = math indices)."""
    xv, xp = _f64(xv)
    uu, up = _f64(u)
    fv = np.zeros(13)
    F = np.zeros((13, 13), order="F")
    Q = np.zeros((13, 13), order="F")
    f = ref_models().ref_motion if use_ref else lib().orc_motion
    f(xp, up, C.c_double(dt), _p(fv, f64p), _p(F, f64p), _p(Q, f64p))
    return fv, F, Q


def dxvnorm_by_dxv(xv, use_ref=False):
    xv, xp = _f64(xv)
    J = np.zeros((13, 13), order="F")
    if use_ref:
        xn = np.zeros(13)
        ref_models().ref_dxvnorm_by_dxv(xp, _p(J, f64p), _p(xn, f64p))
        return J, xn
    lib().orc_dxvnorm_by_dxv(xp, _p(J, f64p))
    return J


def _colmajor(a):
    a = np.asfortranarray(np.asarray(a, np.float64))
    return a, _p(a, f64p)


def predict_feature(cam8, xv, y, Pxx, Pxy, Pyy, use_ref=False):
    cam8, cp = _f64(cam8)
    xv, xp = _f64(xv)
    y, yp = _f64(y)
    Pxx, a = _colmajor(Pxx)
    Pxy, b = _colmajor(Pxy)
    Pyy, c = _colmajor(Pyy)
    h = np.zeros(2)
    dxv = np.zeros((2, 13), order="F")
    dy = np.zeros((2, 3), order="F")
    R = np.zeros((2, 2), order="F")
    S = np.zeros((2, 2), order="F")
    f = ref_models().ref_predict_feature if use_ref else lib().orc_predict_feature
    f(cp, xp, yp, a, b, c, _p(h, f64p), _p(dxv, f64p), _p(dy, f64p), _p(R, f64p), _p(S, f64p))
    return h, dxv, dy, R, S


def predict_particles(cam8, xv, ypi, lam, Pxx, Pxy, Pyy, use_ref=False):
    """N2 prediction (monoslam.cpp:1347-1400, one feature): K particles -> h (K,2), S (K,2,2), Sinv3 (K,3), detS (K)."""
    cam8, cp = _f64(cam8)
    xv, xp = _f64(xv)
    ypi, yp = _f64(ypi)
    lam = np.ascontiguousarray(lam, np.float64).ravel()
    Pxx, a = _colmajor(Pxx)
    Pxy, b = _colmajor(Pxy)
    Pyy, c = _colmajor(Pyy)
    K = lam.size
    h = np.zeros((K, 2))
    S = np.zeros((K, 4))
    Sinv3 = np.zeros((K, 3))
    det = np.zeros(K)
    if use_ref:
        f = ref_models().ref_predict_particle
        f.restype = None
        for k in range(K):
            hk, Sk, Sik, dk = np.zeros(2), np.zeros(4), np.zeros(4), C.c_double(0.0)
            f(cp, xp, yp, C.c_double(lam[k]), a, b, c, _p(hk, f64p), _p(Sk, f64p), _p(Sik, f64p), C.byref(dk))
            h[k], S[k], Sinv3[k], det[k] = hk, Sk, (Sik[0], Sik[2], Sik[3]), dk.value
    else:
        f = lib().orc_predict_particles
        f.restype = None
        f(cp, xp, yp, C.c_int32(K), _p(lam, f64p), a, b, c, _p(h, f64p), _p(S, f64p), _p(Sinv3, f64p), _p(det, f64p))
    return h, S.reshape(K, 2, 2).transpose(0, 2, 1), Sinv3, det


def visibility_test(cam8, xp, y, xp_org, h, use_ref=False):
    cam8, cp = _f64(cam8)
    xp, a = _f64(xp)
    y, b = _f64(y)
    xp_org, c = _f64(xp_org)
    h, d = _f64(h)
    f = ref_models().ref_visibility_test if use_ref else lib().orc_visibility_test
    return f(cp, a, b, c, d)


def kalman_update_dense(x, P, H, R, nu):
    """A6 dense, as written in kalman.cpp:100-115.  Returns (x_new, P_new)."""
    x = np.array(x, np.float64)
    P = np.array(P, np.float64, order="F")
    H, hp = _colmajor(H)
    R, rp = _colmajor(R)
    nu, np_ = _f64(nu)
    lib().orc_kalman_update_dense(x.size, nu.size, _p(x, f64p), _p(P, f64p), hp, rp, np_)
    return x, P


class Slam:
    """Whole-step oracle (monoslam.cpp:108-180, tracking only)."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.h = C.c_void_p(lib().orc_slam_create(C.byref(cfg)))

    def __del__(self):
        if getattr(self, "h", None):
            lib().orc_slam_destroy(self.h)
            self.h = None

    def add_feature(self, y, xp_org, patch):
        y, a = _f64(y)
        xp_org, b = _f64(xp_org)
        patch, c = _u8(patch)
        lib().orc_slam_add_feature(self.h, a, b, c)

    @property
    def num_features(self):
        return lib().orc_slam_num_features(self.h)

    @property
    def n(self):
        return lib().orc_slam_state_size(self.h)

    def set_state(self, x, P):
        x, a = _f64(x)
        P, b = _colmajor(P)
        lib().orc_slam_set_state(self.h, a, b)

    def get_state(self):
        n = self.n
        x = np.zeros(n)
        P = np.zeros((n, n), order="F")
        lib().orc_slam_get_state(self.h, _p(x, f64p), _p(P, f64p))
        return x, P

    def step(self, frame):
        frame, fp = _u8(frame)
        lib().orc_slam_step(self.h, fp)

    def predict(self):
        lib().orc_slam_predict(self.h)

    def select(self):
        return lib().orc_slam_select(self.h)

    def measure(self, frame):
        frame, fp = _u8(frame)
        return lib().orc_slam_measure(self.h, fp)

    def update(self):
        lib().orc_slam_update(self.h)

    def normalise(self):
        lib().orc_slam_normalise(self.h)

    def finish(self):
        lib().orc_slam_finish(self.h)

    def features(self):
        nf = self.num_features
        out = dict(label=np.zeros(nf, np.int32), h=np.zeros((nf, 2)), z=np.zeros((nf, 2)),
                   S=np.zeros((nf, 4)), flags=np.zeros(nf, np.uint8),
                   attempted=np.zeros(nf, np.int32), successful=np.zeros(nf, np.int32),
                   select_rank=np.zeros(nf, np.int32))
        lib().orc_slam_get_features(self.h, _p(out["label"], i32p), _p(out["h"], f64p),
                                    _p(out["z"], f64p), _p(out["S"], f64p), _p(out["flags"], u8p),
                                    _p(out["attempted"], i32p), _p(out["successful"], i32p),
                                    _p(out["select_rank"], i32p))
        return out


class RefSlam:
    """The REFERENCE'S OWN MonoSLAM (monoslam.cpp, kalman.cpp, feature.cpp, models, improc compiled
    unmodified against oracle/stubs_arith; see oracle/ref_slam_shim.cpp).  Same surface as Slam.
    Built from a scene through the reference's own Init(cfg): the cfg (data/SceneLib2.cfg format) carries the
    camera, parameters, initial state and the first four features; further features go through
    AddNewKnownFeature; the total state / covariance are then set through fill_states / fill_covariances."""

    def __init__(self, sc, workdir):
        R = ref_models()
        R.ref_slam_create.restype = C.c_void_p
        os.makedirs(workdir, exist_ok=True)
        assert sc.n_features >= 4, "MonoSLAM::Init always adds four known features"
        paths = []
        for i in range(sc.n_features):
            pth = os.path.join(workdir, "patch%03d.pgm" % i)
            with open(pth, "wb") as f:
                f.write(b"P5\n%d %d\n255\n" % (sc.boxsize, sc.boxsize) + np.ascontiguousarray(sc.patches[i]).tobytes())
            paths.append(pth)
        lines = ["cam.width = %d;" % sc.width, "cam.height = %d;" % sc.height, "cam.fku = %d;" % sc.cam8[2],
                 "cam.fkv = %d;" % sc.cam8[3], "cam.u0 = %d;" % sc.cam8[4], "cam.v0 = %d;" % sc.cam8[5],
                 "cam.kd1 = %r;" % float(sc.cam8[6]), "cam.sd = %d;" % sc.cam8[7],
                 "params.delta_t = %r;" % float(sc.delta_t),
                 "params.number_of_features_to_select = %d;" % sc.n_select,
                 "params.number_of_features_to_keep_visible = 12;",
                 # data/SceneLib2.cfg:63-69
                 "params.min_lambda = 0.5;", "params.max_lambda = 5.0;", "params.number_of_particles = 100;",
                 "params.standard_deviation_depth_ratio = 0.3;", "params.min_number_of_particles = 20;",
                 "params.prune_probability_threshold = 0.05;",
                 "params.erase_partially_init_feature_after_this_many_attempts = 10;"]
        names = ["rw_x", "rw_y", "rw_z", "qwr_w", "qwr_x", "qwr_y", "qwr_z", "vw_x", "vw_y", "vw_z", "ww_x",
                 "ww_y", "ww_z"]
        for k, nm in enumerate(names):
            lines.append("state.%s = %r;" % (nm, float(sc.x0[k])))
        for i in range(4):
            y = sc.x0[13 + 3 * i:16 + 3 * i]
            lines += ["f%d.yi_%s = %r;" % (i + 1, c, float(v)) for c, v in zip("xyz", y)]
            lines += ["f%d.xp_org_%d = %r;" % (i + 1, k, float(sc.xp_org[i, k])) for k in range(7)]
            lines.append("f%d.identifier = %s;" % (i + 1, paths[i]))
        cfg = os.path.join(workdir, "ref.cfg")
        open(cfg, "w").write("\n".join(lines) + "\n")
        self.R = R
        self.h = C.c_void_p(R.ref_slam_create(cfg.encode()))
        for i in range(4, sc.n_features):
            y, a = _f64(sc.x0[13 + 3 * i:16 + 3 * i])
            xp, b = _f64(sc.xp_org[i])
            R.ref_slam_add_feature(self.h, a, b, paths[i].encode())
        self.width, self.height = sc.width, sc.height
        self.set_state(sc.x0, sc.P0)

    def __del__(self):
        if getattr(self, "h", None):
            self.R.ref_slam_destroy(self.h)
            self.h = None

    def set_params(self, n_select=-1, min_attempts=-1, match_fraction=-1.0):
        self.R.ref_slam_set_params(self.h, n_select, min_attempts, C.c_double(match_fraction))

    @property
    def num_features(self):
        return self.R.ref_slam_num_features(self.h)

    @property
    def n(self):
        return self.R.ref_slam_state_size(self.h)

    def set_state(self, x, P):
        x, a = _f64(x)
        P, b = _colmajor(P)
        self.R.ref_slam_set_state(self.h, a, b)

    def get_state(self):
        n = self.n
        x = np.zeros(n)
        P = np.zeros((n, n), order="F")
        self.R.ref_slam_get_state(self.h, _p(x, f64p), _p(P, f64p))
        return x, P

    def step(self, frame):
        frame, fp = _u8(frame)
        self.R.ref_slam_step(self.h, fp, self.width, self.height)

    def init_partial_feature(self, frame, u, v):
        """MonoSLAM::InitialiseFeature at pixel (u, v) (monoslam.cpp:1211-1236)."""
        frame, fp = _u8(frame)
        self.R.ref_slam_init_partial(self.h, fp, self.width, self.height, int(u), int(v))

    def particle_cycle(self, frame, cap=256):
        """One predict / measure / re-weight cycle of the first partially-initialised feature (see
        ref_slam_particle_cycle).  None when no measurement is made on this step."""
        frame, fp = _u8(frame)
        o = dict(h=np.zeros((cap, 2)), sinv3=np.zeros((cap, 3)), detS=np.zeros(cap), lam=np.zeros(cap),
                 prob_before=np.zeros(cap), z=np.zeros((cap, 2), np.int32), found=np.zeros(cap, np.uint8),
                 prob_after=np.zeros(cap), keep=np.zeros(cap, np.uint8), cum=np.zeros(cap), mean_var=np.zeros(2))
        ka = C.c_int32(0)
        K = self.R.ref_slam_particle_cycle(self.h, fp, self.width, self.height, cap, _p(o["h"], f64p),
                                           _p(o["sinv3"], f64p), _p(o["detS"], f64p), _p(o["lam"], f64p),
                                           _p(o["prob_before"], f64p), _p(o["z"], i32p), _p(o["found"], u8p),
                                           _p(o["prob_after"], f64p), _p(o["keep"], u8p), _p(o["cum"], f64p),
                                           _p(o["mean_var"], f64p), C.byref(ka))
        if K < 0:
            return None
        out = {k: (v[:K] if k != "mean_var" else v) for k, v in o.items()}
        out["K"], out["K_after"] = K, ka.value
        return out

    def features(self):
        nf = self.num_features
        out = dict(label=np.zeros(nf, np.int32), h=np.zeros((nf, 2)), z=np.zeros((nf, 2)),
                   S=np.zeros((nf, 4)), flags=np.zeros(nf, np.uint8),
                   attempted=np.zeros(nf, np.int32), successful=np.zeros(nf, np.int32),
                   select_rank=np.zeros(nf, np.int32))
        self.R.ref_slam_get_features(self.h, _p(out["label"], i32p), _p(out["h"], f64p), _p(out["z"], f64p),
                                     _p(out["S"], f64p), _p(out["flags"], u8p), _p(out["attempted"], i32p),
                                     _p(out["successful"], i32p), _p(out["select_rank"], i32p))
        return out


def run_slams(slams, frames, nsteps, nthreads):
    """Step every Slam nsteps times over its own frame ring; returns wall seconds."""
    n = len(slams)
    handles = (C.c_void_p * n)(*[s.h for s in slams])
    keep = [np.ascontiguousarray(f, np.uint8) for f in frames]
    ptrs = (u8p * n)(*[_p(f, u8p) for f in keep])
    nframes = keep[0].shape[0]
    return lib().orc_slam_run(handles, n, ptrs, nframes, nsteps, nthreads)


def run_slams_pinned(slams, frames, nsteps, nthreads, pin=True):
    """Like run_slams with one thread pinned per usable CPU; returns (wall seconds, gather/scatter seconds summed
    over the streams)."""
    n = len(slams)
    handles = (C.c_void_p * n)(*[s.h for s in slams])
    keep = [np.ascontiguousarray(f, np.uint8) for f in frames]
    ptrs = (u8p * n)(*[_p(f, u8p) for f in keep])
    gs = C.c_double(0.0)
    t = lib().orc_slam_run_pinned(handles, n, ptrs, keep[0].shape[0], nsteps, nthreads, 1 if pin else 0, C.byref(gs))
    return t, gs.value


def hardware_threads():
    return lib().orc_hardware_threads()


def usable_cpus():
    """CPUs this process may use: scheduler affinity capped by the cgroup CPU quota."""
    return lib().orc_usable_cpus()
