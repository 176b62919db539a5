"""Small end-to-end exercise of every kernel for compute-sanitizer (memcheck / racecheck).
`python tools/sanitize.py update-shapes` runs only the batched EKF update launch shapes at the end."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
from scenelib2_b200 import synth
from gpu_util import ctx_from_scenes, random_puinv, recipe_scene


def update_shapes():
    """One fused step per batched update shape of tests/test_gpu_update_shapes.py, 8 streams of different m and n per
    context: upd_solve_kernel<10> (capacity 80) spread and batched; the walking solve at NP = 4 and 7 (148 streams);
    the one-CTA plain upd_hp with two column chunks (capacity 104, 296 streams); a 296-stream two-group step."""
    from test_gpu_update_shapes import BATCH_RECIPES
    for cap, B, groups in ((80, 8, 1), (80, 296, 1), (32, 148, 1), (56, 148, 1), (104, 296, 1), (80, 296, 2)):
        uniq = [recipe_scene(cap, *r, stream_id=i, n_frames=1) for i, r in enumerate(BATCH_RECIPES[cap])]
        scs = [uniq[(5 * s) % 8] for s in range(B)]
        c = ctx_from_scenes(scs, max_features=cap)
        c.set_step_groups(groups)
        c.set_frames(0, np.stack([sc_.frames[0] for sc_ in scs])); c.step(0); c.sync()
        print("update shape cap=%d streams=%d groups=%d: map sizes %s, state finite: %s" % (
            cap, B, groups, [c.num_features(s) for s in range(8)],
            all(np.isfinite(c.get_state(s)[1]).all() for s in range(0, B, 37))))
        c.close()


if sys.argv[1:] == ["update-shapes"]:
    update_shapes()
    sys.exit(0)

scenes = [synth.make_scene("C2", stream_id=s, n_frames=3, n_features=21, override=(s == 0)) for s in range(2)]
ctx = ctx_from_scenes(scenes, frame_slots=2)
for t in range(3):
    ctx.set_frames(t % 2, np.stack([sc.frames[t] for sc in scenes]))
    ctx.step(t % 2)
ctx.sync()
ctx.set_step_groups(2)                       # staggered stream groups on the internal streams
for t in range(3):
    ctx.step(t % 2)
ctx.sync()
ctx.set_step_groups(1)
ctx.find_best_patch(0, 0, [[100, 80, 180, 140], [5, 5, 60, 50]])   # Shi-Tomasi detector
rng = np.random.default_rng(0)
sc = scenes[0]
n = sc.n_features
u, v, f, b = ctx.patch_search(0, 0, np.arange(n, dtype=np.int32), sc.pix + rng.uniform(-3, 3, (n, 2)),
                              random_puinv(rng, n, 5, 30, 0.3))
ctx.score_map(0, 0, 2, sc.pix[2].astype(float), [0.02, 0.001, 0.03])
ctx.smoe_search(0, 0, 1, random_puinv(rng, 4, 5, 12, 0.5), np.tile(sc.pix[1].astype(float), (4, 1)))
K = 12
pu = random_puinv(rng, K, 4, 10, 0.5)
ctx.measure_particles(0, 0, 1, np.tile(sc.pix[1].astype(float), (K, 1)) + rng.normal(0, 3, (K, 2)), pu,
                      1.0 / (pu[:, 0] * pu[:, 2] - pu[:, 1] ** 2), np.linspace(0.5, 4.5, K), 0.05, np.full(K, 1.0 / K))
ctx.measure_particles(0, 0, -1, np.tile(sc.pix[1].astype(float), (K, 1)), pu, 1.0 / (pu[:, 0] * pu[:, 2] - pu[:, 1] ** 2),
                      np.linspace(0.5, 4.5, K), 0.05, np.full(K, 1.0 / K), patch=sc.patches[2])
ctx.smoe_search_patch(0, 0, sc.patches[3], pu[:4], np.tile(sc.pix[3].astype(float), (4, 1)))
# all partially-initialised features of a stream in one call: particle prediction, score maps, re-weighting
Fp, Kp = 3, 20
ypi = np.zeros((Fp, 6))
ypi[:, 3:] = [[0.1, 0.05, 1.0], [-0.2, 0.1, 1.0], [0.05, -0.15, 1.0]]
ypi[:, 3:] /= np.linalg.norm(ypi[:, 3:], axis=1)[:, None]
Ap = rng.normal(0, 1, (Fp, 19, 19))
Pp = Ap @ Ap.transpose(0, 2, 1) * 2e-6
ctx.measure_partial_features(0, 0, sc.patches[:Fp], ypi, Pp[:, :13, 13:], Pp[:, 13:, 13:],
                             np.tile(np.linspace(0.5, 5, Kp), (Fp, 1)), 0.05, np.full((Fp, Kp), 1.0 / Kp),
                             K=np.array([Kp, Kp - 3, 1], np.int32))
ctx.delete_feature(1, 5)
ctx.ekf_predict(0); ctx.predict_measurements(0); ctx.make_measurements(0, 0); ctx.ekf_update_measured(0)
# staged update with caller-supplied rows (13 dense columns of H: the other instantiation of upd_hp)
ms = 6
nf0 = ctx.num_features(0)
ctx.ekf_update(0, np.array([0, 2, 4], np.int32), rng.normal(0, 1, (ms, 13)), rng.normal(0, 1, (ms, 3)),
               np.tile(np.eye(2) * 4.0, (ms // 2, 1, 1)), rng.normal(0, 0.1, ms))
sc3 = synth.make_scene("C3", n_frames=1, n_features=9)
c3 = ctx_from_scenes([sc3])
c3.set_frames(0, sc3.frames[:1]); c3.step(0); c3.sync()
# round 2: full-size map (13 Cholesky panels, the register-resident solve with bulk copies + mbarriers + warp-pair
# barriers, 15 syrk tiles), 3 streams so that streams differ; ragged m (one template spoiled -> one match fails)
big = [synth.make_scene("C4", stream_id=s, n_frames=2) for s in range(3)]
big[1].patches = big[1].patches.copy()
big[1].patches[7] = rng.integers(0, 256, big[1].patches[7].shape, dtype=np.uint8)
cb = ctx_from_scenes(big, frame_slots=1)
for t in range(2):
    cb.set_frames(0, np.stack([sc_.frames[t] for sc_ in big])); cb.step(0)
cb.sync()
# the BATCHED launch shapes (>= 296 streams): software-pipelined upd_hp, one solve CTA per stream walking the column
# groups on its predicate-free path (m = 56 rows reach the last panel of the 4-panel instantiation), syrk with two
# diagonal tiles per stream (block masks)
uniq = [synth.make_scene("C2", stream_id=s, n_frames=1, n_features=28) for s in range(4)]
many = [uniq[s % 4] for s in range(296)]
cm = ctx_from_scenes(many, frame_slots=1)
cm.set_frames(0, np.stack([sc_.frames[0] for sc_ in many])); cm.step(0); cm.sync()
print("batched: matched", int((cm.features(295)["flags"] & 2).astype(bool).sum()), "of 28, state finite:",
      bool(np.isfinite(cm.get_state(295)[1]).all()))
cm.close()
# device-side map growth
n10 = 13 + 3 * 10
ca = ctx_from_scenes([synth.make_scene("C2", n_frames=1, n_features=10)], max_features=12)
ca.append_feature(0, np.array([0.1, 0.2, 1.5]), scenes[0].xp_org[0], scenes[0].patches[0])
ca.append_feature(0, np.array([0.0, 0.1, 1.2]), scenes[0].xp_org[1], scenes[0].patches[1], np.zeros((n10 + 6, 3)))
print("big state finite:", bool(np.isfinite(cb.get_state(1)[1]).all()), "appended:", ca.num_features(0))
print("found", int(f.sum()), "of", n, "| state finite:", bool(np.isfinite(ctx.get_state(0)[1]).all()),
      bool(np.isfinite(c3.get_state(0)[1]).all()))
update_shapes()
