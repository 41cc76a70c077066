#!/usr/bin/env python
"""K4d measurements (pgp_topk_distinct, pgp_distinct_dev): python tools/distinct_run.py [--hyp N] [--reps R] [--out FILE]

1. Whether it pays, on the configs[2] / C3 workload of tools/configs_run.py (4 objects, each with its own segment, StoCS generation
   of N hypotheses, weighted scoring; the box's three 180 degree turns registered as symmetries): how many of the plain top-64
   survive suppression at 1 cm / 10 degrees and at 0.5 cm / 5 degrees, and -- after pgp_refine_batch of the plain top-64 and of
   the distinct 64 from a 4096-pool -- how many distinct placements (1 cm / 10 degrees, same symmetries) each refined set holds,
   with the best refined pose's error against ground truth.
2. Cost: device events around pgp_distinct_dev for 1 and 4 lists x 4096 -> 64, with 0 and 3 symmetries, and around pgp_topk_dev
   (4096) for scale; median of R calls each.
3. The chain for 4 objects on one scene: score (pgp_score_generated) -> top-4096 (pgp_topk_dev) -> distinct 64 (pgp_distinct_dev)
   -> pgp_refine_batch_dev, queued with no host stop and ended by one synchronise, against the same chain through host calls
   (pgp_score_generated, pgp_topk_distinct, pgp_centred_to_pose, pgp_refine_batch); host clock, median of R, outputs compared.
   The device chain refines all 4 x 64 rows (identity padding after each list's kept ones), the host chain the kept rows only, so
   the selection stage alone (score -> top-4096 -> distinct, one synchronise) is timed in both forms too.
The GPU's name and power limit are read in the same run."""
import argparse, json, math, subprocess, sys, time
sys.path.insert(0, '.')
import numpy as np, torch
from oracle.select_port import distinct
from physimglobalpose_b200 import synth
from physimglobalpose_b200.engine import PoseEngine

ap = argparse.ArgumentParser()
ap.add_argument('--hyp', type=int, default=1_000_000, help='hypotheses generated per object (C3: 1M)')
ap.add_argument('--reps', type=int, default=21)
ap.add_argument('--out', default=None)
a = ap.parse_args()

FLIPS = [np.diag(d) for d in ([-1.0, -1.0, 1.0], [-1.0, 1.0, -1.0], [1.0, -1.0, -1.0])]
TH = {"1cm_10deg": (0.01, math.radians(10.0)), "0.5cm_5deg": (0.005, math.radians(5.0))}
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
res = {"gpu": smi.splitlines()[0] if smi else "unknown", "hyp_per_object": a.hyp}

e = PoseEngine(0)
objs = [synth.make_segment_problem(2000, 2000, 0.005, seed=100 + k) for k in range(4)]


def n_placements(eng, k, poses44):
    """distinct placements among camera-frame poses: greedy suppression at 1 cm / 10 degrees with the box symmetries"""
    T = eng.pose_to_centred(k, poses44).reshape(-1, 12)
    return int(len(distinct(T, np.arange(len(T)), len(T), 0.01, math.cos(math.radians(10.0)), FLIPS)))


def refine(eng, k, seg, poses44):
    return eng.refine_batch([seg], [(k, 0, np.zeros((0, 4, 4)), poses44)])[0][0]


# ---- 1. whether it pays
pays = []
for k, prob in enumerate(objs):
    e.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    e.set_model(k, prob.model_xyz, prob.model_nrm)
    e.set_symmetries(k, FLIPS)
    e.build_ppf_map(k)
    n = e.generate_pcs(k, seed=5 + k, max_hyp=a.hyp, n_bases=max(a.hyp // 100, 1), max_quads_per_base=100, mode=1)
    e.score_generated(k, "weighted")
    top = e.topk(k, 64)
    row = dict(obj=k, hypotheses=n)
    for name, (d, ang) in TH.items():
        row[f"top64_survivors_{name}"] = len(e.topk_distinct(k, 64, 64, d, ang))
        row[f"distinct64_from_4096_{name}"] = len(e.topk_distinct(k, 4096, 64, d, ang))
    dis = e.topk_distinct(k, 4096, 64, *TH["1cm_10deg"])
    for name, recs in (("top64", top), ("distinct64", dis)):
        P = refine(e, k, prob.scene_xyz, e.centred_to_pose(k, recs["T"]))
        row[f"{name}_refined_placements"] = n_placements(e, k, P)
        errs = [synth.pose_error(p, prob.gt_pose) for p in P]
        row[f"{name}_refined_best_dt_m"] = float(min(x[0] for x in errs))
        row[f"{name}_refined_within_1cm_10deg"] = int(sum(1 for x in errs if x[0] <= 0.01 and x[1] <= math.radians(10.0)))
    pays.append(row)
    print(json.dumps(row), flush=True)
res["pays"] = pays

# ---- 2. cost, on one scene with the four models (pools = the real top-4096 of each object)
scene = objs[0]
e.set_scene(scene.scene_xyz, scene.scene_nrm, scene.delta)
M, K = 4096, 64
pool = torch.zeros(4 * M * 64, dtype=torch.uint8, device="cuda")
for k, prob in enumerate(objs):
    e.set_model(k, prob.model_xyz, prob.model_nrm)
    e.build_ppf_map(k)
    e.generate_pcs(k, seed=5 + k, max_hyp=a.hyp, n_bases=max(a.hyp // 100, 1), max_quads_per_base=100, mode=1)
    e.score_generated(k, "weighted")
    e.topk_device(k, M, 0, pool[k * M * 64:(k + 1) * M * 64])
out = torch.zeros(4 * K * 64, dtype=torch.uint8, device="cuda")
poses = torch.zeros((4 * K, 16), dtype=torch.float64, device="cuda")
n_kept = torch.zeros(4, dtype=torch.int32, device="cuda")
topk_out = torch.zeros(M * 64, dtype=torch.uint8, device="cuda")
e.set_stream(torch.cuda.current_stream().cuda_stream)


def timed(fn, reps):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(reps):
        s, t = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record(); fn(); t.record(); t.synchronize()
        ts.append(s.elapsed_time(t))
    return dict(median_ms=float(np.median(ts)), min_ms=float(np.min(ts)), max_ms=float(np.max(ts)))


cost = {}
for n_sym in (0, 3):
    for k in range(4):
        e.set_symmetries(k, FLIPS[:n_sym])
    for n_lists in (1, 4):
        objs_l = list(range(n_lists))
        cost[f"distinct_dev_{n_lists}x4096_to_64_{n_sym}sym"] = timed(
            lambda: e.distinct_device(objs_l, np.arange(n_lists + 1) * M, pool, K, *TH["1cm_10deg"], out, poses, n_kept), a.reps)
cost["topk_dev_4096"] = timed(lambda: e.topk_device(3, M, 0, topk_out), a.reps)      # last scored batch: object 3
res["cost"] = cost
print(json.dumps(cost), flush=True)

# ---- 3. the chain, 4 objects on one scene, box symmetries registered
for k in range(4):
    e.set_symmetries(k, FLIPS)
segs = [p.scene_xyz for p in objs]
seg_dev = torch.from_numpy(np.concatenate(segs)).cuda()
seg_off = np.concatenate([[0], np.cumsum([len(s) for s in segs])]).astype(np.int64)
items = np.array([(k, k, 0, 0) for k in range(4)], np.int32)
placed = torch.zeros((0, 16), dtype=torch.float64, device="cuda")
status = torch.zeros(1, dtype=torch.int32, device="cuda")
d, ang = TH["1cm_10deg"]


def chain_dev():
    for k in range(4):
        e.score_generated(k, "weighted")
        e.topk_device(k, M, 0, pool[k * M * 64:(k + 1) * M * 64])
    e.distinct_device(list(range(4)), np.arange(5) * M, pool, K, d, ang, out, poses, n_kept)
    e.refine_batch_device(seg_dev, seg_off, placed, items, np.arange(5) * K, poses, status)
    e.synchronize()


def chain_host():
    got = []
    for k in range(4):
        e.score_generated(k, "weighted")
        recs = e.topk_distinct(k, M, K, d, ang)
        got.append((k, k, np.zeros((0, 4, 4)), e.centred_to_pose(k, recs["T"])))
    return e.refine_batch(segs, got)


def wall(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter(); r = fn(); ts.append(time.perf_counter() - t0)
    return dict(median_ms=1e3 * float(np.median(ts)), min_ms=1e3 * float(np.min(ts)), max_ms=1e3 * float(np.max(ts))), r


def select_dev():
    for k in range(4):
        e.score_generated(k, "weighted")
        e.topk_device(k, M, 0, pool[k * M * 64:(k + 1) * M * 64])
    e.distinct_device(list(range(4)), np.arange(5) * M, pool, K, d, ang, out, poses, n_kept)
    e.synchronize()


def select_host():
    for k in range(4):
        e.score_generated(k, "weighted")
        e.topk_distinct(k, M, K, d, ang)


chain = {"note": "device rows: 4 x 64 poses refined, the rows after each list's kept ones are identity padding; host rows: the kept poses only"}
chain["device"], _ = wall(chain_dev, a.reps)
nk = n_kept.cpu().numpy()
P = poses.cpu().numpy().reshape(4, K, 4, 4)
chain["status"] = int(status.item())
chain["host"], host_res = wall(chain_host, a.reps)
chain["select_only_device"], _ = wall(select_dev, a.reps)
chain["select_only_host"], _ = wall(select_host, a.reps)
chain["n_kept"] = nk.tolist()
chain["device_equals_host"] = bool(all(np.array_equal(P[k, :nk[k]], host_res[k][0]) for k in range(4)))
res["chain"] = chain
print(json.dumps(chain), flush=True)
e.set_stream(None)
e.close()
print(json.dumps(res))
if a.out:
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
