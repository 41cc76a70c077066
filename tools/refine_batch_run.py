"""pgp_refine_batch and pgp_refine_batch_dev against the per-item loop of single calls they replace (timing, with a bitwise check
of the arms): python tools/refine_batch_run.py [--reps N] [--out FILE]

Shapes, each for the point-to-point and the point-to-plane fit:
  frame:   the C4 frame of tools/configs_run.py -- 4 objects x their top-64 generated poses, each against the other three objects'
           ground truth shifted 5 cm; loop = pgp_mcts_tricp x 4 (point) or pgp_remove_explained + pgp_tricp_plane x 4 (plane).
  rollout: 320 items of one pose each, each object against a random 0-3 of the others (tests/test_gpu_refine_batch.py's shape);
           loop = one single call (or two) per item.
  kernel:  one item, 64 poses, nothing placed: pgp_tricp / pgp_tricp_plane (the single kernel instances) against the batch
           (the batched instances) on identical work.
Arms: loop (the single calls), batch (pgp_refine_batch: host arrays in and out), dev (pgp_refine_batch_dev: segments, placed rows
and poses resident in device memory, the poses reset from a device copy before each call; timed from the call to a device
synchronise).  After a warm-up round the arms alternate; every call ends in a device synchronise.  Reports the median and min-max
wall time per call, with the GPU's name and power limit read in the same run."""
import argparse, json, subprocess, sys, time
sys.path.insert(0, '.')
import numpy as np, torch
from physimglobalpose_b200 import synth
from physimglobalpose_b200.engine import PoseEngine

ap = argparse.ArgumentParser()
ap.add_argument('--reps', type=int, default=7)
ap.add_argument('--out', default=None, help='also write the result as JSON to this file')
a = ap.parse_args()
THR = 0.008

e = PoseEngine(0)
objs = [synth.make_segment_problem(2000, 2000, 0.005, seed=100 + k) for k in range(4)]
segs = [p.scene_xyz for p in objs]
top_poses = []
for k, prob in enumerate(objs):                        # as tools/configs_run.py's C4
    e.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    e.set_model(k, prob.model_xyz, prob.model_nrm)
    e.generate_pcs(k, seed=5 + k, max_hyp=10000, mode=0)
    e.score_generated(k, "weighted")
    top_poses.append(e.centred_to_pose(k, e.topk(k, 64)["T"]))


def shifted(js):
    P = np.array([objs[j].gt_pose for j in js]).reshape(-1, 4, 4)
    P[:, 0, 3] += 0.05
    return P


def single(metric, item):
    obj, s, placed, poses = item
    if len(placed) == 0:
        return (e.tricp if metric == "point" else e.tricp_plane)(obj, segs[s], poses) + (len(segs[s]),)
    if metric == "point":
        return e.mcts_tricp(obj, segs[s], placed, poses, THR)
    mask = e.remove_explained(obj, segs[s], placed, THR)
    return e.tricp_plane(obj, segs[s][~mask], poses) + (int((~mask).sum()),)


rng = np.random.default_rng(41)
rollout = []
for r in range(320):
    k = int(rng.integers(4))
    which = rng.permutation([j for j in range(4) if j != k])[:int(rng.integers(4))]
    rollout.append((k, k, shifted(which), top_poses[k][r % 64][None]))
shapes = {"frame": [(k, k, shifted([j for j in range(4) if j != k]), top_poses[k]) for k in range(4)],
          "rollout": rollout,
          "kernel": [(0, 0, np.zeros((0, 4, 4)), top_poses[0])]}


class Resident:
    """One shape's arrays for pgp_refine_batch_dev: the bulk data on the device, the structure on the host."""

    def __init__(self, items):
        placed = [np.asarray(it[2], np.float64).reshape(-1, 16) for it in items]
        poses = [np.asarray(it[3], np.float64).reshape(-1, 16) for it in items]
        lo = np.concatenate([[0], np.cumsum([len(p) for p in placed])])
        self.rec = np.array([(it[0], it[1], lo[i], len(placed[i])) for i, it in enumerate(items)], np.int32)
        self.seg_off = np.concatenate([[0], np.cumsum([len(s) for s in segs])]).astype(np.int64)
        self.pose_off = np.concatenate([[0], np.cumsum([len(p) for p in poses])]).astype(np.int64)
        dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
        self.seg, self.placed = dev(np.concatenate(segs)), dev(np.concatenate(placed))
        self.poses0 = dev(np.concatenate(poses))
        self.poses = self.poses0.clone()
        n = self.poses.shape[0]
        self.iters = torch.zeros(n, dtype=torch.int32, device="cuda")
        self.energy = torch.zeros(n, dtype=torch.float32, device="cuda")
        self.nun = torch.zeros(len(items), dtype=torch.int32, device="cuda")
        self.status = torch.zeros(1, dtype=torch.int32, device="cuda")

    def call(self, metric):
        e.refine_batch_device(self.seg, self.seg_off, self.placed, self.rec, self.pose_off, self.poses, self.status, self.iters, self.energy,
                              self.nun, metric=metric, threshold=THR)

    def results(self):
        assert int(self.status.cpu()[0]) == 0
        P, it, en, nun = self.poses.cpu().numpy(), self.iters.cpu().numpy(), self.energy.cpu().numpy(), self.nun.cpu().numpy()
        return [(P[a:b].reshape(-1, 4, 4), it[a:b], en[a:b], int(nun[i])) for i, (a, b) in enumerate(zip(self.pose_off[:-1], self.pose_off[1:]))]


def run(arm, metric, items, res):
    if arm == "dev":
        res.poses.copy_(res.poses0)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    if arm == "dev":
        res.call(metric)
        e.synchronize()
    else:
        out = [single(metric, it) for it in items] if arm == "loop" else e.refine_batch(segs, items, metric, THR)
    torch.cuda.synchronize()
    t = (time.perf_counter() - t0) * 1e3
    return t, (res.results() if arm == "dev" else out)


def same(x, y):
    return all(np.ascontiguousarray(u).tobytes() == np.ascontiguousarray(v).tobytes() for u, v in zip(x[:3], y[:3])) and int(x[3]) == int(y[3])


smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "reps": a.reps, "shapes": {}}
ARMS = ("loop", "batch", "dev")
for name, items in shapes.items():
    resident = Resident(items)
    for metric in ("point", "plane"):
        ms = {arm: [] for arm in ARMS}
        for rep in range(a.reps + 1):                    # rep 0 warms up (module load, target grids, scratch)
            outs = {}
            for arm in ARMS:
                t, outs[arm] = run(arm, metric, items, resident)
                if rep:
                    ms[arm].append(t)
            for arm in ARMS[1:]:
                assert len(outs["loop"]) == len(outs[arm]) and all(same(x, y) for x, y in zip(outs["loop"], outs[arm])), \
                    f"{name}/{metric}: {arm} differs from the single calls"
        row = {"items": len(items), "poses": int(sum(len(it[3]) for it in items)), "bitwise_equal": True,
               "iters_mean": round(float(np.mean(np.concatenate([o[1] for o in outs["batch"]]))), 2)}
        for arm in ARMS:
            t = np.array(ms[arm])
            row[arm] = {"ms_median": round(float(np.median(t)), 3), "ms_min": round(float(t.min()), 3), "ms_max": round(float(t.max()), 3)}
        row["speedup_median"] = round(row["loop"]["ms_median"] / row["batch"]["ms_median"], 2)
        res["shapes"][f"{name}_{metric}"] = row
        print(name, metric, *(f"{arm} {row[arm]}" for arm in ARMS), "x", row["speedup_median"])
print(json.dumps(res))
if a.out:
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
