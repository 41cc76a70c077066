"""TrICP of the top-64 generated poses on a 2k-pt segment / 2k-pt model request (timing):
python tools/tricp_run.py [--metric point|plane|both] [--reps N] [--out FILE]

--metric both runs the point-to-point fit (pgp_tricp) and the point-to-plane fit (pgp_tricp_plane) alternately on the same 64
poses and reports, for each, the host time per call (ending in the copy-back, so the device has finished) and the iteration
counts, with the GPU's name and power limit read in the same run."""
import argparse, json, subprocess, sys, time
sys.path.insert(0, '.')
import numpy as np, torch
from physimglobalpose_b200 import synth
from physimglobalpose_b200.engine import PoseEngine

ap = argparse.ArgumentParser()
ap.add_argument('--metric', choices=('point', 'plane', 'both'), default='point')
ap.add_argument('--reps', type=int, default=20)
ap.add_argument('--out', default=None, help='also write the result as JSON to this file')
a = ap.parse_args()

seg = synth.make_segment_problem(2000, 2000, 0.005, seed=5)
e = PoseEngine(0)
e.set_scene(seg.scene_xyz, seg.scene_nrm, seg.delta); e.set_model(1, seg.model_xyz, seg.model_nrm)
e.generate_pcs(1, seed=3, max_hyp=20000)
e.score_generated(1, "weighted")
top = e.topk(1, 64)
poses = e.centred_to_pose(1, top["T"])
fits = {'point': e.tricp, 'plane': e.tricp_plane}
names = ['point', 'plane'] if a.metric == 'both' else [a.metric]
ms = {n: [] for n in names}
last = {}
for rep in range(a.reps + 1):                            # rep 0 warms up (module load, target grid, scratch)
    for n in names:
        torch.cuda.synchronize(); t0 = time.perf_counter()
        out, iters, en = fits[n](1, seg.scene_xyz, poses, trim=0.5, ratio=0.99, max_iter=100)
        dt = time.perf_counter() - t0
        if rep:
            ms[n].append(dt * 1e3)
        last[n] = (out, iters, en)
smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
gt = seg.gt_pose
res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi[0] if smi else None, "poses": len(poses), "segment": len(seg.scene_xyz),
       "model": len(seg.model_xyz), "reps": a.reps, "fits": {}}
for n in names:
    out, iters, en = last[n]
    t = np.array(ms[n])
    dt = np.linalg.norm(out[:, :3, 3] - gt[:3, 3], axis=1)
    res["fits"][n] = {"ms_per_call": round(float(np.median(t)), 3), "ms_min": round(float(t.min()), 3), "ms_max": round(float(t.max()), 3),
                      "iters_mean": round(float(iters.mean()), 2), "iters_max": int(iters.max()),
                      "iters_hist": {int(k): int(v) for k, v in zip(*np.unique(iters, return_counts=True))},
                      "poses_within_5mm_of_gt": int((dt < 0.005).sum())}
    print(n, 'ms', res["fits"][n]["ms_per_call"], 'poses/s', round(len(poses) / (res["fits"][n]["ms_per_call"] * 1e-3)), 'iters mean',
          res["fits"][n]["iters_mean"], 'max', res["fits"][n]["iters_max"])
print(json.dumps(res))
if a.out:
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
