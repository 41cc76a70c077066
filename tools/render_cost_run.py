"""K8 rendered-depth cost on the test scene: python tools/render_cost_run.py [out.json]

640 x 480 frame with the test scene's intrinsics, depth and class mask; three objects placed on the table near their segments, with
tessellated meshes of 12k-20k triangles (two boxes, one ellipsoid); 25, 256 and 4096 states of three objects per pgp_depth_cost
call, each object jittered by 2 cm / up to 0.3 rad.  Times come from CUDA events on the stream the context runs on, after a
warm-up, as the median of the repeats.  A separate torch.profiler pass splits the time over the three phases (vertex pass,
triangle setup + binning, tile pass).  There is no reference arm: the reference's OpenGL renderer cannot be built here."""
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from physimglobalpose_b200 import synth
from physimglobalpose_b200.engine import PoseEngine

G = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
CLASSES = {"kleenex_tissue_box": 8, "expo_dry_erase_board_eraser": 2, "folgers_classic_roast_coffee": 3}
PHASES = {"vertex": ("k8_vertex",), "setup + binning": ("k8_setup", "k1_scan", "k8_list", "k8_fill"), "tiles": ("k8_tiles",)}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    raw = np.repeat(g["depth_raw_rle"][0], g["depth_raw_rle"][1]).astype(np.uint16).reshape(480, 640)
    mask = np.repeat(g["mask_all_rle"][0], g["mask_all_rle"][1]).astype(np.uint8).reshape(480, 640)
    meshes = [synth.box_mesh((0.12, 0.10, 0.24), 37), synth.box_mesh((0.15, 0.05, 0.035), 32), synth.ellipsoid_mesh((0.05, 0.05, 0.075), 64, 128)]
    cents = [g[f"{n}_seg_xyz"].astype(np.float64).mean(0) for n in g["names"]]
    e = PoseEngine(0)
    stream = torch.cuda.current_stream()
    e.set_stream(stream.cuda_stream)
    e.set_depth_observation(raw, mask, g["K"])
    for i, (n, (v, t)) in enumerate(zip(g["names"], meshes)):
        e.set_mesh(i, v, t, CLASSES[str(n)])
    rng = np.random.default_rng(0)

    def states(n):
        out = []
        for _ in range(n):
            P = np.tile(np.eye(4), (3, 1, 1))
            for k in range(3):
                P[k, :3, :3] = synth.rot_axis_angle(rng.normal(size=3), rng.uniform(0, 0.3))
                P[k, :3, 3] = cents[k] + rng.normal(scale=0.02, size=3) + [0, 0, 0.03]
            out.append((np.arange(3, dtype=np.int32), P))
        return out

    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    report = {"device": props.name, "nvidia_smi": smi, "frame": [480, 640], "triangles_per_object": [len(t) for _, t in meshes], "runs": []}
    tris_per_state = sum(len(t) for _, t in meshes)
    for n in (25, 256, 4096):
        st = states(n)
        for _ in range(3):
            counts = e.depth_cost(st, 0.01)                    # warm-up: the scratch reaches its size for this batch
        reps = 20 if n < 4096 else 5
        ms = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            counts = e.depth_cost(st, 0.01)
            b.record(stream)
            b.synchronize()
            ms.append(a.elapsed_time(b))
        t = float(np.median(ms))
        covered = int(counts[:, 0].sum())
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            e.depth_cost(st, 0.01)
            torch.cuda.synchronize()
        split = {k: 0.0 for k in PHASES}
        for ev in prof.key_averages():
            for k, names in PHASES.items():
                if any(x in ev.key for x in names):
                    split[k] += ev.device_time_total / 1e3
        run = {"states": n, "ms_per_call": round(t, 3), "ms_min": round(min(ms), 3), "ms_max": round(max(ms), 3),
               "states_per_s": round(n / t * 1e3), "triangles_per_s": round(n * tris_per_state / t * 1e3), "covered_pixels": covered,
               "covered_pixels_per_s": round(covered / t * 1e3), "phase_ms_profiled": {k: round(v, 3) for k, v in split.items()},
               "agree_fraction": round(float(counts[:, 1].sum()) / max(covered, 1), 4)}
        report["runs"].append(run)
        print(json.dumps(run))
    print(json.dumps({k: v for k, v in report.items() if k != "runs"}))
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            json.dump(report, f, indent=1)
    e.close()


if __name__ == "__main__":
    main()
