"""K8 rendered frames on the test scene: python tools/render_depth_run.py [out.json] [--reps N] [--no-profile]

The test scene of tools/render_cost_run.py: a 640 x 480 frame with the test scene's intrinsics, depth and class mask; three objects
placed on the table near their segments, with tessellated meshes of 12k-20k triangles; 25, 256 and 4096 states of three objects per
call, each object jittered by 2 cm / up to 0.3 rad.  Arms, each timed with CUDA events on the stream the context runs on, after two
warm-up calls, as the median of the repeats:
  loop_host: pgp_render_depth once per state into one reused pair of host frames (depth and slot), the only way to get frames
             without pgp_render_depth_dev (a torch cost on the GPU would still have to upload them again: not included);
  dev:       one pgp_render_depth_dev call into device tensors (depth and slot, n_states x 480 x 640 each);
  cost_dev:  pgp_depth_cost_dev on the same states: the same pipeline with the fused comparison instead of frames.
and, for the observed frame: pgp_set_depth_observation (host arrays) against pgp_set_depth_observation_dev (device tensors).
After the timing, every frame of dev is compared bitwise with pgp_render_depth of its state, and SHA-256 digests of the frames (in
state order) are reported.  A separate torch.profiler pass gives the dev arm's kernel time per phase, with the frame clear apart."""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np
import torch

from physimglobalpose_b200 import synth
from physimglobalpose_b200.engine import PoseEngine

ap = argparse.ArgumentParser()
ap.add_argument("out", nargs="?", default=None, help="also write the report as JSON to this file")
ap.add_argument("--reps", type=int, default=0, help="timed calls per arm and size (default: 20, 5 at 4096 states)")
ap.add_argument("--no-profile", action="store_true", help="skip the torch.profiler pass")
args = ap.parse_args()

G = os.path.join(ROOT, "tests", "golden")
CLASSES = {"kleenex_tissue_box": 8, "expo_dry_erase_board_eraser": 2, "folgers_classic_roast_coffee": 3}
PHASES = {"clear": ("k8_clear",), "vertex": ("k8_vertex",), "setup + binning": ("k8_setup", "k1_scan", "k8_list", "k8_fill"), "tiles": ("k8_tiles",)}
TAU = 0.01


def main():
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    raw = np.repeat(g["depth_raw_rle"][0], g["depth_raw_rle"][1]).astype(np.uint16).reshape(480, 640)
    mask = np.repeat(g["mask_all_rle"][0], g["mask_all_rle"][1]).astype(np.uint8).reshape(480, 640)
    meshes = [synth.box_mesh((0.12, 0.10, 0.24), 37), synth.box_mesh((0.15, 0.05, 0.035), 32), synth.ellipsoid_mesh((0.05, 0.05, 0.075), 64, 128)]
    names = [str(n) for n in g["names"]]
    cents = [g[f"{n}_seg_xyz"].astype(np.float64).mean(0) for n in names]
    e = PoseEngine(0)
    stream = torch.cuda.current_stream()
    e.set_stream(stream.cuda_stream)
    e.set_depth_observation(raw, mask, g["K"])
    for i, (n, (v, t)) in enumerate(zip(names, meshes)):
        e.set_mesh(i, v, t, CLASSES[n])
    rng = np.random.default_rng(0)
    rows, cols = raw.shape

    def states(n):
        out = []
        for _ in range(n):
            P = np.tile(np.eye(4), (3, 1, 1))
            for k in range(3):
                P[k, :3, :3] = synth.rot_axis_angle(rng.normal(size=3), rng.uniform(0, 0.3))
                P[k, :3, 3] = cents[k] + rng.normal(scale=0.02, size=3) + [0, 0, 0.03]
            out.append((np.arange(3, dtype=np.int32), P))
        return out

    def timed(fn, reps):
        fn()                                                   # warm-up: the scratch reaches its size for this batch
        fn()
        ms = []
        for _ in range(reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            fn()
            b.record(stream)
            b.synchronize()
            ms.append(a.elapsed_time(b))
        return {"ms_median": round(float(np.median(ms)), 3), "ms_min": round(float(min(ms)), 3), "ms_max": round(float(max(ms)), 3)}

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    report = {"device": torch.cuda.get_device_properties(0).name, "nvidia_smi": smi, "frame": [rows, cols],
              "triangles_per_object": [len(t) for _, t in meshes], "runs": []}
    lib, ctx = e._lib, e._ctx
    host_d, host_s = np.zeros((rows, cols), np.float32), np.zeros((rows, cols), np.int32)
    for n in (25, 256, 4096):
        st = states(n)
        reps = args.reps or (20 if n < 4096 else 5)
        ids = [i for i, _ in st]
        P = np.ascontiguousarray(np.concatenate([p for _, p in st]).reshape(-1, 16))
        run = {"states": n, "reps": reps, "frame_bytes_depth_and_slot": 2 * n * rows * cols * 4}

        def loop_host():
            for s in range(n):
                rc = lib.pgp_render_depth(ctx, ids[s].ctypes.data, P[3 * s:3 * s + 3].ctypes.data, 3, host_d.ctypes.data, host_s.ctypes.data)
                assert rc == 0, rc

        poses = torch.from_numpy(P).cuda()
        depth = torch.empty((n, rows, cols), dtype=torch.float32, device="cuda")
        slot = torch.empty((n, rows, cols), dtype=torch.int32, device="cuda")
        out = torch.empty((len(P), 5), dtype=torch.int32, device="cuda")
        status, status2 = torch.full((1,), 55, dtype=torch.int32, device="cuda"), torch.full((1,), 55, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()

        def dev():
            e.render_depth_device(ids, poses, depth, status, slot)

        def cost_dev():
            e.depth_cost_device(ids, poses, out, status2, TAU)

        run["loop_host"] = timed(loop_host, reps)
        run["dev"] = timed(dev, reps)
        run["cost_dev"] = timed(cost_dev, reps)
        torch.cuda.synchronize()
        assert int(status.cpu()[0]) == 0 and int(status2.cpu()[0]) == 0
        # every frame of dev against pgp_render_depth of its state, bitwise; digests over the frames in state order
        hd, hs = hashlib.sha256(), hashlib.sha256()
        for a in range(0, n, 256):
            d, s = depth[a:a + 256].cpu().numpy(), slot[a:a + 256].cpu().numpy()
            for k in range(len(d)):
                want_d, want_s = e.render_depth(ids[a + k], P[3 * (a + k):3 * (a + k) + 3])
                assert np.array_equal(d[k].view(np.uint32), want_d.view(np.uint32)) and np.array_equal(s[k], want_s), f"{n}: frame {a + k} differs"
            hd.update(d.tobytes())
            hs.update(s.tobytes())
        counts = out.cpu().numpy()
        assert np.array_equal(counts, e.depth_cost(st, TAU)), f"{n}: cost_dev differs from depth_cost"
        run.update({"bitwise_equal_dev_loop_host": True, "digest_depth": hd.hexdigest()[:16], "digest_slot": hs.hexdigest()[:16],
                    "digest_counts": hashlib.sha256(counts.tobytes()).hexdigest()[:16],
                    "covered_pixels": int(counts[:, 0].sum())})
        if not args.no_profile:
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                dev()
                torch.cuda.synchronize()
            split = {k: 0.0 for k in PHASES}
            for ev in prof.key_averages():
                for k, names_ in PHASES.items():
                    if any(x in ev.key for x in names_):
                        split[k] += ev.device_time_total / 1e3
            run["dev_phase_ms_profiled"] = {k: round(v, 3) for k, v in split.items()}
            if split["clear"] > 0:
                run["clear_GB_per_s"] = round(run["frame_bytes_depth_and_slot"] / (split["clear"] * 1e-3) / 1e9, 1)
        del depth, slot
        torch.cuda.empty_cache()
        report["runs"].append(run)
        print(json.dumps(run), flush=True)
    # the observed frame: host arrays against device tensors
    r_dev = torch.from_numpy(raw.view(np.int16)).cuda()
    m_dev = torch.from_numpy(mask).cuda()
    hist_dev = torch.empty(256, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    obs = {"observation_host": timed(lambda: e.set_depth_observation(raw, mask, g["K"]), 50),
           "observation_dev": timed(lambda: e.set_depth_observation_device(r_dev, m_dev, g["K"], hist_dev), 50)}
    torch.cuda.synchronize()
    assert np.array_equal(hist_dev.cpu().numpy(), e.set_depth_observation(raw, mask, g["K"]))
    report["observation"] = obs
    print(json.dumps(obs))
    print(json.dumps({k: v for k, v in report.items() if k != "runs"}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    e.close()


if __name__ == "__main__":
    main()
