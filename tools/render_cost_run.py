"""K8 rendered-depth cost on the test scene: python tools/render_cost_run.py [out.json] [--reps N] [--root TREE] [--no-profile]

640 x 480 frame with the test scene's intrinsics, depth and class mask; three objects placed on the table near their segments, with
tessellated meshes of 12k-20k triangles (two boxes, one ellipsoid); 25, 256 and 4096 states of three objects per call, each object
jittered by 2 cm / up to 0.3 rad.  Arms, each timed with CUDA events on the stream the context runs on, after a warm-up, as the
median of the repeats:
  host:       pgp_depth_cost (poses and counts in host memory);
  dev:        pgp_depth_cost_dev, the poses resident in device memory;
  chain_host: an MCTS expansion with a host round trip -- pgp_refine_batch of every state's poses (one item per object: its
              segment of the test scene, its model, nothing placed; max_iter 20), then pgp_depth_cost of the refined poses;
  chain_dev:  the same on the device with no host in between -- pgp_refine_batch_dev into a tensor, then pgp_depth_cost_dev on
              that tensor (the poses are reset from a device copy before each call, outside the timing).
The arms' outputs are checked bitwise (dev against host, chain_dev against chain_host), and SHA-256 digests of the counts and of the
refined poses are reported so that two builds can be compared.  --root runs the library and package of another tree (an older
build has only the host arms).  A separate torch.profiler pass splits the host arm's time over the phases (vertex pass, triangle
setup + binning, tile pass).  There is no reference arm: the reference's OpenGL renderer cannot be built here."""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ap = argparse.ArgumentParser()
ap.add_argument("out", nargs="?", default=None, help="also write the report as JSON to this file")
ap.add_argument("--reps", type=int, default=0, help="timed calls per arm and size (default: 20, 5 at 4096 states)")
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))), help="tree whose build to run")
ap.add_argument("--no-profile", action="store_true", help="skip the torch.profiler pass")
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))
import numpy as np
import torch

from physimglobalpose_b200 import synth
from physimglobalpose_b200.engine import PoseEngine

G = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
CLASSES = {"kleenex_tissue_box": 8, "expo_dry_erase_board_eraser": 2, "folgers_classic_roast_coffee": 3}
PHASES = {"vertex": ("k8_vertex",), "setup + binning": ("k8_setup", "k1_scan", "k8_list", "k8_fill"), "tiles": ("k8_tiles",)}
TAU, MAX_ITER = 0.01, 20


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def main():
    g = np.load(os.path.join(G, "c1_test_scene.npz"))
    raw = np.repeat(g["depth_raw_rle"][0], g["depth_raw_rle"][1]).astype(np.uint16).reshape(480, 640)
    mask = np.repeat(g["mask_all_rle"][0], g["mask_all_rle"][1]).astype(np.uint8).reshape(480, 640)
    meshes = [synth.box_mesh((0.12, 0.10, 0.24), 37), synth.box_mesh((0.15, 0.05, 0.035), 32), synth.ellipsoid_mesh((0.05, 0.05, 0.075), 64, 128)]
    names = [str(n) for n in g["names"]]
    cents = [g[f"{n}_seg_xyz"].astype(np.float64).mean(0) for n in names]
    segs = [g[f"{n}_seg_xyz"] for n in names]
    e = PoseEngine(0)
    has_dev = hasattr(e, "depth_cost_device")
    stream = torch.cuda.current_stream()
    e.set_stream(stream.cuda_stream)
    e.set_depth_observation(raw, mask, g["K"])
    e.set_scene(segs[0], g[f"{names[0]}_seg_nrm"], float(g["delta"]))
    for i, (n, (v, t)) in enumerate(zip(names, meshes)):
        e.set_mesh(i, v, t, CLASSES[n])
        e.set_model(i, g[f"{n}_model_xyz"], g[f"{n}_model_nrm"])
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

    props = torch.cuda.get_device_properties(0)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    report = {"device": props.name, "nvidia_smi": smi, "root": os.path.abspath(args.root), "frame": [480, 640],
              "triangles_per_object": [len(t) for _, t in meshes], "runs": []}
    tris_per_state = sum(len(t) for _, t in meshes)
    seg_xyz = np.ascontiguousarray(np.concatenate(segs))
    seg_off = np.concatenate([[0], np.cumsum([len(s) for s in segs])]).astype(np.int64)
    for n in (25, 256, 4096):
        st = states(n)
        reps = args.reps or (20 if n < 4096 else 5)
        ids = [i for i, _ in st]
        P = np.concatenate([p for _, p in st])
        items = [(k, k, np.zeros((0, 4, 4)), P[3 * s + k][None]) for s in range(n) for k in range(3)]
        run = {"states": n, "reps": reps}
        res = {}

        def host():
            res["host"] = e.depth_cost(st, TAU)

        def chain_host():
            refined = np.concatenate([r[0] for r in e.refine_batch(segs, items, "point", max_iter=MAX_ITER)])
            res["chain_host"] = (refined, e.depth_cost([(i, refined[3 * s:3 * s + 3]) for s, i in enumerate(ids)], TAU))

        run["host"] = timed(host, reps)
        run["chain_host"] = timed(chain_host, reps)
        if has_dev:
            dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()   # noqa: E731
            poses0 = dev(P.reshape(-1, 16))
            poses, refined = poses0.clone(), poses0.clone()
            out = torch.zeros((len(P), 5), dtype=torch.int32, device="cuda")
            out2 = torch.zeros_like(out)
            status, status2 = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
            seg_dev, placed_dev = dev(seg_xyz), torch.zeros((0, 16), dtype=torch.float64, device="cuda")
            rec = np.array([(k, k, 0, 0) for _ in range(n) for k in range(3)], np.int32)
            pose_off = np.arange(len(items) + 1, dtype=np.int64)
            torch.cuda.synchronize()

            def dev_arm():
                e.depth_cost_device(ids, poses, out, status, TAU)

            def chain_dev(a=None):
                refined.copy_(poses0)                          # the reset runs before the start event
                if a is not None:
                    a.record(stream)
                e.refine_batch_device(seg_dev, seg_off, placed_dev, rec, pose_off, refined, status2, max_iter=MAX_ITER)
                e.depth_cost_device(ids, refined, out2, status, TAU)

            run["dev"] = timed(dev_arm, reps)
            chain_dev(), chain_dev()
            ms = []
            for _ in range(reps):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                chain_dev(a)
                b.record(stream)
                b.synchronize()
                ms.append(a.elapsed_time(b))
            run["chain_dev"] = {"ms_median": round(float(np.median(ms)), 3), "ms_min": round(float(min(ms)), 3), "ms_max": round(float(max(ms)), 3)}
            torch.cuda.synchronize()
            assert int(status.cpu()[0]) == 0 and int(status2.cpu()[0]) == 0
            assert np.array_equal(out.cpu().numpy(), res["host"]), f"{n}: dev differs from host"
            assert refined.cpu().numpy().tobytes() == res["chain_host"][0].tobytes(), f"{n}: refined poses differ"
            assert np.array_equal(out2.cpu().numpy(), res["chain_host"][1]), f"{n}: chain_dev differs from chain_host"
            run["bitwise_equal_across_arms"] = True
        counts = res["host"]
        covered = int(counts[:, 0].sum())
        t = run["host"]["ms_median"]
        run.update({"states_per_s": round(n / t * 1e3), "triangles_per_s": round(n * tris_per_state / t * 1e3), "covered_pixels": covered,
                    "agree_fraction": round(float(counts[:, 1].sum()) / max(covered, 1), 4),
                    "digest_host_counts": digest(counts), "digest_chain": digest(*res["chain_host"])})
        if not args.no_profile:
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
                e.depth_cost(st, TAU)
                torch.cuda.synchronize()
            split = {k: 0.0 for k in PHASES}
            for ev in prof.key_averages():
                for k, names_ in PHASES.items():
                    if any(x in ev.key for x in names_):
                        split[k] += ev.device_time_total / 1e3
            run["host_phase_ms_profiled"] = {k: round(v, 3) for k, v in split.items()}
        report["runs"].append(run)
        print(json.dumps(run))
    print(json.dumps({k: v for k, v in report.items() if k != "runs"}))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(report, f, indent=1)
    e.close()


if __name__ == "__main__":
    main()
