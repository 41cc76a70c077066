#!/usr/bin/env python
"""Benchmark of the PCS -> LCP hot path (BASELINE.json metric: LCP hypotheses scored per second).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2|c2w|c2d5|c5|c3]      our arm (CUDA, libpgp.so)
  python bench.py --impl reference [...]                                                 the reference's CPU code on the host cores
  python bench.py [...] --dump-outputs DIR      also write what the last timed step computed (counts, scores, merged top-k) as
                                                DIR/<name>.npy; the inputs are seeded, so two builds can be compared array by array

Configs (BASELINE.json `configs`, SURVEY.md 8):
  c2    configs[1], the headline: 2k-pt model, 100k-pt scene, 100k hypotheses per GPU, delta = 1 cm, Verify (count)      weak scaling
  c2w   the same workload through WeightedVerify (the scorer the reference ships)                                         weak
  c2d5  the same at delta = 5 mm (the shipped default, S4/super4pcs_test.cc:20)                                            weak
  c5    configs[4], dense stress: 30k-pt model, 300k-pt scene, 10 M hypotheses per step sharded over the GPUs             strong
  c3    configs[2]: PCS generation (StoCS + PPF map) + WeightedVerify + top-64, 4 objects x 1 M hypotheses per step,
        bases sharded over the GPUs                                                                                        strong

One step = one pass of the hot path over one batch: K3 scores the rank's hypotheses, K4 selects the rank's top 64, the per-rank
records are all-gathered (NCCL, inside libpgp.so: pgp_topk_begin / pgp_topk_end) on the context's exchange stream -- overlapping
the next step's scoring -- and merged.  N > 1 is launched by torchrun, one rank per GPU; torch.distributed is only the launcher's
host channel (NCCL id hand-over, barriers, the max over ranks): nothing of it is on the data path.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the tree may be read-only: leave no __pycache__ behind

TOPK = 64
DUMP_MAX_HYP = 1 << 20                  # per-hypothesis arrays beyond this are dumped as a fixed, seeded sample (<= 20 MB)
METRIC = "LCP hypotheses scored/sec at 1/2/4/8 B200 (2k-pt model, 100k-pt scene)"
UNIT = "hyp/s"
CONFIGS = {
    "c2": dict(n_model=2000, n_scene=100_000, n_hyp=100_000, delta=0.01, mode="count", scaling="weak", metric=METRIC,
               workload="configs[1]: synthetic LCP scoring, 2k-pt model, 100k-pt scene, 100k hypotheses per GPU, delta=1 cm"),
    "c2w": dict(n_model=2000, n_scene=100_000, n_hyp=100_000, delta=0.01, mode="weighted", scaling="weak",
                metric="WeightedVerify hypotheses scored/sec (2k-pt model, 100k-pt scene)",
                workload="configs[1] through WeightedVerify (binary priors): 2k-pt model, 100k-pt scene, 100k hypotheses per GPU, delta=1 cm"),
    "c2d5": dict(n_model=2000, n_scene=100_000, n_hyp=100_000, delta=0.005, mode="count", scaling="weak",
                 metric="LCP hypotheses scored/sec (2k-pt model, 100k-pt scene, delta = 5 mm)",
                 workload="configs[1] at the shipped delta=5 mm: 2k-pt model, 100k-pt scene, 100k hypotheses per GPU"),
    "c5": dict(n_model=30_000, n_scene=300_000, n_hyp=10_000_000, delta=0.01, mode="count", scaling="strong",
               metric="LCP hypotheses scored/sec, dense stress (30k-pt model, 300k-pt scene)",
               workload="configs[4]: dense stress, 30k-pt model, 300k-pt scene, 10M hypotheses per step sharded over the GPUs, delta=1 cm"),
    "c3": dict(n_model=2000, n_scene=2000, n_hyp=1_000_000, delta=0.005, mode="weighted", scaling="strong", objects=4, n_bases=13_000,
               metric="PCS hypotheses generated + LCP-scored/sec (4 objects x 1M hypotheses)",
               workload="configs[2]: PCS congruent-set generation (StoCS + PPF map) + WeightedVerify + top-64, 1M hypotheses per object, "
                        "4 objects, 2k-pt models, 2k-pt segments, delta=5 mm, bases sharded over the GPUs"),
}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, uuid: str | None, period_ms: int = 20):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        cmd = ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", str(period_ms)]
        if uuid:
            cmd += ["-i", uuid]
        try:
            self.p = None if os.environ.get("PGP_BENCH_NO_SAMPLER") == "1" else subprocess.Popen(cmd, stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def wait_started(self, timeout_s: float = 20.0) -> None:
        """Blocks until nvidia-smi has written its first sample: on a fresh box its start-up (driver attach) takes seconds and holds
        driver locks, which stretches a launch-heavy timed region that happens to overlap it (c3: 160 instead of 83 ms per step)."""
        if self.p is None:
            return
        t0 = time.perf_counter()
        while time.perf_counter() - t0 < timeout_s and os.path.getsize(self.f.name) == 0 and self.p.poll() is None:
            time.sleep(0.05)

    def stop(self) -> dict:
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 7:
                continue
            try:
                sm.append(float(c[0])); mx.append(float(c[1]))
            except ValueError:
                continue
            for nm, v in zip(names, c[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def ncu_static(cfg_name: str) -> dict | None:
    """Per-launch figures of the dominant kernel that cannot be measured inside a timed run (ncu replays kernels): DRAM bytes,
    L2 -> L1 sectors and the pipe utilisations of ONE launch, from the committed `ncu --set full` capture of the same command
    (profiles/k3_traffic.json, written by tools/ncu_summary.py).  Static evidence; the file says which capture it came from."""
    try:
        with open(os.path.join(ROOT, "profiles", "k3_traffic.json")) as f:
            t = json.load(f)
        return t.get(cfg_name) or (t if cfg_name == "c2" and "dram_bytes_read" in t else None)
    except Exception:
        return None


def make_inputs(cfg: dict, rank: int, world: int):
    """Scene / model clouds (the same on every rank) and this rank's hypotheses.  weak: H per rank, its own seed; strong: the
    rank's shard of ONE global list of H hypotheses whose content does not depend on the number of ranks."""
    from physimglobalpose_b200 import synth
    from physimglobalpose_b200.sharding import shard_range
    prob = synth.make_problem(cfg["n_model"], cfg["n_scene"], cfg["delta"], seed=1234)
    if cfg["scaling"] == "weak":
        T = synth.make_hypotheses(prob, cfg["n_hyp"], seed=4321 + rank)
        lo = rank * cfg["n_hyp"]
    else:
        lo, hi = shard_range(cfg["n_hyp"], rank, world)
        T = synth.make_hypotheses_range(prob, lo, hi, seed=4321)
    return prob, T, lo


def algorithmic_bytes_per_hyp(prob, T, n_model) -> tuple[float, float, float]:
    """B_hyp = 48 + 4 + N_m (27*8 + 16 k-bar)   (SURVEY.md 8(d)); k-bar from the actual inputs."""
    from physimglobalpose_b200 import synth
    kbar, nonempty = synth.kbar_27(prob, T, max_hyp=512 if n_model <= 4000 else 64)
    return 52.0 + n_model * (27 * 8 + 16.0 * kbar), kbar, nonempty


def oracle_for(prob):
    """The CPU checker: the reference engine itself (oracle/_ref/libs4ref.so, compiled from /root/reference where that exists and
    shipped to the GPU box as a built file) or, without it, the C restatement."""
    from oracle import pyoracle
    args = (prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    if pyoracle.have_ref():
        return pyoracle.RefOracle(*args), "reference"
    pyoracle.build_port()
    return pyoracle.PortOracle(*args), "port"


# ------------------------------------------------------------------------------------------ CPU
def cpu_reference_run(prob, T, seconds_per_step: float, steps: int, warmup: int, mode: str = "count"):
    """Times the reference's own CPU LCP (Match4PCSBase::Verify through oracle/_ref when that .so was built from /root/reference,
    else the C restatement) on all host threads."""
    cores = os.cpu_count() or 1
    o, kind = oracle_for(prob)
    probe = min(len(T), max(cores, 64 * cores if prob.model_xyz.shape[0] <= 4000 else 2 * cores))
    _, s = o.verify_mt(T[:probe], cores)
    rate = probe / max(s, 1e-6)
    sample = int(max(cores, min(len(T), rate * seconds_per_step)))
    times = []
    counts = None
    for i in range(warmup + steps):
        counts, s = o.verify_mt(T[:sample], cores)
        if i >= warmup:
            times.append(s)
    total = sum(times)
    return dict(value=sample * steps / total, unit=UNIT, cores=cores, kind=kind,
                sample=f"first {sample} of the {len(T)} hypotheses per step, {steps} steps, Verify with full counts, {cores} threads"), \
        total / steps * 1e3, counts, sample


def cpu_secondary(prob, T) -> dict:
    """BASELINE.md 3: the reference's WeightedVerify (the shipped scorer) and its kd-tree build (Match4PCSBase::init), timed on one
    host thread next to the device figures of `secondary` (weighted_lcp, scene_grid_build_ms).  A bounded sample: ~2 s."""
    from oracle import pyoracle
    if not pyoracle.have_ref():
        return {}
    args = (prob.scene_xyz, prob.scene_nrm, prob.model_xyz, prob.model_nrm, prob.model_xyz, prob.model_nrm, prob.delta)
    t0 = time.perf_counter()
    o = pyoracle.RefOracle(*args)
    init_ms = (time.perf_counter() - t0) * 1e3
    n = 1000
    t0 = time.perf_counter()
    o.weighted_verify(T[:n])
    dt = time.perf_counter() - t0
    return {"cpu_weighted_verify": {"value": n / dt, "unit": UNIT, "cores": 1, "kind": "reference", "sample": f"first {n} hypotheses, WeightedVerify, 1 thread"},
            "cpu_init_kdtree_ms": {"value": init_ms, "unit": "ms", "what": "Match4PCSBase::init incl. the kd-tree build, 100k-pt scene, 1 thread"}}


def cpu_pcs_run(cfg: dict, steps: int):
    """configs[2] on the host: the reference's own Perform_N_steps in the shipped operMode 1 (StoCS bases, PPF-map pairs,
    WeightedVerify), one object request per step, one thread (the reference is single-threaded here and its matcher is not
    re-entrant).  Its hard caps (100 bases x <= 100 quads, match4pcsBase.cc:290,1858) bound the sample."""
    from oracle import pyoracle
    from physimglobalpose_b200 import synth
    if not pyoracle.have_ref():
        return None
    seg = synth.make_segment_problem(cfg["n_model"], cfg["n_scene"], cfg["delta"], seed=5)
    keys, offs, pairs = ppf_map_host(seg)
    n_tot, t_tot = 0, 0.0
    for s in range(steps):
        # a fresh matcher per request, as the node constructs one per object (S4/super4pcs_test.cc:100): Perform_N_steps is not
        # re-entrant on one instance (its hypothesis lists and best index carry over)
        o = pyoracle.RefOracle(seg.scene_xyz, seg.scene_nrm, seg.model_xyz, seg.model_nrm, seg.model_xyz, seg.model_nrm, seg.delta, srand_seed=100 + s)
        o.set_ppf_map(keys, offs, pairs)
        t0 = time.perf_counter()
        r = o.perform_n_steps(mode=1, seed=100 + s)
        t_tot += time.perf_counter() - t0
        n_tot += len(r["transforms"])
        del o
    return dict(value=n_tot / t_tot, unit="hyp/s", cores=1, kind="reference",
                sample=f"{steps} object requests of Perform_N_steps (operMode 1, 100 bases x <=100 quads = {n_tot // max(steps, 1)} hypotheses each), "
                       f"generation + WeightedVerify, 1 thread"), t_tot / max(steps, 1) * 1e3


def ppf_map_host(seg):
    """PPF map of the model for the CPU arm: built by the numpy restatement of computePPF (oracle/stocs_port.py)."""
    from oracle import stocs_port
    return stocs_port.build_ppf_map(seg.model_xyz, seg.model_nrm)


def run_reference(args, rank):
    if rank != 0:
        return
    cfg = CONFIGS[args.config]
    if args.config == "c3":
        base, ms = cpu_pcs_run(cfg, args.steps)
        sample_n = None
    else:
        prob, T, _ = make_inputs(dict(cfg, n_hyp=min(cfg["n_hyp"], 100_000)), 0, 1)
        base, ms, _, sample_n = cpu_reference_run(prob, T, seconds_per_step=2.0, steps=args.steps, warmup=args.warmup, mode=cfg["mode"])
    line = {"impl": "reference", "metric": cfg["metric"], "value": base["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": cfg["workload"], "hypotheses_per_step": sample_n, "device": "host CPU", "name": args.config},
            "cpu_baseline": base, "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


# ------------------------------------------------------------------------------------------ GPU
class Dist:
    """The launcher's host channel (torch.distributed under torchrun): barrier, max / sum over ranks, NCCL id hand-over."""

    def __init__(self, rank, local_rank, world):
        import torch
        self.torch, self.rank, self.world = torch, rank, world
        torch.cuda.set_device(local_rank)
        if world > 1:
            import torch.distributed as dist
            os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")      # keep stdout to the ONE JSON line
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            self.dist = dist

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def reduce(self, x: float, op="max") -> float:
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX if op == "max" else self.dist.ReduceOp.SUM)
        return float(t.item())

    def gather(self, x: float) -> list:
        """x of every rank, in rank order (the per-rank spread behind a max-over-ranks figure)."""
        if self.world == 1:
            return [x]
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o.item()) for o in out]

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def gpu_uuid(torch, local_rank):
    try:
        return "GPU-" + str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        return None


def timed_ms(torch, stream, fn, reps=5, pre=None):
    out = []
    for _ in range(reps):
        if pre:
            pre()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream); fn(); b.record(stream)
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b))
    return statistics.median(out)


def secondary_metrics(eng, prob, cfg, T_dev, counts_dev, scores_dev, flush, stream) -> dict:
    """SURVEY.md 8(d) secondary figures, measured after the headline (N = 1 only, outside its timed region): the other scoring
    mode on the same workload, scene-grid build time, PCS hypotheses generated/s and TrICP poses refined/s on a test-scene-sized
    object request, the dense-stress shape.  Device-timed with CUDA events."""
    import torch
    from physimglobalpose_b200 import synth
    n_hyp = T_dev.shape[0]
    sec = {}
    other = "weighted" if cfg["mode"] == "count" else "count"
    eng.score_lcp_device(0, T_dev, counts_dev, scores_dev, other)     # (weighted: builds the K1c lists once)
    ms = timed_ms(torch, stream, lambda: eng.score_lcp_device(0, T_dev, counts_dev, scores_dev, other), pre=flush.zero_)
    sec[f"{other}_lcp"] = {"value": n_hyp / ms * 1e3, "unit": UNIT, "kernel_ms": ms,
                           "mode": ("WeightedVerify, binary priors" if other == "weighted" else "Verify (count)") + ", same workload"}
    ms = timed_ms(torch, stream, lambda: eng.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta), reps=3)
    sec["scene_grid_build_ms"] = {"value": ms, "unit": "ms", "what": f"pgp_set_scene: H2D of {len(prob.scene_xyz)} points + K1 grid + K1b labels/lists + K1d"}
    seg = synth.make_segment_problem(2000, 2000, 0.005, seed=5)
    eng.set_scene(seg.scene_xyz, seg.scene_nrm, seg.delta)
    eng.set_model(1, seg.model_xyz, seg.model_nrm)
    n_gen = [0]
    def gen():
        n_gen[0] = eng.generate_pcs(1, seed=3, max_hyp=20000)
    ms = timed_ms(torch, stream, gen, reps=3)
    sec["pcs_generation"] = {"value": n_gen[0] / ms * 1e3, "unit": "hyp generated/s", "ms": ms, "hypotheses": n_gen[0],
                             "what": "operMode 0, 100 bases x <=100 congruent quads, 2k-pt model, 2k-pt segment (pgp_generate_pcs)"}
    eng.score_generated(1, "weighted")
    top = eng.topk(1, 64)
    poses = eng.centred_to_pose(1, top["T"])
    eng.tricp(1, seg.scene_xyz, poses, trim=0.5, ratio=0.99, max_iter=100)
    t0 = time.perf_counter()
    _, iters, _ = eng.tricp(1, seg.scene_xyz, poses, trim=0.5, ratio=0.99, max_iter=100)
    dt = time.perf_counter() - t0
    sec["tricp"] = {"value": len(poses) / dt, "unit": "poses refined/s", "ms": dt * 1e3, "poses": int(len(poses)), "mean_iterations": float(iters.mean()),
                    "what": "top-64 of the generated set, trim 0.5, 2k-pt segment vs 2k-pt model (pgp_tricp, host call incl. copies)"}
    # configs[4] shape on this GPU: 30k-pt model, 300k-pt scene, 1 M hypotheses, both scorers (kernel time alone)
    try:
        c5 = CONFIGS["c5"]
        big = synth.make_problem(c5["n_model"], c5["n_scene"], c5["delta"], seed=1234)
        n5 = 1_000_000
        T5 = torch.from_numpy(synth.make_hypotheses_range(big, 0, n5, seed=4321).reshape(-1, 12).copy()).cuda()
        c5c = torch.zeros(n5, dtype=torch.int32, device="cuda"); c5s = torch.zeros(n5, dtype=torch.float32, device="cuda")
        eng.set_scene(big.scene_xyz, big.scene_nrm, big.delta)
        eng.set_model(2, big.model_xyz, big.model_nrm)
        out = {}
        for mode in ("count", "weighted"):
            eng.score_lcp_device(2, T5, c5c, c5s, mode)
            ms = timed_ms(torch, stream, lambda: eng.score_lcp_device(2, T5, c5c, c5s, mode), reps=2, pre=flush.zero_)
            out[mode] = {"value": n5 / ms * 1e3, "unit": UNIT, "kernel_ms": ms, "point_queries_per_s": n5 * c5["n_model"] / ms * 1e3}
        out["what"] = "configs[4] shape on one GPU: 30k-pt model, 300k-pt scene, 1M hypotheses (first 1M of the config's list), delta = 1 cm; the full 10M line: --config c5"
        sec["c5"] = out
        del T5, c5c, c5s
    except Exception as e:      # a secondary figure must not take the headline down
        sec["c5"] = {"error": repr(e)}
    eng.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    return sec


def sharding_invariance(eng, D: Dist, cfg, prob, stream) -> dict:
    """SURVEY.md 4(4): the SAME hypothesis list sharded `world` ways must give the identical global top-K.  Every rank scores its
    shard of list L (seed 4321, the N = 1 benchmark's list) and the collective pgp_topk merges; rank 0 also scores ALL of L alone
    and selects locally (pgp_topk_dev, no collective) -- the N = 1 answer -- and compares the 64 records byte for byte."""
    import torch
    from physimglobalpose_b200 import synth
    from physimglobalpose_b200.engine import HYP_DTYPE
    from physimglobalpose_b200.sharding import shard_range
    n = min(cfg["n_hyp"], 100_000)
    L = synth.make_hypotheses_range(prob, 0, n, seed=4321)
    lo, hi = shard_range(n, D.rank, D.world)
    Td = torch.from_numpy(L[lo:hi].reshape(-1, 12).copy()).cuda()
    c = torch.zeros(hi - lo, dtype=torch.int32, device="cuda"); s = torch.zeros(hi - lo, dtype=torch.float32, device="cuda")
    eng.score_lcp_device(0, Td, c, s, cfg["mode"])
    merged = eng.topk(0, TOPK, lo)                       # collective
    merged_auto = eng.topk(0, TOPK, -1)                  # collective, PGP_INDEX_AUTO: index bases from the exchanged batch sizes
    out = {"hypotheses": n, "ways": D.world}
    if D.rank == 0:
        Tf = torch.from_numpy(L.reshape(-1, 12).copy()).cuda()
        cf = torch.zeros(n, dtype=torch.int32, device="cuda"); sf = torch.zeros(n, dtype=torch.float32, device="cuda")
        eng.score_lcp_device(0, Tf, cf, sf, cfg["mode"])
        buf = torch.zeros(TOPK * 64, dtype=torch.uint8, device="cuda")
        eng.topk_device(0, TOPK, 0, buf)
        torch.cuda.synchronize()
        single = buf.cpu().numpy().view(HYP_DTYPE)
        out["top64_identical_to_single_gpu"] = bool(merged.tobytes() == single.tobytes())
        out["top64_identical_with_auto_index_base"] = bool(merged_auto.tobytes() == single.tobytes())
    D.barrier()
    return out


def run_scoring(args, D: Dist, local_rank: int):
    import torch

    from physimglobalpose_b200.engine import PoseEngine
    from physimglobalpose_b200.sharding import comm_init_from_env

    cfg = CONFIGS[args.config]
    rank, world = D.rank, D.world
    mode = cfg["mode"]
    prob, T, index_base = make_inputs(cfg, rank, world)
    n_local = len(T)
    n_step_total = cfg["n_hyp"] * world if cfg["scaling"] == "weak" else cfg["n_hyp"]
    peaks, peak_kind = measured_peaks()

    eng = PoseEngine(local_rank)          # no fallback: raises without libpgp.so / a B200
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    no_comm = os.environ.get("PGP_BENCH_NO_COMM") == "1"      # diagnosis only: N independent replicas, no collective at all
    if not no_comm:
        comm_init_from_env(eng, rank, world)  # pgp_comm_init: the communicator lives in libpgp.so
    if os.environ.get("PGP_STREAM_UPLOAD", "1") == "0":       # for captures under ncu, which serialises streams: upload first, then score
        eng.set_option("stream_upload", 0)
    eng.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta)
    eng.set_model(0, prob.model_xyz, prob.model_nrm)
    grid = eng.grid_info()

    T_host = torch.from_numpy(T.reshape(-1, 12).copy()).pin_memory()
    counts_host = [torch.zeros(n_local, dtype=torch.int32).pin_memory() for _ in range(2)]
    scores_host = [torch.zeros(n_local, dtype=torch.float32).pin_memory() for _ in range(2)]
    T_dev = T_host.cuda(non_blocking=True)
    counts_dev = torch.zeros(n_local, dtype=torch.int32, device="cuda")
    scores_dev = torch.zeros(n_local, dtype=torch.float32, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > 126 MB L2

    def step_resident():
        eng.score_lcp_device(0, T_dev, counts_dev, scores_dev, mode)
        return eng.topk_end(eng.topk_begin(0, TOPK, index_base))

    # ---- warm-up (+ lead-in for the nvidia-smi sampler: ~0.3 s under this benchmark's load before the timed region)
    sampler = ClockSampler(gpu_uuid(torch, local_rank)) if rank == 0 else None
    if sampler:
        sampler.wait_started()
    eng.score_lcp_device(0, T_dev, counts_dev, scores_dev, mode)          # first call (weighted: builds the K1c lists)
    est_ms = timed_ms(torch, stream, lambda: eng.score_lcp_device(0, T_dev, counts_dev, scores_dev, mode), reps=1)
    lead_in = int(D.reduce(min(300, max(0, 300.0 / max(est_ms, 0.05)))))  # the same count on every rank
    for _ in range(max(args.warmup, 3) + lead_in):
        flush.zero_()
        top = step_resident()
    D.barrier()

    # ---- timed region: K steps, device-timed.  A step = K3 (score) -> K4 (top-k into the exchange slot) on the scoring stream;
    # the step's all-gather + download run on the context's exchange stream under the NEXT step's L2 flush / scoring, the host
    # does not wait between steps.  Device time = sum of the per-step event pairs (the L2 flush between steps is outside the
    # pairs) + the ONE exchange that nothing overlaps, the last step's (a pair around a stream wait on its ticket).
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps + 1)]
    launches0 = eng.launch_count
    wall0 = time.perf_counter()
    tickets = []
    for a, b in ev[:-1]:
        flush.zero_()
        a.record(stream)
        eng.score_lcp_device(0, T_dev, counts_dev, scores_dev, mode)
        tickets.append(eng.topk_begin(0, TOPK, index_base))
        b.record(stream)
        if len(tickets) >= 6:                        # 8 exchange slots: collect the oldest while newer steps are queued
            top = eng.topk_end(tickets.pop(0))
    ev[-1][0].record(stream)
    eng.topk_stream_wait(tickets[-1])
    ev[-1][1].record(stream)
    for t in tickets:
        top = eng.topk_end(t)
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - wall0) * 1e3
    D.barrier()
    launches = eng.launch_count - launches0
    rank_ms = D.gather(sum(a.elapsed_time(b) for a, b in ev))
    total_ms = max(rank_ms)
    exchange_tail_ms = ev[-1][0].elapsed_time(ev[-1][1])
    wall_ms = D.reduce(wall_ms)
    value = n_step_total * args.steps / (total_ms * 1e-3)
    outputs = {}
    if args.dump_outputs:       # the last timed step's counts / scores (later passes reuse the buffers) and its merged top-k
        sfx = f"_rank{rank}" if world > 1 else ""
        per_hyp = hypothesis_arrays(counts_dev.cpu().numpy(), scores_dev.cpu().numpy(), index_base, world)
        outputs = {k + sfx: v for k, v in per_hyp.items()}
        if rank == 0:
            outputs.update(topk_arrays(top))

    # ---- the same K steps back to back WITHOUT the L2 flush, one event pair around all of them incl. the last exchange: what a
    # pipelined caller sees (warm L2; reported next to the headline, not instead of it)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    a.record(stream)
    tickets = []
    for _ in range(args.steps):
        eng.score_lcp_device(0, T_dev, counts_dev, scores_dev, mode)
        tickets.append(eng.topk_begin(0, TOPK, index_base))
        if len(tickets) >= 6:
            eng.topk_end(tickets.pop(0))
    eng.topk_stream_wait(tickets[-1])
    b.record(stream)
    for t in tickets:
        eng.topk_end(t)
    torch.cuda.synchronize()
    noflush_ms = D.reduce(a.elapsed_time(b))

    # ---- the dominant kernel alone (K3), for the roofline
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(min(args.steps, 10))]
    for a, b in kev:
        flush.zero_()
        a.record(stream)
        eng.score_lcp_device(0, T_dev, counts_dev, scores_dev, mode)
        b.record(stream)
    torch.cuda.synchronize()
    kernel_ms = statistics.mean(a.elapsed_time(b) for a, b in kev)

    # ---- end to end through the host-buffer API: pinned host transforms in, counts / scores / merged top-k on the host out, TWO
    # batches in flight (upload of step i+1 under the scoring of step i, downloads of step i under the scoring of step i+1).
    # Wall clock around all K steps; the L2 is flushed by the 256 MiB memset enqueued between steps (its ~45 us ARE inside).
    def e2e_begin(i):
        eng.score_lcp_begin(0, T_host.data_ptr(), n_local, counts_host[i & 1].data_ptr(), scores_host[i & 1].data_ptr(), mode)
        return eng.topk_begin(0, TOPK, index_base)

    def e2e_end(ticket):
        if eng.score_lcp_end():                      # the streamed upload stalled and the batch was re-scored: select again
            eng.topk_end(ticket)
            ticket = eng.topk_begin(0, TOPK, index_base)
        return eng.topk_end(ticket)

    def e2e_loop(k):
        t_prev = e2e_begin(0)
        for i in range(1, k):
            flush.zero_()
            t_next = e2e_begin(i)
            e2e_end(t_prev)
            t_prev = t_next
        return e2e_end(t_prev)

    e2e_loop(3)
    D.barrier()
    t0 = time.perf_counter()
    top_e2e = e2e_loop(args.steps)                   # returns with every step's counts / scores / merged top-k on the host
    torch.cuda.synchronize()
    e2e_s = D.reduce(time.perf_counter() - t0)
    D.barrier()
    e2e_value = n_step_total * args.steps / e2e_s
    clocks = sampler.stop() if sampler else None

    # ---- correctness inside the run: (a) every rank checks a sample of ITS hypotheses against the CPU checker, (b) N > 1: the
    # same list sharded N ways gives the single-GPU top-64
    o, kind = oracle_for(prob)
    n_chk = min(n_local, 256 if cfg["n_model"] <= 4000 else 16) if world > 1 else 0
    mism = 0.0
    if n_chk:
        sel = np.linspace(0, n_local - 1, n_chk).astype(np.int64)
        got = counts_host[(args.steps - 1) & 1].numpy()[sel].astype(np.uint32)
        if mode == "count":
            want = o.verify(T[sel])
            mism = float((got != want).sum())
        else:
            ws, wn = o.weighted_verify(T[sel])
            gs = scores_host[(args.steps - 1) & 1].numpy()[sel]
            mism = float((got != wn.astype(np.uint32)).sum() + (gs != ws).sum())
    mism_total = D.reduce(mism, "sum")
    invariance = sharding_invariance(eng, D, cfg, prob, stream) if world > 1 and not no_comm else None

    if rank == 0:
        b_hyp, kbar, nonempty = algorithmic_bytes_per_hyp(prob, T, cfg["n_model"])
        achieved = b_hyp * n_local / (kernel_ms * 1e-3) / 1e9
        stat = ncu_static(args.config) or {}
        gather = {"l2_resident_64MiB": eng.bench_sector_gather(64 << 20, 512), "hbm_4GiB": eng.bench_sector_gather(4 << 30, 256)}
        moved = stat.get("l2_to_l1_sectors")
        dram = (stat.get("dram_bytes_read", 0) + stat.get("dram_bytes_write", 0)) if stat else None
        roofline = {
            "bound": "l1tex+issue (L2-resident sector gather; tensor cores do not apply, DRAM is at dram_frac of its peak)",
            "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"], "traffic": dram or None,
            "peak_kind": peak_kind, "kernel": f"k3_fine_kernel<smem table, {mode}>", "kernel_ms": kernel_ms,
            "algorithmic_bytes_per_hyp": b_hyp, "kbar_27": kbar, "nonempty_query_fraction": nonempty,
            "algorithmic_frac": achieved / peaks["hbm_gbs"],
            "moved_bytes_frac": (moved * 32 / (kernel_ms * 1e-3) / 1e9 / gather["l2_resident_64MiB"]) if moved else None,
            "dram_frac": (dram / (kernel_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]) if dram else None,
            "sector_gather_peak_gbs": gather, "ncu_static": stat or None,
            "note": "algorithmic = bytes of the canonical 27-cell probe (SURVEY.md 8d) / kernel time / measured HBM copy peak: > 1 because the group "
                    "cull and the tri-state labels answer ~95 % of the queries without touching a scene point; moved = L2->L1 sectors of one "
                    "launch (committed ncu capture) x 32 B / this run's kernel time / the random-sector gather peak measured in this run "
                    "(pgp_bench_sector_gather, L2-resident footprint); dram = DRAM bytes of one launch (same capture) / kernel time / HBM peak"}
        line = {
            "metric": cfg["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": total_ms / args.steps, "ms_per_step_per_rank": [round(x / args.steps, 5) for x in rank_ms], "exchange_tail_ms": exchange_tail_ms,
            "ms_per_step_pipelined_no_l2_flush": noflush_ms / args.steps,
            "wall_ms_per_step_incl_l2_flush_and_host_merge": wall_ms / args.steps, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"name": args.config, "workload": cfg["workload"], "n_model": cfg["n_model"], "n_scene": cfg["n_scene"],
                       "hypotheses_per_gpu": n_local, "hypotheses_per_step": n_step_total, "delta": cfg["delta"],
                       "topk": TOPK, "mode": mode, "grid_dims": grid["dims"], "grid_bytes": grid["bytes"],
                       "l2": "256 MiB device memset between timed steps (outside the timed events; inside the e2e wall clock)",
                       "parallelism": f"hypotheses sharded over {world} GPU(s), scene grid replicated; top-k exchange = ncclAllGather inside libpgp.so on "
                                      "the exchange stream, overlapped with the next step"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n_local * 48 * world, "d2h_bytes_per_step": (n_local * 8 + world * (TOPK + 1) * 64) * world,
                    "ms_per_step": e2e_s / args.steps * 1e3, "batches_in_flight": 2},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "best": {"index": int(top["index"][0]), "count": int(top["count"][0])},
        }
        if world == 1:
            line["secondary"] = secondary_metrics(eng, prob, cfg, T_dev, counts_dev, scores_dev, flush, stream)
            base, _, cpu_counts, sample = cpu_reference_run(prob, T, seconds_per_step=12.0, steps=1, warmup=0)
            line["cpu_baseline"] = base
            if cfg["n_model"] <= 4000:
                line["secondary"].update(cpu_secondary(prob, T))
            if mode == "count":
                got = counts_host[(args.steps - 1) & 1].numpy()[:sample].astype(np.uint32)
                line["parity"] = {"checked": int(sample), "mismatches": int((got != cpu_counts).sum()), "against": kind}
            else:
                ws, wn = o.weighted_verify(T[:2000])
                gs = scores_host[(args.steps - 1) & 1].numpy()[:2000]
                gc = counts_host[(args.steps - 1) & 1].numpy()[:2000].astype(np.uint32)
                line["parity"] = {"checked": 2000, "mismatches": int((gs != ws).sum() + (gc != wn.astype(np.uint32)).sum()), "against": kind + " WeightedVerify"}
        else:
            line["parity"] = {"checked": int(n_chk * world), "mismatches": int(mism_total), "against": kind, "what": f"{n_chk} hypotheses of every rank's shard"}
            line["sharding_invariance"] = invariance
        emit(line)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    eng.close()


def run_pcs(args, D: Dist, local_rank: int):
    """configs[2]: per step, for each of 4 objects: scene grid of the object's segment -> StoCS bases of this rank's base range ->
    PPF-map pairs -> quad join -> transforms (pgp_generate_pcs_range) -> global cap (pgp_comm_sync_generated) -> WeightedVerify
    of the rank's own hypotheses (no transform traffic) -> top-64 (K4 + all-gather + merge).  Models and their PPF maps are
    uploaded once (GlobalCfg::loadObjects, PPE/src/data_layer/GlobalCfg.cpp:30-64)."""
    import torch

    from physimglobalpose_b200 import synth
    from physimglobalpose_b200.engine import HYP_DTYPE, PoseEngine
    from physimglobalpose_b200.sharding import comm_init_from_env, shard_range

    cfg = CONFIGS["c3"]
    rank, world = D.rank, D.world
    eng = PoseEngine(local_rank)
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    comm_init_from_env(eng, rank, world)
    objs = [synth.make_segment_problem(cfg["n_model"], cfg["n_scene"], cfg["delta"], seed=5 + o) for o in range(cfg["objects"])]
    t0 = time.perf_counter()
    eng.set_scene(objs[0].scene_xyz, objs[0].scene_nrm, cfg["delta"])
    for o, seg in enumerate(objs):
        eng.set_model(o, seg.model_xyz, seg.model_nrm)
        eng.build_ppf_map(o)
    eng.synchronize()
    setup_ms = (time.perf_counter() - t0) * 1e3
    B = cfg["n_bases"]
    lo, hi = shard_range(B, rank, world)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    kept = {}                                       # object -> (global index of this rank's first hypothesis, hypotheses it kept)

    def request(o, seed):
        seg = objs[o]
        eng.set_scene(seg.scene_xyz, seg.scene_nrm, cfg["delta"])
        n_gen = eng.generate_pcs_range(o, lo, hi, seed=seed, max_hyp=cfg["n_hyp"], mode=1, n_bases=B)
        base, total = eng.sync_generated(o, cfg["n_hyp"])
        kept[o] = (base, max(0, min(n_gen, total - base)))     # the global cap is filled in rank order
        eng.score_generated(o, "weighted")
        return eng.topk_begin(o, TOPK, base), total

    def step(seed):
        tot, tops = 0, []
        tickets = []
        for o in range(cfg["objects"]):
            t, n = request(o, seed + o)
            tickets.append(t); tot += n
        for t in tickets:
            tops.append(eng.topk_end(t))
        return tot, tops

    sampler = ClockSampler(gpu_uuid(torch, local_rank), period_ms=100) if rank == 0 else None    # (a step is ~100 ms and hundreds of launches)
    if sampler:
        sampler.wait_started()
    for w in range(max(1, min(args.warmup, 2))):
        step(1000 + 10 * w)
    # where a step's time goes: one extra, untimed step with a device synchronisation after every phase
    phase = {}
    for rep in range(2):                            # (the second pass: buffers have their final sizes)
      phase = {"scene_grid": 0.0, "generate": 0.0, "cap_exchange": 0.0, "score_weighted": 0.0, "topk": 0.0}
      for o in range(cfg["objects"]):
          seg = objs[o]
          def lap(key, fn):
              torch.cuda.synchronize(); t0 = time.perf_counter(); r = fn(); torch.cuda.synchronize(); phase[key] += (time.perf_counter() - t0) * 1e3; return r
          lap("scene_grid", lambda: eng.set_scene(seg.scene_xyz, seg.scene_nrm, cfg["delta"]))
          lap("generate", lambda: eng.generate_pcs_range(o, lo, hi, seed=7 + o, max_hyp=cfg["n_hyp"], mode=1, n_bases=B))
          base_o, _ = lap("cap_exchange", lambda: eng.sync_generated(o, cfg["n_hyp"]))
          lap("score_weighted", lambda: eng.score_generated(o, "weighted"))
          lap("topk", lambda: eng.topk_end(eng.topk_begin(o, TOPK, base_o)))
    D.barrier()
    launches0 = eng.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    n_total, tops = 0, None
    wall0 = time.perf_counter()
    for i, (a, b) in enumerate(ev):
        flush.zero_()
        a.record(stream)
        n, tops = step(7)                       # the same seed every step: the same request (and the N-invariance check below)
        b.record(stream)
        n_total += n
    torch.cuda.synchronize()
    wall_s = D.reduce(time.perf_counter() - wall0)
    D.barrier()
    total_ms = D.reduce(sum(a.elapsed_time(b) for a, b in ev))
    launches = eng.launch_count - launches0
    clocks = sampler.stop() if sampler else None
    if rank == 0:
        digest = [{"object": o, "best_index": int(t["index"][0]), "best_score": float(t["score"][0]), "top64_crc": int(np.bitwise_xor.reduce(np.frombuffer(t.tobytes(), np.uint32)))}
                  for o, t in enumerate(tops)]
        cpu = cpu_pcs_baseline_subprocess() if world == 1 else None       # the CPU leg: rank 0 at N = 1 only
        line = {"metric": cfg["metric"], "value": n_total / (total_ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(1, min(args.warmup, 2)),
                "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"name": "c3", "workload": cfg["workload"], "objects": cfg["objects"], "n_bases_per_object": B, "hypotheses_per_step": n_total // args.steps,
                           "parallelism": f"bases sharded over {world} GPU(s): each GPU generates and scores its own hypotheses; scene grid, models and PPF maps replicated",
                           "one_time_setup_ms": setup_ms, "phase_ms_per_step_rank0": {k: round(v, 3) for k, v in phase.items()},
                           "l2": "256 MiB memset between steps (outside the events)"},
                "e2e": {"value": n_total / wall_s, "unit": UNIT, "h2d_bytes_per_step": int(sum(len(s.scene_xyz) * 24 for s in objs)) * world,
                        "d2h_bytes_per_step": cfg["objects"] * world * world * (TOPK + 1) * 64,
                        "what": "wall clock around the same steps: segment clouds in from host memory, merged top-64 per object out (the hypotheses never leave the GPU that generated them)"},
                "gpu_launches": launches, "clocks": clocks,
                "roofline": {"bound": "issue/latency (generation: 30+ dependent launches per object with host-read totals; scoring: as c2w)", "achieved": None, "peak": None,
                             "unit": "GB/s", "frac": None, "traffic": None},
                "top64_digest": digest,
                "note": "top64_digest must be identical for every --gpus N (same seed -> same bases -> same hypotheses whichever GPU generates them)"}
        line["cpu_baseline"] = cpu
        emit(line)
    if args.dump_outputs:       # the last timed step: per object, the merged top-64 and a sample of this rank's generated hypotheses
        top = np.zeros((cfg["objects"], TOPK), HYP_DTYPE)
        top["index"] = -1                           # a list shorter than TOPK is padded like the engine pads it
        for o, t in enumerate(tops):
            top[o, :len(t)] = t
        sfx = f"_rank{rank}" if world > 1 else ""
        outputs = dict(topk_arrays(top), hypotheses_generated=np.array([n], np.float64)) if rank == 0 else {}
        for o in range(cfg["objects"]):
            base, n_kept = kept[o]
            T_gen, c_gen, s_gen = (a[:n_kept] for a in eng.get_generated(o))
            per_hyp = hypothesis_arrays(c_gen, s_gen, base, world * cfg["objects"] * 2)      # / 2: T too, 68 bytes a hypothesis
            per_hyp["generated_T"] = T_gen[(per_hyp["hypothesis_index"] - base).astype(np.int64)].astype(np.float32)
            outputs.update({f"object{o}_{k}{sfx}": v for k, v in per_hyp.items()})
        dump_outputs(args.dump_outputs, outputs)
    eng.close()


def cpu_pcs_baseline_subprocess() -> dict:
    """The CPU arm of configs[2] in its own process (`bench.py --impl reference --config c3`): the reference's generator has
    undefined behaviour of its own (SURVEY.md 3.2: out-of-bounds best index) and must not be able to take this line down."""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--config", "c3", "--steps", "2", "--warmup", "0"],
                             capture_output=True, text=True, timeout=600, env=dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0"))
        return json.loads(out.stdout.strip().splitlines()[-1])["cpu_baseline"]
    except Exception as e:
        return {"error": repr(e)[:200]}


_RESULT_FD = None


def _claim_stdout():
    """stdout carries exactly ONE JSON line.  Libraries (the NCCL version banner under NCCL_DEBUG=VERSION, torchrun's OMP notice)
    write to file descriptor 1 directly, so fd 1 is pointed at stderr for the whole run and the result goes to a saved duplicate."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def topk_arrays(top: np.ndarray) -> dict:
    """Merged top-k records (engine.HYP_DTYPE, any leading shape) as the arrays a caller reads from them."""
    return {"topk_index": top["index"].astype(np.float64), "topk_count": top["count"].astype(np.float64),
            "topk_score": top["score"].astype(np.float32), "topk_T": top["T"].reshape(*top.shape, 3, 4).astype(np.float32)}


def hypothesis_arrays(counts: np.ndarray, scores: np.ndarray, index_base: int, world: int) -> dict:
    """Per-hypothesis counts and scores of a rank's batch with their global hypothesis indices; a batch larger than this rank's
    share of DUMP_MAX_HYP is reduced to a sample drawn with a fixed seed, so two runs dump the same hypotheses."""
    n, cap = len(counts), DUMP_MAX_HYP // world
    sel = np.arange(n) if n <= cap else np.sort(np.random.default_rng(0).choice(n, cap, replace=False))
    return {"hypothesis_index": (sel + index_base).astype(np.float64), "counts": counts[sel].astype(np.float64),
            "scores": scores[sel].astype(np.float32)}


def dump_outputs(out_dir: str, arrays: dict):
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float32 / float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {"c5": 5, "c3": 3}.get(args.config, 20)
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the CUDA path (--impl ours)")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    D = Dist(rank, local_rank, world)
    if args.config == "c3":
        run_pcs(args, D, local_rank)
    else:
        run_scoring(args, D, local_rank)
    D.close()


if __name__ == "__main__":
    main()
