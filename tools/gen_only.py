"""PCS generation only (for ncu launch lists and generator timings):
    python tools/gen_only.py mode n_bases [scene_points (2000)] [max_quads_per_base (100; 0 = every quad)]"""
import sys, time
sys.path.insert(0, '.')
import torch
from physimglobalpose_b200 import synth
from physimglobalpose_b200.engine import PoseEngine
mode, nb = int(sys.argv[1]), int(sys.argv[2])
n_scene = int(sys.argv[3]) if len(sys.argv) > 3 else 2000
cap = int(sys.argv[4]) if len(sys.argv) > 4 else 100
max_hyp = nb * cap if cap > 0 else 1 << 22
prob = synth.make_segment_problem(2000, n_scene, 0.005, seed=100)
e = PoseEngine(0)
e.set_scene(prob.scene_xyz, prob.scene_nrm, prob.delta); e.set_model(0, prob.model_xyz, prob.model_nrm)
if mode == 1: e.build_ppf_map(0)
e.generate_pcs(0, seed=1, max_hyp=1000, n_bases=8, mode=mode)
for rep in range(3):        # the first call grows the buffers
    torch.cuda.synchronize(); t0 = time.perf_counter(); l0 = e.launch_count
    n = e.generate_pcs(0, seed=5, max_hyp=max_hyp, n_bases=nb, max_quads_per_base=cap, mode=mode)
    torch.cuda.synchronize(); dt = time.perf_counter() - t0
    print('mode', mode, 'bases', nb, 'scene', n_scene, 'cap', cap, 'hypotheses', n, 'ms', round(dt * 1e3, 3), 'hyp/s', round(n / dt),
          'launches', e.launch_count - l0)
