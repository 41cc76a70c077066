"""The C++ drop-in (physimglobalpose_b200/adaptor/libsuper4pcs.so): exports the reference's mangled
symbol, and -- on the GPU -- fills bestHypothesis / hypothesisSet / registered_points from the same
files the reference's caller writes (PCL-style ASCII PLY with 10 vertex properties, 16-bit prior PNG)."""
import json
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from physimglobalpose_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AD = os.path.join(ROOT, "physimglobalpose_b200", "adaptor")
SYMBOL_PREFIX = "_Z30getProbableTransformsSuper4PCSNSt7__cxx1112basic_string"


def _build():
    if not os.path.exists(os.path.join(ROOT, "physimglobalpose_b200", "libpgp.so")):
        import __graft_entry__ as g
        g.build()
    subprocess.check_call(["make", "-s", "-C", AD])


def _exported():
    out = subprocess.check_output(["nm", "-D", "--defined-only", os.path.join(AD, "libsuper4pcs.so")], text=True)
    return [l.split()[-1] for l in out.splitlines() if "getProbableTransformsSuper4PCS" in l]


def test_dropin_exports_the_reference_symbol():
    _build()
    syms = _exported()
    assert len(syms) == 1 and syms[0].startswith(SYMBOL_PREFIX)
    # Isometry3d and Matrix3f appear with Eigen's own template arguments
    assert "N5Eigen9TransformIdLi3ELi1ELi0EEE" in syms[0] and "6MatrixIfLi3ELi3ELi0ELi3ELi3EEE" in syms[0]


def test_symbol_equals_the_one_real_eigen_produces(tmp_path):
    """tests/golden/dropin_symbol.txt holds the mangled name g++ gives the reference-side declaration (ObjectPoseCandidateSet.cpp:5-9)
    compiled against the reference's own vendored Eigen headers; the drop-in must export exactly that name, and the Eigen stand-ins
    it is built with must have the layouts real Eigen gives those types (Isometry3d: 128 bytes 16-aligned and Matrix3f: 36 bytes,
    asserted in eigen_abi.h itself; pair<Isometry3d, float>: 144 bytes, asserted here)."""
    _build()
    with open(os.path.join(ROOT, "tests", "golden", "dropin_symbol.txt")) as f:
        real = f.read().split()
    assert real == _exported()
    src = tmp_path / "layout.cc"
    src.write_text('''#include <utility>
#include "eigen_abi.h"
static_assert(sizeof(std::pair<Eigen::Isometry3d, float>) == 144, "pair layout");
''')
    subprocess.check_call(["g++", "-std=c++17", "-fsyntax-only", "-I" + AD, str(src)])


def write_pcl_ply(path, xyz, nrm):
    """ASCII PLY as pcl::io::savePLYFile writes a PointXYZRGBNormal cloud (10 vertex properties + camera element)."""
    with open(path, "w") as f:
        f.write("ply\nformat ascii 1.0\ncomment PCL generated\nelement vertex %d\n" % len(xyz))
        f.write("property float x\nproperty float y\nproperty float z\nproperty uchar red\nproperty uchar green\nproperty uchar blue\n")
        f.write("property float nx\nproperty float ny\nproperty float nz\nproperty float curvature\n")
        f.write("element camera 1\nproperty float view_px\nproperty float view_py\nend_header\n")
        for p, n in zip(xyz, nrm):
            f.write("%.9g %.9g %.9g 128 128 128 %.9g %.9g %.9g 0\n" % (p[0], p[1], p[2], n[0], n[1], n[2]))
        f.write("0 0\n")


def write_png16(path, img):
    h, w = img.shape
    raw = b"".join(b"\x00" + img[r].astype(">u2").tobytes() for r in range(h))

    def chunk(t, d):
        return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xFFFFFFFF)

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 16, 0, 0, 0, 0)) + chunk(b"IDAT", zlib.compress(raw)) + chunk(b"IEND", b""))


@pytest.mark.gpu
def test_dropin_end_to_end(tmp_path, engine):
    _build()
    prob = synth.make_segment_problem(800, 1500, 0.005, seed=13)
    seg, val, search = (str(tmp_path / n) for n in ("pclSegment_obj.ply", "pclModel_obj.ply", "pclModelSampled_obj.ply"))
    write_pcl_ply(seg, prob.scene_xyz, prob.scene_nrm)
    write_pcl_ply(val, prob.model_xyz, prob.model_nrm)
    write_pcl_ply(search, prob.model_xyz, prob.model_nrm)
    png = str(tmp_path / "obj.png")
    write_png16(png, np.full((480, 640), 10000, np.uint16))                # GT mask: prior 1.0 everywhere
    env = dict(os.environ, PGP_SEED="3")
    out = subprocess.check_output([os.path.join(AD, "dropin_driver"), seg, val, search, png, "600", "600", "320", "240"], env=env, text=True)
    res = json.loads(out.strip().splitlines()[-1])
    assert res["n_hypotheses"] >= 1 and res["best_score"] > 0.3
    assert res["scores"] == sorted(res["scores"]) and abs(res["scores"][-1] - res["best_score"]) < 1e-7
    assert res["n_registered"] == round(res["best_score"] * len(prob.model_xyz))      # binary priors: score * |Qval| = gated matches
    pose = np.array(res["best_pose"]).reshape(4, 4)
    errs = []
    for flip in (np.eye(3), np.diag([-1.0, -1, 1]), np.diag([-1.0, 1, -1]), np.diag([1.0, -1, -1])):
        gt = prob.gt_pose.copy(); gt[:3, :3] = gt[:3, :3] @ flip
        errs.append(synth.pose_error(pose, gt))
    dt, ang = min(errs, key=lambda e: e[0] + e[1])
    assert dt < 0.01 and ang < 0.1, (dt, ang)
    # the same request through the Python host mirror gives the same answer (the PLY text round-trips %.9g exactly)
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, 0.005)
    engine.set_model(0, prob.model_xyz, prob.model_nrm)
    engine.generate_pcs(0, seed=3, max_hyp=10000)
    engine.score_generated(0, "weighted")
    chain = engine.improving_chain(0)
    assert len(chain) == res["n_hypotheses"]
    assert np.array_equal(chain["score"], np.array(res["scores"], np.float32))
    assert np.allclose(engine.centred_to_pose(0, chain["T"][-1])[0], pose, atol=1e-12)


@pytest.mark.gpu
def test_dropin_stocs_with_ppf_map_file(tmp_path, engine):
    """The shipped configuration: the node hands over the model's PPFMap (loaded from PPFMap.txt) and the engine runs operMode 1.
    The map file is produced by the device-side builder (the reference does not ship its generator) in the reference's text
    format, read back by the driver the way Objects::readPPFMap does, and the answer must equal the host mirror's."""
    _build()
    prob = synth.make_segment_problem(500, 900, 0.005, seed=17)
    seg, val, search = (str(tmp_path / n) for n in ("pclSegment_obj.ply", "pclModel_obj.ply", "pclModelSampled_obj.ply"))
    write_pcl_ply(seg, prob.scene_xyz, prob.scene_nrm)
    write_pcl_ply(val, prob.model_xyz, prob.model_nrm)
    write_pcl_ply(search, prob.model_xyz, prob.model_nrm)
    png = str(tmp_path / "obj.png")
    write_png16(png, np.full((480, 640), 10000, np.uint16))
    engine.set_scene(prob.scene_xyz, prob.scene_nrm, 0.005)
    engine.set_model(0, prob.model_xyz, prob.model_nrm)
    engine.build_ppf_map(0)
    keys, offs, pairs = engine.get_ppf_map(0)
    ppf_txt = str(tmp_path / "PPFMap.txt")
    with open(ppf_txt, "w") as f:
        for k in range(len(keys)):
            rows = pairs[offs[k]:offs[k + 1]]
            f.write("%d %d %d %d %d\n" % (*keys[k], len(rows)))
            f.write(" ".join("%d %d" % (a, b) for a, b in rows) + "\n")
    env = dict(os.environ, PGP_SEED="5")
    out = subprocess.check_output([os.path.join(AD, "dropin_driver"), seg, val, search, png, "600", "600", "320", "240", ppf_txt], env=env, text=True)
    res = json.loads(out.strip().splitlines()[-1])
    assert res["n_hypotheses"] >= 1 and res["best_score"] > 0.1       # StoCS bases are not forced to be wide: coarser poses than mode 0
    engine.generate_pcs(0, seed=5, max_hyp=10000, mode=1)
    engine.score_generated(0, "weighted")
    chain = engine.improving_chain(0)
    assert len(chain) == res["n_hypotheses"]
    assert np.array_equal(chain["score"], np.array(res["scores"], np.float32))
    pose = np.array(res["best_pose"]).reshape(4, 4)
    assert np.allclose(engine.centred_to_pose(0, chain["T"][-1])[0], pose, atol=1e-12)
    # No pose-accuracy assertion here: StoCS bases are not forced to be wide and a box has only three normal directions, so its PPF
    # keys barely discriminate -- with 100 bases the sampler (bit-equal to the reference's, tests/test_gpu_golden.py) settles on a
    # 90-degree-rotated fit of this synthetic box about as often as on the true pose.  That is the algorithm, not the port.


@pytest.mark.gpu
def test_dropin_is_a_service_component(tmp_path):
    """A long-lived node calls the entry point once per object per request: the second and third call of the same process must
    return exactly what the first did (the caller's hypothesisSet is cleared, not appended to), hit the per-object model cache
    (no PLY parse / upload of the model: faster), and append one line per returned pose to <scene>/debug_super4PCS/<obj>_time.txt
    like Perform_N_steps does (match4pcsBase.cc:1909-1913).  With >= 2 GPUs, PGP_DEVICES shards the bases and the answer is the same."""
    import torch
    _build()
    prob = synth.make_segment_problem(800, 1500, 0.005, seed=13)
    seg, val, search = (str(tmp_path / n) for n in ("pclSegment_obj.ply", "pclModel_obj.ply", "pclModelSampled_obj.ply"))
    write_pcl_ply(seg, prob.scene_xyz, prob.scene_nrm)
    write_pcl_ply(val, prob.model_xyz, prob.model_nrm)
    write_pcl_ply(search, prob.model_xyz, prob.model_nrm)
    png = str(tmp_path / "obj.png")
    write_png16(png, np.full((480, 640), 10000, np.uint16))
    scene = str(tmp_path) + "/"
    os.makedirs(os.path.join(scene, "debug_super4PCS"))
    args = [os.path.join(AD, "dropin_driver"), seg, val, search, png, "600", "600", "320", "240"]

    def run(env_extra, repeat):
        env = dict(os.environ, PGP_SEED="3", PGP_DRIVER_REPEAT=str(repeat), PGP_DRIVER_SCENE=scene, **env_extra)
        return json.loads(subprocess.check_output(args, env=env, text=True).strip().splitlines()[-1])

    once = run({}, 1)
    log = os.path.join(scene, "debug_super4PCS", "obj_time.txt")
    assert len(open(log).read().split()) == once["n_hypotheses"]
    thrice = run({}, 3)
    for k in ("best_score", "n_hypotheses", "n_registered", "best_pose", "scores"):
        assert thrice[k] == once[k], k                                   # not 3x the chain: the callee clears the caller's vector
    assert len(open(log).read().split()) == 4 * once["n_hypotheses"]     # append mode, one line per pose and request
    assert min(thrice["call_ms"][1:]) < thrice["call_ms"][0]             # model parse + upload happen once per object
    if torch.cuda.device_count() >= 2:
        multi = run({"PGP_DEVICES": "0,1"}, 2)
        for k in ("best_score", "n_hypotheses", "n_registered", "best_pose", "scores"):
            assert multi[k] == once[k], k
