"""The literal drop-in: the reference renderer's own binary with `B200PathTraceIntegrator` linked in
(oracle/_ref/dropin/tungsten_b200, built by `make -C oracle/ref dropin` where the reference's sources are at hand) renders
scenes whose integrator type is "b200_path_tracer" on the GPU; its PFM output is compared with the framebuffers the
reference's CPU integrator produced for the same scenes (tests/golden/*/ref_pathseed.pfm)."""
import json
import os
import subprocess

import numpy as np
import pytest

from tungsten_b200 import scene

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EXE = os.path.join(ROOT, "oracle", "_ref", "dropin", "tungsten_b200")
G = os.path.join(ROOT, "tests", "golden")


@pytest.mark.skipif(not os.path.exists(EXE), reason="drop-in binary not built (needs the reference's sources at build time)")
@pytest.mark.parametrize("name", ["cornell", "materials", "coat_env", "hair", "curves_plastic", "hair_sky", "dirac", "many_lights", "cube_city", "coats"])
def test_reference_binary_with_b200_integrator(name, tmp_path):
    src = os.path.join(G, name)
    for f in os.listdir(src):
        if not f.endswith(".pfm"):
            os.symlink(os.path.join(src, f), tmp_path/f)
    js = json.load(open(os.path.join(src, "scene.json")))
    js["integrator"]["type"] = "b200_path_tracer"
    js["renderer"]["spp_step"] = 3                     # exercises spp stepping: 3 + 3 + 2
    json.dump(js, open(tmp_path/"b200.json", "w"))
    out = subprocess.run([EXE, "-t", "2", "-d", str(tmp_path/"out"), str(tmp_path/"b200.json")], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True)
    assert out.returncode == 0, out.stdout
    assert "Completed 8/8 spp" in out.stdout, out.stdout
    got = scene.load_pfm(str(tmp_path/"out"/"out.pfm"))
    want = scene.load_pfm(os.path.join(src, "ref_pathseed.pfm"))
    d = np.abs(got - want).max(axis=2)
    close = float((d <= 1e-5*(1.0 + np.abs(want).max(axis=2))).mean())
    print(name, "exact %.4f close %.4f" % (float((d == 0).mean()), close))
    assert close >= (0.97 if name in ("hair", "curves_plastic", "hair_sky") else 0.985)     # curve scenes: see tests/test_gpu_parity.py::test_curves_and_hair


def _run_dropin(tmp_path, js, name="b200.json", expect=None):
    json.dump(js, open(tmp_path/name, "w"))
    out = subprocess.run([EXE, "-t", "2", "-d", str(tmp_path/"out"), str(tmp_path/name)], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True)
    assert out.returncode == 0, out.stdout
    if expect:
        assert expect in out.stdout, out.stdout
    return scene.load_pfm(str(tmp_path/"out"/"out.pfm")), out.stdout


@pytest.mark.skipif(not os.path.exists(EXE), reason="drop-in binary not built (needs the reference's sources at build time)")
def test_dropin_adaptive_sampling_as_shipped_scenes_use_it(tmp_path):
    """renderer.adaptive_sampling = true (the as-shipped setting of data/materialtest and the example scenes) through the
    literal drop-in: generateWork + per-block records in the adapter, tgb200_render_adaptive underneath, vs the reference
    binary's own adaptive render of the same scene (tests/golden/cornell_adaptive)."""
    src = os.path.join(G, "cornell_adaptive")
    js = json.load(open(os.path.join(src, "scene.json")))
    assert js["renderer"]["adaptive_sampling"] is True
    js["integrator"]["type"] = "b200_path_tracer"
    got, log = _run_dropin(tmp_path, js, expect="Completed 48/48 spp")
    want = scene.load_pfm(os.path.join(src, "ref_pathseed.pfm"))
    d = np.abs(got - want).max(axis=2)
    close = float((d <= 1e-5*(1.0 + np.abs(want).max(axis=2))).mean())
    print("adaptive drop-in: exact %.4f close %.4f" % (float((d == 0).mean()), close))
    assert close >= 0.97


@pytest.mark.skipif(not os.path.exists(EXE), reason="drop-in binary not built (needs the reference's sources at build time)")
def test_dropin_writes_resume_state(tmp_path):
    """Integrator::saveRenderResumeData (Integrator.cpp:108-129) with the adapter's saveState: the resume file the drop-in
    writes after 16 spp holds the colour buffer and, behind it, the 4x4-block SampleRecords + the integrator's sampler state --
    the same records the Integrator twin holds after the same step (same library, same arithmetic: bit for bit).
    (Reading the file back is the reference's job and does not work in this build of the reference, with or without this
    adapter: Integrator::resumeRender keeps a `const Path &` into a temporary RendererSettings (Integrator.cpp:133) and opens a
    garbage path -- the stock binary prints "Resume unsuccessful" for its own resume files too.  The continuation itself is
    covered by tests/test_gpu_parity.py::test_resume_state_round_trip.)"""
    import struct
    from tungsten_b200 import integrator, abi
    src = os.path.join(G, "cornell_adaptive")
    js = json.load(open(os.path.join(src, "scene.json")))
    js["integrator"]["type"] = "b200_path_tracer"
    js["renderer"].update(enable_resume_render=True, spp=16)
    _run_dropin(tmp_path, js, name="scene.json", expect="Completed 16/16 spp")
    blob = open(tmp_path/"out"/"TungstenRenderState.dat", "rb").read()
    z = blob.index(b"\0")
    head = json.loads(blob[:z].decode())
    assert head["current_spp"] == 16 and head["adaptive_sampling"] is True
    w, h = js["camera"]["resolution"]
    n = w*h; nb = ((w + 3)//4)*((h + 3)//4)
    off = z + 1 + 8
    mean = np.frombuffer(blob, dtype=np.float32, count=3*n, offset=off).reshape(h, w, 3); off += 12*n
    count = np.frombuffer(blob, dtype=np.uint32, count=n, offset=off); off += 4*n
    assert (count == 16).all()
    recs = np.frombuffer(blob, dtype=np.uint8, count=24*nb, offset=off); off += 24*nb
    sampler_state = struct.unpack_from("<Q", blob, off)[0]; off += 8
    assert off == len(blob)
    fs = scene.load_scene(os.path.join(src, "scene.json"))
    it = integrator.B200PathTraceIntegrator(); it.prepareForRender(fs, 0xBA5EBA11)
    it.startRender(); it.waitForCompletion()
    st = it.save_state(); it.teardownAfterRender()
    assert st["current_spp"] == 16
    assert np.array_equal(mean, st["mean"])
    assert bytes(recs) == st["records"]
    assert sampler_state == st["sampler_state"]


@pytest.mark.skipif(not os.path.exists(EXE), reason="drop-in binary not built (needs the reference's sources at build time)")
def test_dropin_on_two_gpus_equals_one_gpu(tmp_path):
    """"devices": [0, 1] in the integrator block -> tgb_settings::devices: the library replicates the scene, deals the tiles
    in Morton order, gathers the shares on devices[0] over NVLink.  Under the per-path reseed contract the image does not
    depend on who rendered which tile: bit for bit the one-GPU image."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    js = json.load(open(os.path.join(G, "materials", "scene.json")))
    for f in os.listdir(os.path.join(G, "materials")):
        if not f.endswith(".pfm") and f != "scene.json":
            os.symlink(os.path.join(G, "materials", f), tmp_path/f)
    js["integrator"]["type"] = "b200_path_tracer"
    one, _ = _run_dropin(tmp_path, js, name="one.json")
    js["integrator"]["devices"] = [0, 1]
    two, _ = _run_dropin(tmp_path, js, name="two.json")
    assert np.array_equal(one, two)
