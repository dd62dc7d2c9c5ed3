"""Product vs the reference's own CUDA code, both run on the B200 on the same
inputs (BASELINE.json: "primary-ray hit primitive IDs bit-exact, hit distance t
within 1e-5 relative").  The reference runs through oracle/_ref/ref_harness
(its unmodified Bvh::traverse); skipped when that binary was not built."""
import json
import os
import subprocess

import numpy as np
import pytest

from rtcuda_b200 import capi
from conftest import random_rays

pytestmark = pytest.mark.gpu


def harness_path():
    from oracle import binding
    return binding.REF_HARNESS


def run_harness(scene_file, *cmd):
    out = subprocess.run([harness_path(), scene_file] + [str(c) for c in cmd], capture_output=True, text=True, timeout=1200)
    assert out.returncode == 0, out.stderr[-2000:]
    return [json.loads(l[5:]) for l in out.stdout.splitlines() if l.startswith("JSON ")]


@pytest.fixture(scope="module")
def setup(gpu, bunny, tmp_path_factory):
    if not os.path.exists(harness_path()):
        pytest.skip("oracle/_ref/ref_harness not built (needs the original rtcuda sources at build time, oracle/Makefile REF)")
    td = tmp_path_factory.mktemp("ref")
    hs = gpu.host_scene(capi.RTB_SCENE_S1, *bunny)
    sf = str(td / "s1.rtbs")
    hs.save(sf)
    sc = gpu.context(0).scene(hs.desc)
    return gpu, hs, sc, sf, td


def compare(hits, ref):
    diff = np.nonzero(hits["prim"] != ref["prim"])[0]
    # a differing id is tolerated only as an exact tie: both report the same t bits
    ties = diff[hits["t"][diff].view(np.uint32) == ref["t"][diff].view(np.uint32)]
    same = hits["prim"] == ref["prim"]
    rel = np.abs(hits["t"][same] - ref["t"][same]) / np.maximum(np.abs(ref["t"][same]), 1e-30)
    return len(diff), len(ties), float(rel.max()) if same.any() else 0.0, bool((hits["t"][same].view(np.uint32) == ref["t"][same].view(np.uint32)).all())


@pytest.mark.parametrize("w,h", [(600, 600), (1920, 1080)])
def test_primary_hit_ids_match_the_reference(setup, w, h):
    L, hs, sc, sf, td = setup
    rays = L.primary_rays(hs.camera(w / h), w, h)
    rf, hf = str(td / "rays.bin"), str(td / "hits.bin")
    rays.tofile(rf)
    run_harness(sf, "trace", rf, hf)
    ref = np.fromfile(hf, dtype=capi.HIT_DTYPE)
    for entry, hits in (("per-ray kernel", sc.trace_closest(rays)), ("render path's persistent kernel", sc.trace_wavefront(rays)[0])):
        ndiff, nties, max_rel, bitexact = compare(hits, ref)
        print(f"{w}x{h} {entry}: {ndiff} id differences ({nties} exact-t ties), max rel t err {max_rel:.2e}, t bit-exact {bitexact}")
        assert ndiff == nties, "a hit id differs from the reference without being an exact tie in t"
        assert ndiff <= 1e-5 * len(rays)
        assert max_rel <= 1e-5


def test_incoherent_rays_match_the_reference(setup):
    L, hs, sc, sf, td = setup
    rays = random_rays(1000000, seed=99)
    rf, hf = str(td / "rays.bin"), str(td / "hits.bin")
    rays.tofile(rf)
    run_harness(sf, "trace", rf, hf)
    ref = np.fromfile(hf, dtype=capi.HIT_DTYPE)
    for entry, hits in (("per-ray kernel", sc.trace_closest(rays)), ("render path's persistent kernel", sc.trace_wavefront(rays)[0])):
        ndiff, nties, max_rel, bitexact = compare(hits, ref)
        print(f"random, {entry}: {ndiff} id differences ({nties} ties), max rel t err {max_rel:.2e}, bit-exact {bitexact}")
        assert ndiff == nties and ndiff <= 1e-5 * len(rays) and max_rel <= 1e-5
