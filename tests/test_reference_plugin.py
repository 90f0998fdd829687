"""End to end through the two command-line front-ends, on the GPU (-m gpu):

  * the UNMODIFIED reference CLI (oracle/_ref/bin/luisa-render-cli, built by oracle/ref from LuisaRender's sources) with THIS
    repository's integrator plugin - `integrator : B200Path`, integration/b200_path.cpp, loaded through the reference's own
    plugin mechanism (src/base/scene.cpp:64-75, LUISA_RENDER_MAKE_SCENE_NODE_PLUGIN): the reference parses the scene, builds
    its scene graph and pipeline, calls Integrator::Instance::render - which runs libb200pt.so on the GPU - and writes the
    EXR with its own save_image.  The EXR is compared with the committed render of the same scene by the reference's own
    WavePath integrator (tests/golden/ref_renders.npz);
  * this repository's luisa-render-cli -b cuda (csrc/host/cli.cpp, the reference's flags): scene file in, EXR out, compared
    with the same fixture; a -D macro on the command line reaches the scene.

The first needs the reference built into oracle/_ref/ (oracle/ref/README.md) and is skipped without it.
"""
from __future__ import annotations

import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))
sys.path.insert(0, str(REPO / "tools"))

import gen_ref_renders as G  # noqa: E402
from luisarender_b200 import _ffi as F  # noqa: E402

pytestmark = pytest.mark.gpu
GOLDEN = REPO / "tests" / "golden" / "ref_renders.npz"
PLUGIN = REPO / "oracle" / "_ref" / "bin" / "libluisa-render-integrator-b200path.so"


def _check(got, want, name):
    got, want = got[..., :3], want[..., :3]
    rel_l2 = float(np.linalg.norm(got - want) / np.linalg.norm(want))
    off = (np.abs(got - want) > 1e-4 * np.maximum(np.abs(want), 1.0)).any(axis=-1)
    assert rel_l2 <= 1e-3, f"{name}: rel-L2 {rel_l2}"
    assert off.mean() <= 0.005, f"{name}: {off.mean():.4f} of the pixels off"


@pytest.mark.parametrize("name", ["cornell_wavepath", "spheres_disney", "flatten_stress"])
def test_reference_cli_with_b200path_plugin(tmp_path, name):
    if not (G.CLI.exists() and PLUGIN.exists()):
        pytest.skip("oracle/_ref (the reference front-end + this repository's plugin for it) is not built")
    golden = np.load(GOLDEN)
    source = bytes(golden[f"{name}/scene"]).decode()
    assert source.count("integrator : WavePath") == 1
    image = G.render_with_reference(source.replace("integrator : WavePath", "integrator : B200Path"), tmp_path, name)
    _check(image, golden[f"{name}/image"], name)


def test_own_cli_renders_a_scene_file_to_exr(tmp_path):
    cli = F.LIB_DIR / "luisa-render-cli"
    golden = np.load(GOLDEN)
    source = bytes(golden["cornell_wavepath/scene"]).decode()
    # the sample count through a command-line macro (src/apps/cli.cpp:105-152): the scene says `spp { #SPP }`
    import re

    spp = re.search(r"spp\s*\{\s*(\d+)\s*\}", source).group(1)
    (tmp_path / "scene.luisa").write_text(re.sub(r"spp\s*\{\s*\d+\s*\}", "spp { #SPP }", source, count=1))
    out_name = re.search(r'Camera\b.*?\bfile\s*\{\s*"([^"]+)"\s*\}', source, re.S).group(1)
    r = subprocess.run([str(cli), "-b", "cuda", "-d", "0", "-D", f"SPP={spp}", "scene.luisa"], cwd=tmp_path, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "Rendering finished in" in r.stdout + r.stderr
    _check(G.read_image(tmp_path / out_name), golden["cornell_wavepath/image"], "own cli")
    # a backend this build does not have is an error, not a fallback
    r = subprocess.run([str(cli), "-b", "cpu", "scene.luisa"], cwd=tmp_path, capture_output=True, text=True, timeout=60)
    assert r.returncode != 0
