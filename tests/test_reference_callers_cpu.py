"""Row a1 / b of SURVEY.md §8: the reference's OWN callers, unmodified, on the drop-in classes.

What those callers compute (the unmodified ``release_server.GenerationSession`` and
``CausalInferencePipeline.inference`` on the drop-ins) is stored in tests/golden/reference_callers_small.npz by
tests/golden/make_reference_callers_golden.py, which needs the reference checkout.  Each case runs
tests/run_reference_callers.py in a subprocess (the kernels are swapped for the CPU stand-ins process-wide): the
harness/ stand-in that bench.py, smoke() and the GPU tests drive must make the same calls and produce the same
outputs."""
import json
import subprocess
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent


def run(*args):
    r = subprocess.run([sys.executable, str(ROOT / "tests" / "run_reference_callers.py"), *args],
                       capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("mode", ["keep", "reencode"])
def test_unmodified_generation_session_on_the_dropins(mode):
    """release_server.GenerationSession generates 4 blocks on the drop-ins (window slides at block 2; 'reencode' =
    the default first-frame re-encode through VAEEncoderWrapper): harness/server_loop.py makes the same transformer /
    VAE calls and reproduces its latents and pixels, and stays within bf16 tolerance of the reference-executed
    golden."""
    res = run("server", mode)
    assert res["blocks"] == 4 and res["latents_rel_l2"] < 1e-2


def test_unmodified_classic_pipeline_on_the_dropins():
    res = run("classic")
    assert res["latents_rel_l2"] < 1e-3
