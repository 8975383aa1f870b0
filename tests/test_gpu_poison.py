"""The parity tests once more with every scratch slot of the library poisoned (0xFF bytes: NaN doubles, -1 counts) each time
an entry point asks for it -- ORT_POISON_SCRATCH=1, csrc/ort_api.cu ort_ensure.  A kernel that reads scratch it did not
write, or an output the library forgets to write (k_paraxial_final's clip_idx without the clip test was one: the result
depended on what the block held before), then fails a parity assertion instead of passing by the luck of the allocation.
compute-sanitizer is closed on the GPU pool this repository is measured on; this is the check of our own that stands in."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FILES = ["tests/test_gpu_trace3d.py", "tests/test_gpu_first_order.py", "tests/test_gpu_random_systems.py",
         "tests/test_gpu_sweep_outputs.py"]


@pytest.mark.gpu
@pytest.mark.skipif(os.environ.get("ORT_POISON_SCRATCH") == "1", reason="already inside the poisoned run")
def test_parity_suite_with_poisoned_scratch():
    env = dict(os.environ, ORT_POISON_SCRATCH="1")
    r = subprocess.run([sys.executable, "-m", "pytest", *FILES, "-m", "gpu", "-x", "-q", "-p", "no:cacheprovider"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-2000:]
    assert " passed" in r.stdout
