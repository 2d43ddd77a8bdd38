"""The opt-out paths selected by environment variables (read once per process, hence the subprocess): the register
butterflies for 8x8 .. 32x32 transforms (HEIC_B200_TRANSFORM_MMA=0, the A/B partner of the tensor-core kernels; on the
ordinary synthetic streams and at the value-range extremes), the unordered chunk pipeline (HEIC_B200_PIPE_ORDER=0), and
SAO in its own pass (HEIC_B200_FUSE_SAO=0) together with the one-warp-per-picture intra path that bench.py's batches run
(HEIC_B200_INTRA_SLOTS=1), on the random configuration sweep, must stay bit-exact too."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize(
    "env,target",
    [
        ({"HEIC_B200_TRANSFORM_MMA": "0"}, "tests/test_gpu_synth.py::test_stages_match_oracle"),
        ({"HEIC_B200_TRANSFORM_MMA": "0"}, "tests/test_gpu_extremes.py"),
        ({"HEIC_B200_PIPE_ORDER": "0"}, "tests/test_gpu_pipeline.py"),
        ({"HEIC_B200_FUSE_SAO": "0", "HEIC_B200_INTRA_SLOTS": "1"}, "tests/test_gpu_loopfilter.py"),
    ],
    ids=["transform_butterflies", "transform_butterflies_extremes", "pipeline_unordered", "sao_pass_intra_one_warp_sweep"],
)
def test_opt_out_path_is_bit_exact(built, env, target):
    e = dict(os.environ)
    e.update(env)
    r = subprocess.run([sys.executable, "-m", "pytest", target, "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider"], cwd=ROOT, env=e,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
