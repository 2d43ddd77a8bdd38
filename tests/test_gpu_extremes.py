"""GPU parity at the value-range extremes (tests/synth/configs.py EXTREME_CONFIGS): escape-coded levels up to 32767,
scaled coefficients saturating at both int16 ends, the 64-bit scaling branch, clipped first transform stages, QP 0 / 51
with cu_qp_delta wrap-around, chroma QP offsets of +-12 and deblocking offsets of +-6.  Stage by stage against the CPU
oracle, the residual also against the numpy restatement of 8.6.x (tests/transform_ref.py), and all of it in one call
mixed with the ordinary synthetic streams so that 64-bit and 32-bit scaled blocks share the transform kernels' warps."""
import numpy as np
import pytest

from oracle import oracle_py as O
from tests import transform_ref as R
from tests.synth import synth
from tests.synth.configs import CONFIGS, EXTREME_CONFIGS, EXTREME_SEEDS, SEEDS
from tests.test_gpu_synth import check_stages

pytestmark = pytest.mark.gpu
CASES = [(name, cfg, seed) for name, cfg in EXTREME_CONFIGS for seed in EXTREME_SEEDS]


@pytest.mark.parametrize("name,cfg,seed", CASES, ids=[f"{n}/{s}" for n, _, s in CASES])
def test_extreme_stages_match_oracle_and_reference(decoder, name, cfg, seed):
    pic = synth.encode(seed, **cfg)
    resid = check_stages(decoder, pic)
    t = pic.tile
    ref = O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len), parse_only=True)
    exp, _ = R.residuals(pic.sps, pic.pps, t.header, ref["tu_map"], ref["level"])
    for c, (a, b) in enumerate(zip(resid, exp)):
        assert np.array_equal(a, b), f"residual {c} differs from the numpy reference in {int((a != b).sum())} samples"


def test_extremes_mixed_with_ordinary_streams_in_one_call(decoder):
    pics = [synth.encode(seed, **cfg) for _, cfg, seed in CASES]
    pics += [synth.encode(seed, **cfg) for _, cfg in CONFIGS for seed in SEEDS]
    order = np.random.default_rng(7).permutation(len(pics))  # interleave the two kinds of tiles
    pics = [pics[i] for i in order]
    res = decoder.decode_grids_yuv([p.desc for p in pics])
    for pic, planes in zip(pics, res):
        t = pic.tile
        ref = O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len), intermediates=False)
        for c in range(len(ref["plane"])):
            assert np.array_equal(planes[c], ref["plane"][c]), (pic.cfg, c)
