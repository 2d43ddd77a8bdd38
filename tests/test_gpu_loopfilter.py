"""GPU parity of the loop filters on the random configuration sweep (tests/synth/sweep.py): every picture stage by stage
(deblocked planes, SAO planes, RGB) against the CPU oracle after the oracle's deblocked and final planes have been
checked against the numpy restatement of 8.7.2 / 8.7.3 (tests/loopfilter_ref.py); then the whole sweep in one
heterogeneous call for the planes and one resident batch for the RGB.  tests/test_gpu_variants.py runs this file again
with SAO in its own pass (HEIC_B200_FUSE_SAO=0) and the one-warp-per-picture intra path (HEIC_B200_INTRA_SLOTS=1)."""
import numpy as np
import pytest

from oracle import oracle_py as O
from tests import loopfilter_ref as L
from tests.synth import synth
from tests.synth.sweep import SWEEP
from tests.test_gpu_synth import check_stages

pytestmark = pytest.mark.gpu


def _spec_checked_oracle(pic):
    """The oracle's decode of one picture, its loop-filter outputs asserted equal to the spec reference."""
    t = pic.tile
    ref = O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len))
    deblocked, final, _ = L.loop_filter(pic.sps, pic.pps, t.header, ref["recon"], ref["tu_map"], ref["qp_map"], ref["sao"])
    for c in range(len(final)):
        assert np.array_equal(deblocked[c], ref["deblocked"][c]) and np.array_equal(final[c], ref["plane"][c]), c
    return ref


def _expected_rgb(pic, planes):
    w, h = pic.sps.pic_width_in_luma_samples, pic.sps.pic_height_in_luma_samples
    if len(planes) == 1:  # 4:0:0 converts with neutral chroma
        neutral = np.full((h // 2) * (w // 2), 128, np.uint8)
        flat = np.concatenate([planes[0].ravel(), neutral, neutral])
    else:
        flat = np.concatenate([p.ravel() for p in planes])
    return O.color_stitch(flat, 1, 1, w, h, w, h, pic.sps.video_full_range_flag, pic.sps.matrix_coeffs)


@pytest.mark.parametrize("name,cfg,seed", SWEEP, ids=[n for n, _, _ in SWEEP])
def test_sweep_stages_match_reference(decoder, name, cfg, seed):
    pic = synth.encode(seed, **cfg)
    _spec_checked_oracle(pic)
    check_stages(decoder, pic)


def test_sweep_in_one_heterogeneous_call(decoder):
    """Every sweep picture in the same launches: CTB 16 / 32 / 64, 4:0:0 and 4:2:0, SAO and deblocking on and off
    side by side.  Planes through decode_grids_yuv, RGB through one resident batch decode."""
    pics = [synth.encode(seed, **cfg) for _, cfg, seed in SWEEP]
    exp = [_spec_checked_oracle(p)["plane"] for p in pics]
    res = decoder.decode_grids_yuv([p.desc for p in pics])
    for (name, _, _), planes, e in zip(SWEEP, res, exp):
        for c in range(len(e)):
            assert np.array_equal(planes[c], e[c]), (name, c)
    with decoder.batch([p.desc for p in pics]) as b:
        b.decode()
        b.sync()
        for i, ((name, _, _), pic, e) in enumerate(zip(SWEEP, pics, exp)):
            assert np.array_equal(b.download_image(i), _expected_rgb(pic, e)), name
