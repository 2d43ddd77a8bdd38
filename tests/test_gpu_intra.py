"""GPU intra prediction on the directed INTRA_CONFIGS streams (tests/synth/configs.py): every picture stage by stage
against the CPU oracle (after the oracle's `recon` has been checked against the numpy restatement of 8.4.4.2,
tests/intra_ref.py), and the GPU's intra stage against that restatement run on the GPU's own `tu_map` and residuals;
then all the pictures in one heterogeneous call against the reference chain (intra_ref, then loopfilter_ref where the
loop filters are on).  tests/test_gpu_variants.py runs this file again with the one-warp-per-picture intra path
(HEIC_B200_INTRA_SLOTS=1); the default run takes the multi-warp wavefront for these batch sizes."""
import numpy as np
import pytest

import heif_b200 as H
from oracle import oracle_py as O
from tests import intra_ref as I
from tests import loopfilter_ref as L
from tests.synth import synth
from tests.synth.configs import INTRA_CONFIGS, INTRA_SEEDS
from tests.test_gpu_synth import check_stages

pytestmark = pytest.mark.gpu
INTRA_STREAMS = [(name, cfg, seed) for name, cfg in INTRA_CONFIGS for seed in INTRA_SEEDS]


def _spec_checked_oracle(pic):
    """The oracle's decode of one picture, its `recon` asserted equal to the spec reference; and the reference's final
    planes (the loop-filter reference applied to the intra reference)."""
    t = pic.tile
    ref = O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len))
    recon, _ = I.reconstruct(pic.sps, ref["tu_map"], ref["resid"])
    for c in range(len(recon)):
        assert np.array_equal(recon[c], ref["recon"][c]), c
    _, final, _ = L.loop_filter(pic.sps, pic.pps, t.header, recon, ref["tu_map"], ref["qp_map"], ref["sao"])
    return ref, final


def _assert_gpu_intra_matches_reference(decoder, pic):
    """The intra stage's output planes == intra_ref applied to the GPU's own tu_map and residuals."""
    n_comp = 3 if pic.sps.chroma_format_idc else 1
    with decoder.batch([pic.desc]) as b:
        b.run(H.STAGE_CABAC)
        b.sync()
        assert b.status()[0].code == 0
        b.run(H.STAGE_TRANSFORM)
        d = b.dump_tile(0)
        tu_map, resid = d["tu_map"], [np.array(d["coeff"][c]) for c in range(n_comp)]
        b.run(H.STAGE_INTRA)
        planes = b.dump_tile(0)["plane"]
    expected, _ = I.reconstruct(pic.sps, tu_map, resid)
    for c in range(n_comp):
        bad = planes[c] != expected[c]
        assert not bad.any(), f"intra {c}: {int(bad.sum())} samples differ, e.g. (y, x) {np.argwhere(bad)[:4].tolist()}"


@pytest.mark.parametrize("name,cfg,seed", INTRA_STREAMS, ids=[f"{n}/{s}" for n, _, s in INTRA_STREAMS])
def test_intra_stages_match_reference(decoder, name, cfg, seed):
    pic = synth.encode(seed, **cfg)
    _spec_checked_oracle(pic)
    check_stages(decoder, pic)
    _assert_gpu_intra_matches_reference(decoder, pic)


def test_intra_streams_in_one_heterogeneous_call(decoder):
    """Every INTRA_CONFIGS picture in the same launches: CTB 16 / 32 / 64, 4:0:0 and 4:2:0, 8x8 up to 616x312, strong
    smoothing and the loop filters on and off side by side."""
    pics = [synth.encode(seed, **cfg) for _, cfg, seed in INTRA_STREAMS]
    exp = [_spec_checked_oracle(p)[1] for p in pics]
    res = decoder.decode_grids_yuv([p.desc for p in pics])
    for (name, _, seed), planes, e in zip(INTRA_STREAMS, res, exp):
        for c in range(len(e)):
            assert np.array_equal(planes[c], e[c]), (name, seed, c)
