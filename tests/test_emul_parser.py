"""The per-thread device parser (heif_b200/csrc/cuda/cabac_parse.cuh) compiled for the host and run against the oracle:
checks the CUDA syntax logic bit-for-bit without a GPU (tests/emul/cabac_emul.cc is test infrastructure only)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from heif_b200 import _capi as K
from oracle import oracle_py as O

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module", params=["nested"])
def emul(request):
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "emul")])
    name = {"nested": "libcabac_emul.so"}[request.param]
    lib = C.CDLL(os.path.join(HERE, "emul", "_build", name))
    lib.emul_parse_picture.argtypes = ([C.POINTER(K.Sps), C.POINTER(K.Pps), C.POINTER(K.SliceHeader), C.c_void_p, C.c_uint32]
                                       + [C.c_void_p] * 6 + [C.POINTER(C.c_uint32)] * 2 + [C.c_int])
    return lib


@pytest.mark.parametrize("tile", [0, 5, 17, 23, 31, 47])
@pytest.mark.parametrize("per_row_threads", [0, 1])
def test_device_parser_matches_oracle(emul, heic_file, tile, per_row_threads):
    img = heic_file.primary
    td = img.tiles[tile]
    ref = O.decode_picture(img.sps, img.pps, td.header, (td.rbsp, td.rbsp_len), parse_only=True)
    n_tu = len(ref["tu_map"])
    tu = np.zeros(n_tu, np.uint32)
    lv = [np.zeros(n_tu * 16, np.int16), np.zeros(n_tu * 4, np.int16), np.zeros(n_tu * 4, np.int16)]
    qp = np.zeros((64, 64), np.uint8)
    sao = np.zeros(256 * 4, np.uint32)
    bins, ctus = C.c_uint32(), C.c_uint32()
    rc = emul.emul_parse_picture(C.byref(img.sps), C.byref(img.pps), C.byref(td.header), td.rbsp, td.rbsp_len, tu.ctypes.data,
                                 lv[0].ctypes.data, lv[1].ctypes.data, lv[2].ctypes.data, qp.ctypes.data, sao.ctypes.data,
                                 C.byref(bins), C.byref(ctus), per_row_threads)
    assert rc == 0
    assert np.array_equal(tu, ref["tu_map"])
    for c in range(3):
        assert np.array_equal(lv[c], ref["level"][c])
    assert np.array_equal(qp, ref["qp_map"]) and np.array_equal(sao, ref["sao"])
    assert (bins.value, ctus.value) == (ref["bins"], ref["ctus"])


def test_device_parser_rejects_garbage_without_hanging(emul, heic_file):
    img = heic_file.primary
    td = img.tiles[3]
    bad = bytearray(bytes(td.rbsp[: td.rbsp_len]))
    for i in range(td.header.slice_data_byte_offset + 40, len(bad)):
        bad[i] = (bad[i] * 73 + 41) & 0xFF
    buf = (C.c_uint8 * len(bad)).from_buffer(bad)
    n_tu = 256 * 64
    tu = np.zeros(n_tu, np.uint32)
    lv = [np.zeros(n_tu * 16, np.int16), np.zeros(n_tu * 4, np.int16), np.zeros(n_tu * 4, np.int16)]
    qp = np.zeros((64, 64), np.uint8)
    sao = np.zeros(256 * 4, np.uint32)
    bins, ctus = C.c_uint32(), C.c_uint32()
    rc = emul.emul_parse_picture(C.byref(img.sps), C.byref(img.pps), C.byref(td.header), buf, len(bad), tu.ctypes.data,
                                 lv[0].ctypes.data, lv[1].ctypes.data, lv[2].ctypes.data, qp.ctypes.data, sao.ctypes.data,
                                 C.byref(bins), C.byref(ctus), 1)
    assert rc != 0  # end_of_slice / end_of_subset checks trip; no out-of-bounds write, no hang


def _synth_cases():
    from tests.synth.configs import CONFIGS, SEEDS

    return [(name, cfg, SEEDS[0]) for name, cfg in CONFIGS]


def _extreme_cases():
    from tests.synth.configs import EXTREME_CONFIGS, EXTREME_SEEDS

    return [(name, cfg, seed) for name, cfg in EXTREME_CONFIGS for seed in EXTREME_SEEDS]


@pytest.mark.parametrize("name,cfg,seed", _synth_cases() + _extreme_cases(),
                         ids=[c[0] for c in _synth_cases()] + [f"{c[0]}/{c[2]}" for c in _extreme_cases()])
def test_device_parser_matches_oracle_on_synthetic_streams(emul, name, cfg, seed):
    """Every feature configuration of the synthetic generator (CTB 16/64, no WPP, transform skip, sign data hiding,
    cu_qp_delta, transform hierarchy, 4:0:0, ragged sizes, ...) through the host build of the device parser; and the
    value-range extremes (escape-coded levels up to 32767, QP 0 / 51, cu_qp_delta wrap-around)."""
    from tests.synth import synth

    pic = synth.encode(seed, **cfg)
    t = pic.tile
    ref = O.decode_picture(pic.sps, pic.pps, t.header, (t.rbsp, t.rbsp_len), parse_only=True)
    n_tu = len(ref["tu_map"])
    tu = np.zeros(n_tu, np.uint32)
    lv = [np.zeros(n_tu * 16, np.int16), np.zeros(n_tu * 4, np.int16), np.zeros(n_tu * 4, np.int16)]
    qp = np.zeros(ref["qp_map"].shape, np.uint8)
    sao = np.zeros(ref["sao"].size, np.uint32)
    for per_row_threads in (0, 1):
        bins, ctus = C.c_uint32(), C.c_uint32()
        rc = emul.emul_parse_picture(C.byref(pic.sps), C.byref(pic.pps), C.byref(t.header), t.rbsp, t.rbsp_len, tu.ctypes.data,
                                     lv[0].ctypes.data, lv[1].ctypes.data, lv[2].ctypes.data, qp.ctypes.data, sao.ctypes.data,
                                     C.byref(bins), C.byref(ctus), per_row_threads)
        assert rc == 0
        assert np.array_equal(tu, ref["tu_map"])
        for c in range(len(ref["level"])):
            assert np.array_equal(lv[c][: ref["level"][c].size], ref["level"][c]), (name, c)
        assert np.array_equal(qp, ref["qp_map"]) and np.array_equal(sao, ref["sao"].ravel())
        assert (bins.value, ctus.value) == (ref["bins"], ref["ctus"])


# ---- the state-machine walker (tools/experiments/cabac_fsm: a measured, not adopted, alternative to the nested walker) ----
@pytest.fixture(scope="module")
def fsm(emul):
    emul.emul_parse_picture_fsm.argtypes = ([C.POINTER(K.Sps), C.POINTER(K.Pps), C.POINTER(K.SliceHeader), C.c_void_p, C.c_uint32]
                                            + [C.c_void_p] * 6 + [C.POINTER(C.c_uint32)] * 2 + [C.c_int, C.c_int, C.POINTER(C.c_uint64)])
    return emul


def _run_fsm(fsm, sps, pps, header, rbsp, rbsp_len, n_slots, repeat):
    ref = O.decode_picture(sps, pps, header, (rbsp, rbsp_len), parse_only=True)
    n_tu = len(ref["tu_map"])
    tu = np.zeros(n_tu, np.uint32)
    lv = [np.zeros(n_tu * 16, np.int16), np.zeros(n_tu * 4, np.int16), np.zeros(n_tu * 4, np.int16)]
    qp = np.zeros(ref["qp_map"].shape, np.uint8)
    sao = np.zeros(ref["sao"].size, np.uint32)
    bins, ctus, steps = C.c_uint32(), C.c_uint32(), C.c_uint64()
    rc = fsm.emul_parse_picture_fsm(C.byref(sps), C.byref(pps), C.byref(header), rbsp, rbsp_len, tu.ctypes.data, lv[0].ctypes.data,
                                    lv[1].ctypes.data, lv[2].ctypes.data, qp.ctypes.data, sao.ctypes.data, C.byref(bins), C.byref(ctus),
                                    n_slots, repeat, C.byref(steps))
    assert rc == 0
    assert np.array_equal(tu, ref["tu_map"])
    for c in range(len(ref["level"])):
        assert np.array_equal(lv[c][: ref["level"][c].size], ref["level"][c]), c
    assert np.array_equal(qp, ref["qp_map"]) and np.array_equal(sao, ref["sao"].ravel())
    assert (bins.value, ctus.value) == (ref["bins"], ref["ctus"])
    return steps.value, ref["bins"]


@pytest.mark.parametrize("tile", [0, 5, 17, 23, 31, 47])
@pytest.mark.parametrize("n_slots,repeat", [(1, 1), (8, 1), (5, 6)])
def test_state_machine_walker_matches_oracle(fsm, heic_file, tile, n_slots, repeat):
    """One thread for all rows, the device's 8 row slots, and an odd slot count decoding the tile six times in a row through
    the column's 4-entry tile ring (the hand-over protocol of cabac_fsm_kernel.cu, restated in the host environment)."""
    img = heic_file.primary
    td = img.tiles[tile]
    steps, bins = _run_fsm(fsm, img.sps, img.pps, td.header, td.rbsp, td.rbsp_len, n_slots, repeat)
    if n_slots == 1:
        assert steps <= bins + 4096  # an iteration per bin at most (bypass bins come several at a time), plus the no-op hops


@pytest.mark.parametrize("name,cfg,seed", _synth_cases(), ids=[c[0] for c in _synth_cases()])
def test_state_machine_walker_matches_oracle_on_synthetic_streams(fsm, name, cfg, seed):
    from tests.synth import synth

    pic = synth.encode(seed, **cfg)
    t = pic.tile
    for n_slots, repeat in ((1, 1), (3, 5), (8, 2)):
        _run_fsm(fsm, pic.sps, pic.pps, t.header, t.rbsp, t.rbsp_len, n_slots, repeat)


def test_state_machine_walker_rejects_garbage_without_hanging(fsm, heic_file):
    img = heic_file.primary
    td = img.tiles[3]
    bad = bytearray(bytes(td.rbsp[: td.rbsp_len]))
    for i in range(td.header.slice_data_byte_offset + 40, len(bad)):
        bad[i] = (bad[i] * 73 + 41) & 0xFF
    buf = (C.c_uint8 * len(bad)).from_buffer(bad)
    n_tu = 256 * 64
    tu = np.zeros(n_tu, np.uint32)
    lv = [np.zeros(n_tu * 16, np.int16), np.zeros(n_tu * 4, np.int16), np.zeros(n_tu * 4, np.int16)]
    qp = np.zeros((64, 64), np.uint8)
    sao = np.zeros(256 * 4, np.uint32)
    for n_slots in (1, 8):
        bins, ctus = C.c_uint32(), C.c_uint32()
        rc = fsm.emul_parse_picture_fsm(C.byref(img.sps), C.byref(img.pps), C.byref(td.header), buf, len(bad), tu.ctypes.data,
                                        lv[0].ctypes.data, lv[1].ctypes.data, lv[2].ctypes.data, qp.ctypes.data, sao.ctypes.data,
                                        C.byref(bins), C.byref(ctus), n_slots, 2, None)
        assert rc != 0 and rc != -99  # flagged, and the other rows of the tile were released (no hang)
