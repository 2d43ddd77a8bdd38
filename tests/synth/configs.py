"""The synthetic-stream test matrix (BASELINE.json configs[2]: single intra pictures exercising the path's features)."""
CONFIGS = [
    ("default_wpp_sao", dict()),
    ("no_wpp", dict(wpp=0)),
    ("ragged_200x136", dict(width=200, height=136)),
    ("ctb16", dict(log2_ctb=4, log2_max_tb=4, width=72, height=104)),
    ("ctb64", dict(log2_ctb=6, width=192, height=160)),
    ("ctb64_no_wpp_ragged", dict(log2_ctb=6, width=136, height=200, wpp=0)),
    ("transform_hierarchy_depth2", dict(max_transform_hierarchy_depth_intra=2)),
    ("sign_data_hiding", dict(sign_data_hiding=1, lps_gain=1.5)),
    ("transform_skip", dict(transform_skip=1)),
    ("cu_qp_delta_depth2", dict(cu_qp_delta=1, diff_cu_qp_delta_depth=2, init_qp_minus26=-6)),
    ("cu_qp_delta_chroma_offsets", dict(cu_qp_delta=1, diff_cu_qp_delta_depth=1, cb_qp_offset=3, cr_qp_offset=-4,
                                        slice_cb_qp_offset=1, slice_cr_qp_offset=-1, init_qp_minus26=8)),
    ("scaling_default", dict(scaling_list_mode=1)),
    ("scaling_sps_lists", dict(scaling_list_mode=2)),
    ("scaling_pps_lists", dict(scaling_list_mode=3, transform_skip=1)),
    ("monochrome", dict(chroma_format_idc=0)),
    ("no_sao", dict(sao=0)),
    ("no_deblock", dict(deblocking_disabled=1)),
    ("deblock_offsets", dict(beta_offset_div2=2, tc_offset_div2=-3)),
    ("strong_smoothing_high_qp", dict(strong_intra_smoothing=1, init_qp_minus26=15, lps_gain=0.6)),
    ("min_cb16_tb8_ctb64", dict(log2_min_cb=4, log2_min_tb=3, log2_ctb=6, width=160, height=144)),
    ("sao_luma_only", dict(slice_sao_chroma=0)),
    ("sao_chroma_only", dict(slice_sao_luma=0)),
    ("low_qp_busy", dict(init_qp_minus26=-20, lps_gain=2.0)),
    ("high_qp", dict(init_qp_minus26=25)),
    ("limited_range_bt709", dict(full_range=0, matrix_coeffs=1)),
    ("one_ctb_column", dict(width=32, height=160)),
    ("one_ctb", dict(width=32, height=32)),
    ("tiny_8x8", dict(width=8, height=8)),
    ("wide_512x64", dict(width=512, height=64)),
    # as many CTB rows as the CABAC kernel has row slots (every warp owns exactly one row: the shape ADVICE r1 flagged for
    # the persistent hand-over) and a pool-style stream with the encoder-like SAO / split statistics of tests/synth/pool.py
    ("wide_short_512x256", dict(width=512, height=256)),
    ("pool_style_light", dict(width=256, height=256, scaling_list_mode=1, cu_qp_delta=1, diff_cu_qp_delta_depth=2, init_qp_minus26=-11,
                              cb_qp_offset=2, cr_qp_offset=2, slice_qp_delta=24, lps_gain=0.5, split_cu_prob=0.25, sao_on_prob=0.03)),
    ("everything", dict(width=264, height=200, log2_ctb=6, max_transform_hierarchy_depth_intra=1, sign_data_hiding=1,
                        transform_skip=1, cu_qp_delta=1, diff_cu_qp_delta_depth=3, scaling_list_mode=2, strong_intra_smoothing=1,
                        cb_qp_offset=-2, cr_qp_offset=5, init_qp_minus26=-3, lps_gain=1.3)),
]
SEEDS = (0, 1)

# Value-range extremes, kept apart from CONFIGS (whose streams are pinned to FFmpeg hashes): escape-coded levels up to
# 32767 (big_level_prob), explicit scaling lists over the whole legal range 1..255, QP 0 and 51, cu_qp_delta wrapping
# around 0/51, chroma QP offsets of +-12 and deblocking offsets of +-6.  Scaled coefficients saturate at both int16 ends,
# the 64-bit scaling branch of the transform kernels runs, residuals reach ~23 K and reconstructed samples pin to 0 / 255.
_BIG = dict(big_level_prob=0.3, max_transform_hierarchy_depth_intra=1)
_FULL_LISTS = dict(scaling_list_min=1, scaling_list_max=255)
EXTREME_CONFIGS = [
    ("big_qp51_flat", dict(_BIG, init_qp_minus26=25)),
    ("big_qp51_sps_lists", dict(_BIG, **_FULL_LISTS, init_qp_minus26=25, scaling_list_mode=2)),
    ("big_qp51_pps_lists_tskip", dict(_BIG, **_FULL_LISTS, init_qp_minus26=25, scaling_list_mode=3, transform_skip=1)),
    ("big_qp0", dict(_BIG, init_qp_minus26=-26, transform_skip=1)),
    # lists of ones at QP 30 with few, large 16x16 / 32x32 blocks: the kernels' 32-bit product test (which assumes entries
    # up to 255) fails on blocks whose scaled coefficients stay in range, so the 64-bit branch yields unsaturated values
    ("big_qp30_unit_lists", dict(big_level_prob=0.05, init_qp_minus26=4, scaling_list_mode=2, scaling_list_min=1, scaling_list_max=1,
                                 split_cu_prob=0.2, width=256, height=256)),
    ("big_qp51_ctb64", dict(_BIG, init_qp_minus26=25, log2_ctb=6, width=192, height=128, scaling_list_mode=1)),
    ("big_qp51_ctb16", dict(_BIG, init_qp_minus26=25, log2_ctb=4, log2_max_tb=4, width=96, height=80)),
    ("cu_qp_delta_low_qp", dict(_BIG, cu_qp_delta=1, diff_cu_qp_delta_depth=2, init_qp_minus26=-25)),
    ("cu_qp_delta_high_qp", dict(_BIG, cu_qp_delta=1, diff_cu_qp_delta_depth=2, init_qp_minus26=24)),
    ("chroma_offsets_pps12_slice_m12", dict(_BIG, init_qp_minus26=10, cb_qp_offset=12, cr_qp_offset=12, slice_cb_qp_offset=-12,
                                            slice_cr_qp_offset=-12, cu_qp_delta=1, diff_cu_qp_delta_depth=1)),
    ("chroma_offsets_pps_m12_slice12", dict(_BIG, init_qp_minus26=10, cb_qp_offset=-12, cr_qp_offset=-12, slice_cb_qp_offset=12,
                                            slice_cr_qp_offset=12, cu_qp_delta=1, diff_cu_qp_delta_depth=1)),
    ("deblock_plus6_qp51", dict(_BIG, init_qp_minus26=25, beta_offset_div2=6, tc_offset_div2=6)),
    ("deblock_plus6_qp30", dict(_BIG, init_qp_minus26=4, beta_offset_div2=6, tc_offset_div2=6)),
    ("deblock_minus6_qp51", dict(_BIG, init_qp_minus26=25, beta_offset_div2=-6, tc_offset_div2=-6)),
    ("deblock_minus6_qp30", dict(_BIG, init_qp_minus26=4, beta_offset_div2=-6, tc_offset_div2=-6)),
    ("big_monochrome", dict(_BIG, init_qp_minus26=25, chroma_format_idc=0)),
]
EXTREME_SEEDS = (0, 1)

# Directed intra-prediction streams, kept apart from CONFIGS (tests/test_intra_reference.py, test_gpu_intra.py).  Random
# syntax alone puts the picture edge through a below-left or above-right neighbour a handful of times and rarely codes
# large blocks; these pictures do it on purpose:
# - widths and heights = 8, 16 or 24 (mod 32) and 40 .. 56 (mod 64) at CTB 16 / 32 / 64, so that the picture's right and
#   bottom edges cut the above-right and below-left samples of 16x16 / 32x32 luma and 8x8 / 16x16 chroma blocks;
# - few CU splits with MaxTb 32 (many 32x32 luma and 16x16 chroma blocks), and min TB 4 with many 8x8 CUs (NxN
#   partitions: 4x4 luma units, chroma 4x4 of a split 8x8);
# - few coded blocks (cbf_prob) for smooth pictures on which strong intra smoothing passes its flatness tests, each such
#   stream once with strong smoothing on and once off (the same slice data: the walk does not depend on the flag);
# - one CTB row, one CTB column, 8x8 and 4:0:0 pictures;
# - about half with deblocking and SAO off: FFmpeg's output then is the intra reconstruction itself.
_BIG32 = dict(log2_max_tb=5, split_cu_prob=0.1)
_NO_LF = dict(deblocking_disabled=1, sao=0)
_SMOOTH64 = dict(_BIG32, log2_ctb=6, width=512, height=304, cbf_prob=0.15)
_SMOOTH32 = dict(_BIG32, width=480, height=272, cbf_prob=0.3)
INTRA_CONFIGS = [
    ("ctb64_big_520x296", dict(_BIG32, log2_ctb=6, width=520, height=296)),
    ("ctb64_big_584x360_no_lf", dict(_BIG32, **_NO_LF, log2_ctb=6, width=584, height=360)),
    ("ctb64_big_616x312_no_wpp", dict(_BIG32, log2_ctb=6, width=616, height=312, wpp=0)),
    ("ctb32_big_520x280_no_lf", dict(_BIG32, **_NO_LF, width=520, height=280)),
    ("ctb32_big_464x344", dict(_BIG32, width=464, height=344)),
    ("ctb64_smooth_strong_no_lf", dict(_SMOOTH64, **_NO_LF, strong_intra_smoothing=1)),
    ("ctb64_smooth_no_strong_no_lf", dict(_SMOOTH64, **_NO_LF, strong_intra_smoothing=0)),
    ("ctb32_smooth_strong", dict(_SMOOTH32, strong_intra_smoothing=1)),
    ("ctb32_smooth_no_strong", dict(_SMOOTH32, strong_intra_smoothing=0)),
    ("ctb16_208x136_no_lf", dict(_NO_LF, log2_ctb=4, log2_max_tb=4, width=208, height=136, split_cu_prob=0.3)),
    ("ctb32_mid_328x248_mpm", dict(width=328, height=248, split_cu_prob=0.4, log2_max_tb=4, prev_intra_prob=0.8)),
    ("ctb64_mid_344x280_no_lf", dict(_NO_LF, log2_ctb=6, width=344, height=280, split_cu_prob=0.4, log2_max_tb=4,
                                     prev_intra_prob=0.2)),
    ("nxn_264x200", dict(width=264, height=200, split_cu_prob=0.9)),
    ("nxn_ctb16_136x120_no_lf", dict(_NO_LF, log2_ctb=4, log2_max_tb=4, width=136, height=120, split_cu_prob=0.9)),
    ("one_ctb_row_ctb64_584x56_no_lf", dict(_BIG32, **_NO_LF, log2_ctb=6, width=584, height=56)),
    ("one_ctb_column_24x328", dict(_BIG32, width=24, height=328)),
    ("one_ctb_column_ctb64_40x264_no_lf", dict(_BIG32, **_NO_LF, log2_ctb=6, width=40, height=264)),
    ("tiny_8x8_no_lf", dict(_NO_LF, width=8, height=8)),
    ("monochrome_ctb64_520x296", dict(_BIG32, log2_ctb=6, width=520, height=296, chroma_format_idc=0, strong_intra_smoothing=1,
                                      cbf_prob=0.2)),
]
INTRA_SEEDS = (0, 1)
