"""ctypes declarations for include/heic_b200.h (the C ABI).  Pure plumbing — no computation here.

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a) as
``heif_b200/libheic_b200.so``.  There is no fallback: if it is missing, importing the product
API raises.
"""
from __future__ import annotations

import ctypes as C
import os

HEIC_MAX_ENTRY_POINTS = 255

HEIC_OK = 0
HEIC_E_INVALID_ARG = -1
HEIC_E_UNSUPPORTED = -2
HEIC_E_BITSTREAM = -3
HEIC_E_NO_DEVICE = -4
HEIC_E_CUDA = -5
HEIC_E_NOMEM = -6

STAGE_CABAC, STAGE_TRANSFORM, STAGE_INTRA, STAGE_DEBLOCK, STAGE_SAO, STAGE_COLOR = 1, 2, 4, 8, 16, 32
STAGE_ALL = 63

u8, u32, i32 = C.c_uint8, C.c_uint32, C.c_int32


class ScalingList(C.Structure):
    _fields_ = [("list", u8 * 64 * 6 * 4), ("dc", u8 * 6 * 2)]


def _u32_fields(names):
    return [(n.strip(), u32) for n in names.split(",")]


class Sps(C.Structure):
    _fields_ = (
        _u32_fields(
            "sps_video_parameter_set_id,sps_max_sub_layers_minus1,sps_temporal_id_nesting_flag,"
            "sps_seq_parameter_set_id,chroma_format_idc,separate_colour_plane_flag,"
            "pic_width_in_luma_samples,pic_height_in_luma_samples,conformance_window_flag,"
            "conf_win_left_offset,conf_win_right_offset,conf_win_top_offset,conf_win_bottom_offset,"
            "bit_depth_luma_minus8,bit_depth_chroma_minus8,log2_max_pic_order_cnt_lsb_minus4,"
            "log2_min_luma_coding_block_size_minus3,log2_diff_max_min_luma_coding_block_size,"
            "log2_min_luma_transform_block_size_minus2,log2_diff_max_min_luma_transform_block_size,"
            "max_transform_hierarchy_depth_inter,max_transform_hierarchy_depth_intra,"
            "scaling_list_enabled_flag,sps_scaling_list_data_present_flag,amp_enabled_flag,"
            "sample_adaptive_offset_enabled_flag,pcm_enabled_flag,pcm_sample_bit_depth_luma_minus1,"
            "pcm_sample_bit_depth_chroma_minus1,log2_min_pcm_luma_coding_block_size_minus3,"
            "log2_diff_max_min_pcm_luma_coding_block_size,pcm_loop_filter_disabled_flag,"
            "num_short_term_ref_pic_sets,long_term_ref_pics_present_flag,sps_temporal_mvp_enabled_flag,"
            "strong_intra_smoothing_enabled_flag,vui_parameters_present_flag,video_full_range_flag,"
            "colour_primaries,transfer_characteristics,matrix_coeffs"
        )
        + [("scaling_list", ScalingList)]
    )


class Pps(C.Structure):
    _fields_ = [
        ("pps_pic_parameter_set_id", u32), ("pps_seq_parameter_set_id", u32),
        ("dependent_slice_segments_enabled_flag", u32), ("output_flag_present_flag", u32),
        ("num_extra_slice_header_bits", u32), ("sign_data_hiding_enabled_flag", u32),
        ("cabac_init_present_flag", u32), ("num_ref_idx_l0_default_active_minus1", u32),
        ("num_ref_idx_l1_default_active_minus1", u32), ("init_qp_minus26", i32),
        ("constrained_intra_pred_flag", u32), ("transform_skip_enabled_flag", u32),
        ("cu_qp_delta_enabled_flag", u32), ("diff_cu_qp_delta_depth", u32),
        ("pps_cb_qp_offset", i32), ("pps_cr_qp_offset", i32),
        ("pps_slice_chroma_qp_offsets_present_flag", u32), ("weighted_pred_flag", u32),
        ("weighted_bipred_flag", u32), ("transquant_bypass_enabled_flag", u32),
        ("tiles_enabled_flag", u32), ("entropy_coding_sync_enabled_flag", u32),
        ("num_tile_columns_minus1", u32), ("num_tile_rows_minus1", u32), ("uniform_spacing_flag", u32),
        ("loop_filter_across_tiles_enabled_flag", u32),
        ("pps_loop_filter_across_slices_enabled_flag", u32),
        ("deblocking_filter_control_present_flag", u32),
        ("deblocking_filter_override_enabled_flag", u32),
        ("pps_deblocking_filter_disabled_flag", u32), ("pps_beta_offset_div2", i32),
        ("pps_tc_offset_div2", i32), ("pps_scaling_list_data_present_flag", u32),
        ("lists_modification_present_flag", u32), ("log2_parallel_merge_level_minus2", u32),
        ("slice_segment_header_extension_present_flag", u32), ("scaling_list", ScalingList),
    ]


class SliceHeader(C.Structure):
    _fields_ = [
        ("first_slice_segment_in_pic_flag", u32), ("no_output_of_prior_pics_flag", u32),
        ("slice_pic_parameter_set_id", u32), ("slice_type", u32),
        ("slice_sao_luma_flag", u32), ("slice_sao_chroma_flag", u32), ("slice_qp_delta", i32),
        ("slice_cb_qp_offset", i32), ("slice_cr_qp_offset", i32),
        ("deblocking_filter_override_flag", u32), ("slice_deblocking_filter_disabled_flag", u32),
        ("slice_beta_offset_div2", i32), ("slice_tc_offset_div2", i32),
        ("slice_loop_filter_across_slices_enabled_flag", u32), ("num_entry_point_offsets", u32),
        ("entry_point_offset_minus1", u32 * HEIC_MAX_ENTRY_POINTS),
        ("slice_data_byte_offset", u32),
        ("substream_offset", u32 * (HEIC_MAX_ENTRY_POINTS + 1)),
    ]


class TileDesc(C.Structure):
    _fields_ = [("rbsp", C.POINTER(u8)), ("rbsp_len", u32), ("nal_unit_type", u32), ("escaped", u32), ("header", SliceHeader)]


class ImageDesc(C.Structure):
    _fields_ = [
        ("sps", Sps), ("pps", Pps), ("grid_rows", u32), ("grid_cols", u32),
        ("output_width", u32), ("output_height", u32), ("rotation_ccw_quarter_turns", u32),
        ("n_tiles", u32), ("tiles", C.POINTER(TileDesc)),
    ]


class ImageTransform(C.Structure):
    """heic_image_transform: out = canvas[crop_y:crop_y+crop_h, crop_x:crop_x+crop_w], rotated by orientation & 3 ccw quarter
    turns, then mirrored left<->right when orientation & 4."""
    _fields_ = _u32_fields("crop_x,crop_y,crop_w,crop_h,orientation")


class TileStatus(C.Structure):
    _fields_ = [("code", i32), ("bins_decoded", u32), ("ctus_decoded", u32), ("reserved", u32)]


class FileInfo(C.Structure):
    _fields_ = _u32_fields(
        "primary_item_id,ispe_width,ispe_height,rotation_ccw_quarter_turns,rotated_width,"
        "rotated_height,luma_bits,chroma_bits,thumbnail_count,item_count,is_grid"
    )


class TileDump(C.Structure):
    _fields_ = [
        ("tu_map", C.POINTER(u32)), ("tu_map_len", u32),
        ("coeff", C.POINTER(C.c_int16) * 3), ("coeff_len", u32 * 3),
        ("qp_map", C.POINTER(u8)), ("qp_map_len", u32),
        ("sao", C.POINTER(u32)), ("sao_len", u32),
        ("plane", C.POINTER(u8) * 3), ("plane_len", u32 * 3),
    ]


LIB_NAME = "libheic_b200.so"
LIB_PATH = os.environ.get("HEIC_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)  # env: A/B builds

# Every symbol include/heic_b200.h declares: (name, restype, argtypes).
_vp, _sz = C.c_void_p, C.c_size_t
SYMBOLS = [
    ("heic_b200_abi_version", i32, []),
    ("heic_b200_last_error", C.c_char_p, []),
    ("heic_b200_create", i32, [i32, C.POINTER(_vp)]),
    ("heic_b200_destroy", None, [_vp]),
    ("heic_b200_launch_count", C.c_uint64, [_vp]),
    ("heic_b200_remove_emulation_prevention", C.c_int64,
     [C.c_char_p, _sz, C.POINTER(u8), C.POINTER(u32), _sz, C.POINTER(_sz)]),
    ("heic_b200_rbsp_read_ue", i32, [C.c_char_p, _sz, C.POINTER(_sz), C.POINTER(u32)]),
    ("heic_b200_rbsp_read_se", i32, [C.c_char_p, _sz, C.POINTER(_sz), C.POINTER(i32)]),
    ("heic_b200_parse_sps", i32, [C.c_char_p, _sz, C.POINTER(Sps)]),
    ("heic_b200_parse_pps", i32, [C.c_char_p, _sz, C.POINTER(Pps)]),
    ("heic_b200_parse_slice_header", i32,
     [C.c_char_p, _sz, u32, C.POINTER(Sps), C.POINTER(Pps), C.POINTER(u32), _sz, C.POINTER(SliceHeader)]),
    ("heic_b200_parse_slice_header_raw", i32,
     [C.c_char_p, _sz, u32, C.POINTER(Sps), C.POINTER(Pps), C.POINTER(SliceHeader)]),
    ("heic_b200_file_open", i32, [C.c_char_p, _sz, C.POINTER(_vp)]),
    ("heic_b200_file_close", None, [_vp]),
    ("heic_b200_file_primary_image", C.POINTER(ImageDesc), [_vp]),
    ("heic_b200_file_aux_image_count", u32, [_vp]),
    ("heic_b200_file_aux_image", C.POINTER(ImageDesc), [_vp, u32]),
    ("heic_b200_file_primary_image_raw", C.POINTER(ImageDesc), [_vp]),
    ("heic_b200_file_aux_image_raw", C.POINTER(ImageDesc), [_vp, u32]),
    ("heic_b200_file_parameter_set_nal", i32, [_vp, i32, u32, C.POINTER(C.POINTER(u8)), C.POINTER(_sz)]),
    ("heic_b200_file_tile_nal", i32, [_vp, i32, u32, C.POINTER(C.POINTER(u8)), C.POINTER(_sz)]),
    ("heic_b200_file_info", i32, [_vp, C.POINTER(FileInfo)]),
    ("heic_b200_file_image_transform", i32, [_vp, i32, C.POINTER(ImageTransform)]),
    ("heic_b200_unescape", i32,
     [_vp, C.c_char_p, _sz, u32, C.POINTER(u32), u32, C.POINTER(u8), C.POINTER(_sz), C.POINTER(u32), C.POINTER(u32)]),
    ("heic_b200_decode_grids", i32,
     [_vp, C.POINTER(ImageDesc), u32, _vp, _sz, _sz, i32, C.POINTER(TileStatus)]),
    ("heic_b200_decode_grids_submit", i32,
     [_vp, C.POINTER(ImageDesc), u32, _vp, _sz, _sz, i32, C.POINTER(TileStatus), C.POINTER(_vp)]),
    ("heic_b200_job_wait", i32, [_vp]),
    ("heic_b200_decode_grids_transformed", i32,
     [_vp, C.POINTER(ImageDesc), C.POINTER(ImageTransform), u32, _vp, _sz, _sz, C.POINTER(TileStatus)]),
    ("heic_b200_decode_grids_submit_transformed", i32,
     [_vp, C.POINTER(ImageDesc), C.POINTER(ImageTransform), u32, _vp, _sz, _sz, C.POINTER(TileStatus), C.POINTER(_vp)]),
    ("heic_b200_decode_grids_reduced", i32,
     [_vp, C.POINTER(ImageDesc), C.POINTER(ImageTransform), C.POINTER(u32), u32, _vp, _sz, _sz, C.POINTER(TileStatus)]),
    ("heic_b200_decode_grids_submit_reduced", i32,
     [_vp, C.POINTER(ImageDesc), C.POINTER(ImageTransform), C.POINTER(u32), u32, _vp, _sz, _sz, C.POINTER(TileStatus),
      C.POINTER(_vp)]),
    ("heic_b200_decode_grids_yuv", i32,
     [_vp, C.POINTER(ImageDesc), u32, _vp, _vp, _vp, C.POINTER(TileStatus)]),
    ("heic_b200_decode_file", i32, [_vp, C.c_char_p, _sz, _vp, _sz, i32]),
    ("heic_b200_batch_create", i32, [_vp, C.POINTER(ImageDesc), u32, C.POINTER(_vp)]),
    ("heic_b200_batch_create_ex", i32, [_vp, C.POINTER(ImageDesc), u32, i32, C.POINTER(_vp)]),
    ("heic_b200_batch_create_transformed", i32, [_vp, C.POINTER(ImageDesc), C.POINTER(ImageTransform), u32, C.POINTER(_vp)]),
    ("heic_b200_batch_create_reduced", i32,
     [_vp, C.POINTER(ImageDesc), C.POINTER(ImageTransform), C.POINTER(u32), u32, C.POINTER(_vp)]),
    ("heic_b200_batch_destroy", None, [_vp]),
    ("heic_b200_batch_decode", i32, [_vp]),
    ("heic_b200_batch_run_stages", i32, [_vp, u32]),
    ("heic_b200_batch_sync", i32, [_vp]),
    ("heic_b200_batch_stream", _vp, [_vp]),
    ("heic_b200_batch_rgb", i32, [_vp, C.POINTER(_vp), C.POINTER(_sz), C.POINTER(_sz)]),
    ("heic_b200_batch_download_rgb", i32, [_vp, _vp, _sz, _sz]),
    ("heic_b200_batch_download_image", i32, [_vp, u32, _vp, _sz]),
    ("heic_b200_batch_status", i32, [_vp, C.POINTER(TileStatus)]),
    ("heic_b200_batch_tile_count", u32, [_vp]),
    ("heic_b200_batch_cabac_order", _sz, [_vp, C.POINTER(u32), _sz, C.POINTER(u32)]),
    ("heic_b200_batch_dump_tile", i32, [_vp, u32, C.POINTER(TileDump)]),
    ("heic_b200_color_stitch", i32,
     [_vp, _vp, u32, u32, u32, u32, u32, u32, u32, u32, u32, _vp, _sz, _sz]),
]

_lib = None


def load(path: str | None = None, host_only: bool = False) -> C.CDLL:
    """dlopen the C-ABI library and bind every declared symbol.  Raises if absent (no fallback).
    host_only (bench.py's CPU arm): `path` is a build of the host parse layer alone (oracle/_build/libheic_host.so); it
    becomes the process-wide library and only the symbols it has are bound -- every compute entry point is then absent."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise ImportError(
            f"{p} not found: the CUDA library is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(needs nvcc). heif_b200 has no CPU fallback."
        )
    lib = C.CDLL(p)
    for name, restype, argtypes in SYMBOLS:
        if host_only and not hasattr(lib, name):
            continue
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    if path is None or host_only:
        _lib = lib
    return lib


class HeicError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"heic_b200 error {code}: {msg}")
        self.code = code
        self.msg = msg


def check(code: int) -> int:
    if code < 0:
        raise HeicError(code, load().heic_b200_last_error().decode("utf-8", "replace"))
    return code
