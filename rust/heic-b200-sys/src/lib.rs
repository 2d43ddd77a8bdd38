//! SOURCE ONLY (never compiled here: no Rust toolchain in the build image).  `extern "C"` declarations for every entry
//! point of `include/heic_b200.h` (tests/test_capi_exports.py checks this list against the header), plus the safe
//! wrappers that replace the tile loop of `HeicDecoder::decode` (src/heic/decoder.rs:98-119) and
//! `SliceSegmentReader::read_data` (src/hevc/slice.rs:206).  Struct layouts are those of the header, one named field per member (generated from it), and
//! `convert::to_ffi_{sps,pps,slice_header}` copy the reference's parsed structures into them (INTEGRATION.md section 2).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

// heic_status
pub const HEIC_OK: i32 = 0;
pub const HEIC_E_INVALID_ARG: i32 = -1;
pub const HEIC_E_UNSUPPORTED: i32 = -2;
pub const HEIC_E_BITSTREAM: i32 = -3;
pub const HEIC_E_NO_DEVICE: i32 = -4;
pub const HEIC_E_CUDA: i32 = -5;
pub const HEIC_E_NOMEM: i32 = -6;
// stage mask of heic_b200_batch_run_stages
pub const HEIC_STAGE_CABAC: u32 = 1;
pub const HEIC_STAGE_TRANSFORM: u32 = 2;
pub const HEIC_STAGE_INTRA: u32 = 4;
pub const HEIC_STAGE_DEBLOCK: u32 = 8;
pub const HEIC_STAGE_SAO: u32 = 16;
pub const HEIC_STAGE_COLOR: u32 = 32;
pub const HEIC_STAGE_ALL: u32 = 63;

pub const HEIC_MAX_ENTRY_POINTS: usize = 255;

pub const HEIC_RESAMPLE_LANCZOS: u32 = 1;
pub const HEIC_RESAMPLE_BILINEAR: u32 = 2;
pub const HEIC_RESAMPLE_BICUBIC: u32 = 3;
pub const HEIC_RESAMPLE_BOX: u32 = 4;
pub const HEIC_RESAMPLE_HAMMING: u32 = 5;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct heic_scaling_list {
    pub list: [[[u8; 64]; 6]; 4],
    pub dc: [[u8; 6]; 2],
}

/// Mirrors `SequenceParameterSet` (src/hevc/grammar.rs:388-428), one named 32-bit field per member, in the order of
/// include/heic_b200.h.  `[+]` members of the header are what the reference parses and drops.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct heic_sps {
    pub sps_video_parameter_set_id: u32,
    pub sps_max_sub_layers_minus1: u32,
    pub sps_temporal_id_nesting_flag: u32,
    pub sps_seq_parameter_set_id: u32,
    pub chroma_format_idc: u32,
    pub separate_colour_plane_flag: u32,
    pub pic_width_in_luma_samples: u32,
    pub pic_height_in_luma_samples: u32,
    pub conformance_window_flag: u32,
    pub conf_win_left_offset: u32,
    pub conf_win_right_offset: u32,
    pub conf_win_top_offset: u32,
    pub conf_win_bottom_offset: u32,
    pub bit_depth_luma_minus8: u32,
    pub bit_depth_chroma_minus8: u32,
    pub log2_max_pic_order_cnt_lsb_minus4: u32,
    pub log2_min_luma_coding_block_size_minus3: u32,
    pub log2_diff_max_min_luma_coding_block_size: u32,
    pub log2_min_luma_transform_block_size_minus2: u32,
    pub log2_diff_max_min_luma_transform_block_size: u32,
    pub max_transform_hierarchy_depth_inter: u32,
    pub max_transform_hierarchy_depth_intra: u32,
    pub scaling_list_enabled_flag: u32,
    pub sps_scaling_list_data_present_flag: u32,
    pub amp_enabled_flag: u32,
    pub sample_adaptive_offset_enabled_flag: u32,
    pub pcm_enabled_flag: u32,
    pub pcm_sample_bit_depth_luma_minus1: u32,
    pub pcm_sample_bit_depth_chroma_minus1: u32,
    pub log2_min_pcm_luma_coding_block_size_minus3: u32,
    pub log2_diff_max_min_pcm_luma_coding_block_size: u32,
    pub pcm_loop_filter_disabled_flag: u32,
    pub num_short_term_ref_pic_sets: u32,
    pub long_term_ref_pics_present_flag: u32,
    pub sps_temporal_mvp_enabled_flag: u32,
    pub strong_intra_smoothing_enabled_flag: u32,
    pub vui_parameters_present_flag: u32,
    pub video_full_range_flag: u32,
    pub colour_primaries: u32,
    pub transfer_characteristics: u32,
    pub matrix_coeffs: u32,
    pub scaling_list: heic_scaling_list,
}

/// Mirrors `PictureParameterSet` (src/hevc/grammar.rs:511-548).
#[repr(C)]
#[derive(Clone, Copy)]
pub struct heic_pps {
    pub pps_pic_parameter_set_id: u32,
    pub pps_seq_parameter_set_id: u32,
    pub dependent_slice_segments_enabled_flag: u32,
    pub output_flag_present_flag: u32,
    pub num_extra_slice_header_bits: u32,
    pub sign_data_hiding_enabled_flag: u32,
    pub cabac_init_present_flag: u32,
    pub num_ref_idx_l0_default_active_minus1: u32,
    pub num_ref_idx_l1_default_active_minus1: u32,
    pub init_qp_minus26: i32,
    pub constrained_intra_pred_flag: u32,
    pub transform_skip_enabled_flag: u32,
    pub cu_qp_delta_enabled_flag: u32,
    pub diff_cu_qp_delta_depth: u32,
    pub pps_cb_qp_offset: i32,
    pub pps_cr_qp_offset: i32,
    pub pps_slice_chroma_qp_offsets_present_flag: u32,
    pub weighted_pred_flag: u32,
    pub weighted_bipred_flag: u32,
    pub transquant_bypass_enabled_flag: u32,
    pub tiles_enabled_flag: u32,
    pub entropy_coding_sync_enabled_flag: u32,
    pub num_tile_columns_minus1: u32,
    pub num_tile_rows_minus1: u32,
    pub uniform_spacing_flag: u32,
    pub loop_filter_across_tiles_enabled_flag: u32,
    pub pps_loop_filter_across_slices_enabled_flag: u32,
    pub deblocking_filter_control_present_flag: u32,
    pub deblocking_filter_override_enabled_flag: u32,
    pub pps_deblocking_filter_disabled_flag: u32,
    pub pps_beta_offset_div2: i32,
    pub pps_tc_offset_div2: i32,
    pub pps_scaling_list_data_present_flag: u32,
    pub lists_modification_present_flag: u32,
    pub log2_parallel_merge_level_minus2: u32,
    pub slice_segment_header_extension_present_flag: u32,
    pub scaling_list: heic_scaling_list,
}

/// Mirrors `SliceSegmentHeader` (src/hevc/grammar.rs:551-572) + the un-escaped substream offsets.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct heic_slice_header {
    pub first_slice_segment_in_pic_flag: u32,
    pub no_output_of_prior_pics_flag: u32,
    pub slice_pic_parameter_set_id: u32,
    pub slice_type: u32,
    pub slice_sao_luma_flag: u32,
    pub slice_sao_chroma_flag: u32,
    pub slice_qp_delta: i32,
    pub slice_cb_qp_offset: i32,
    pub slice_cr_qp_offset: i32,
    pub deblocking_filter_override_flag: u32,
    pub slice_deblocking_filter_disabled_flag: u32,
    pub slice_beta_offset_div2: i32,
    pub slice_tc_offset_div2: i32,
    pub slice_loop_filter_across_slices_enabled_flag: u32,
    pub num_entry_point_offsets: u32,
    pub entry_point_offset_minus1: [u32; HEIC_MAX_ENTRY_POINTS],
    pub slice_data_byte_offset: u32,
    pub substream_offset: [u32; HEIC_MAX_ENTRY_POINTS + 1],
}

// ---- field-by-field conversions from the reference's parsed structures (what INTEGRATION.md section 2 calls) ----------
// Written against the crate's own types (`heif::hevc::grammar::*`); the `[+]` members the reference does not keep
// (scaling lists, `video_full_range_flag`, the slice-data offset, un-escaped substream offsets) are filled by the host
// additions INTEGRATION.md lists, passed in here as plain arguments.
#[cfg(feature = "heif")]
pub mod convert {
    use super::*;
    use heif::hevc::grammar::{PictureParameterSet, SequenceParameterSet, SliceSegmentHeader};

    const ZERO_LISTS: heic_scaling_list = heic_scaling_list { list: [[[0; 64]; 6]; 4], dc: [[0; 6]; 2] };

    /// `lists`: Some(..) when `sps_scaling_list_data_present_flag` (parameter_set_reader.rs:97-103 parses and drops them).
    pub fn to_ffi_sps(s: &SequenceParameterSet, video_full_range_flag: bool, lists: Option<heic_scaling_list>) -> heic_sps {
        heic_sps {
            sps_video_parameter_set_id: s.sps_video_parameter_set_id as u32,
            sps_max_sub_layers_minus1: s.sps_max_sub_layers_minus1 as u32,
            sps_temporal_id_nesting_flag: s.sps_temporal_id_nesting_flag as u32,
            sps_seq_parameter_set_id: s.sps_seq_parameter_set_id,
            chroma_format_idc: s.chroma_format as u32,
            separate_colour_plane_flag: s.separate_color_plane_flag as u32,
            pic_width_in_luma_samples: s.pic_width_in_luma_samples,
            pic_height_in_luma_samples: s.pic_height_in_luma_samples,
            conformance_window_flag: s.conformance_window_flag as u32,
            conf_win_left_offset: s.conf_win_left_offset,
            conf_win_right_offset: s.conf_win_right_offset,
            conf_win_top_offset: s.conf_win_top_offset,
            conf_win_bottom_offset: s.conf_win_bottom_offset,
            bit_depth_luma_minus8: s.bit_depth_luma_minus8,
            bit_depth_chroma_minus8: s.bit_depth_chroma_minus8,
            log2_max_pic_order_cnt_lsb_minus4: s.log2_max_pic_order_cnt_lsb_minus4,
            log2_min_luma_coding_block_size_minus3: s.log2_min_luma_coding_block_size_minus3,
            log2_diff_max_min_luma_coding_block_size: s.log2_diff_max_min_luma_coding_block_size,
            log2_min_luma_transform_block_size_minus2: s.log2_min_luma_transform_block_size_minus2,
            log2_diff_max_min_luma_transform_block_size: s.log2_diff_max_min_luma_transform_block_size,
            max_transform_hierarchy_depth_inter: s.max_transform_hierarchy_depth_inter,
            max_transform_hierarchy_depth_intra: s.max_transform_hierarchy_depth_intra,
            scaling_list_enabled_flag: s.scaling_list_enabled_flag as u32,
            sps_scaling_list_data_present_flag: lists.is_some() as u32,
            amp_enabled_flag: s.amp_enabled_flag as u32,
            sample_adaptive_offset_enabled_flag: s.sample_adaptive_offset_enabled_flag as u32,
            pcm_enabled_flag: s.pcm_enabled_flag as u32,
            pcm_sample_bit_depth_luma_minus1: s.pcm_sample_bit_depth_luma_minus1.unwrap_or(0) as u32,
            pcm_sample_bit_depth_chroma_minus1: s.pcm_sample_bit_depth_chroma_minus1.unwrap_or(0) as u32,
            log2_min_pcm_luma_coding_block_size_minus3: s.log2_min_pcm_luma_coding_block_size_minus3.unwrap_or(0),
            log2_diff_max_min_pcm_luma_coding_block_size: s.log2_diff_max_min_pcm_luma_coding_block_size.unwrap_or(0),
            pcm_loop_filter_disabled_flag: s.pcm_loop_filter_disabled_flag.unwrap_or(false) as u32,
            num_short_term_ref_pic_sets: s.num_short_term_ref_pic_sets,
            long_term_ref_pics_present_flag: s.long_term_ref_pics_present_flag as u32,
            sps_temporal_mvp_enabled_flag: s.sps_temporal_mvp_enabled_flag as u32,
            strong_intra_smoothing_enabled_flag: s.strong_intra_smoothing_enabled_flag as u32,
            vui_parameters_present_flag: s.vui_parameters_present_flag as u32,
            video_full_range_flag: video_full_range_flag as u32,
            colour_primaries: s.color_primaries.map(|v| v as u32).unwrap_or(2),
            transfer_characteristics: s.transfer_characteristics.map(|v| v as u32).unwrap_or(2),
            matrix_coeffs: s.matrix_coeffs.map(|v| v as u32).unwrap_or(2),
            scaling_list: lists.unwrap_or(ZERO_LISTS),
        }
    }

    /// `lists`: Some(..) when `pps_scaling_list_data_present_flag` (parameter_set_reader.rs:442-445 parses and drops them).
    pub fn to_ffi_pps(p: &PictureParameterSet, lists: Option<heic_scaling_list>) -> heic_pps {
        heic_pps {
            pps_pic_parameter_set_id: p.pps_pic_parameter_set_id,
            pps_seq_parameter_set_id: p.pps_seq_parameter_set_id,
            dependent_slice_segments_enabled_flag: p.dependent_slice_segments_enabled_flag as u32,
            output_flag_present_flag: p.output_flag_present_flag as u32,
            num_extra_slice_header_bits: p.num_extra_slice_header_bits as u32,
            sign_data_hiding_enabled_flag: p.sign_data_hiding_enabled_flag as u32,
            cabac_init_present_flag: p.cabac_init_present_flag as u32,
            num_ref_idx_l0_default_active_minus1: p.num_ref_idx_l0_default_active_minus1,
            num_ref_idx_l1_default_active_minus1: p.num_ref_idx_l1_default_active_minus1,
            init_qp_minus26: p.init_qp_minus26,
            constrained_intra_pred_flag: p.constrained_intra_pred_flag as u32,
            transform_skip_enabled_flag: p.transform_skip_enabled_flag as u32,
            cu_qp_delta_enabled_flag: p.cu_qp_delta_enabled_flag as u32,
            diff_cu_qp_delta_depth: p.diff_cu_qp_delta_depth.unwrap_or(0),
            pps_cb_qp_offset: p.pps_cb_qp_offset,
            pps_cr_qp_offset: p.pps_cr_qp_offset,
            pps_slice_chroma_qp_offsets_present_flag: p.pps_slice_chroma_qp_offsets_present_flag as u32,
            weighted_pred_flag: p.weighted_pred_flag as u32,
            weighted_bipred_flag: p.weighted_bipred_flag as u32,
            transquant_bypass_enabled_flag: p.transquant_bypass_enabled_flag as u32,
            tiles_enabled_flag: p.tiles_enabled_flag as u32,
            entropy_coding_sync_enabled_flag: p.entropy_coding_sync_enabled_flag as u32,
            num_tile_columns_minus1: p.num_tile_columns_minus1.unwrap_or(0),
            num_tile_rows_minus1: p.num_tile_rows_minus1.unwrap_or(0),
            uniform_spacing_flag: p.uniform_spacing_flag.unwrap_or(false) as u32,
            loop_filter_across_tiles_enabled_flag: p.loop_filter_across_tiles_enabled_flag.unwrap_or(false) as u32,
            pps_loop_filter_across_slices_enabled_flag: p.pps_loop_filter_across_slices_enabled_flag as u32,
            deblocking_filter_control_present_flag: p.deblocking_filter_control_present_flag as u32,
            deblocking_filter_override_enabled_flag: p.deblocking_filter_override_enabled_flag.unwrap_or(false) as u32,
            pps_deblocking_filter_disabled_flag: p.pps_deblocking_filter_disabled_flag.unwrap_or(false) as u32,
            pps_beta_offset_div2: p.pps_beta_offset_div2.unwrap_or(0),
            pps_tc_offset_div2: p.pps_tc_offset_div2.unwrap_or(0),
            pps_scaling_list_data_present_flag: lists.is_some() as u32,
            lists_modification_present_flag: p.lists_modification_present_flag as u32,
            log2_parallel_merge_level_minus2: p.log2_parallel_merge_level_minus2,
            slice_segment_header_extension_present_flag: p.slice_segment_header_extension_present_flag as u32,
            scaling_list: lists.unwrap_or(ZERO_LISTS),
        }
    }

    /// `slice_data_byte_offset`: RbspReader::byte_position() after `byte_alignment` (rbsp_reader.rs:65; unreachable in the
    /// reference once slice.rs:29-33 has moved the reader), counted in the un-escaped RBSP.  `epb`: ascending positions, in
    /// the ESCAPED payload, of the emulation prevention bytes `remove_emulation_prevention` dropped; they re-base the raw
    /// entry points (7.4.7.1 counts escaped bytes; slice.rs:155-171 keeps them raw) to un-escaped substream offsets.  Same
    /// arithmetic as `slice_segment_header` in heif_b200/csrc/host/hevc_parse.cc.
    pub fn to_ffi_slice_header(h: &SliceSegmentHeader, pps: &PictureParameterSet, slice_data_byte_offset: u32, epb: &[u32]) -> heic_slice_header {
        let mut o = heic_slice_header {
            first_slice_segment_in_pic_flag: h.first_slice_segment_in_pic_flag as u32,
            no_output_of_prior_pics_flag: h.no_output_of_prior_pics_flag.unwrap_or(false) as u32,
            slice_pic_parameter_set_id: h.slice_pic_parameter_set_id,
            slice_type: h.slice_type as u32,
            slice_sao_luma_flag: h.slice_sao_luma_flag as u32,
            slice_sao_chroma_flag: h.slice_sao_chroma_flag as u32,
            slice_qp_delta: h.slice_qp_delta,
            slice_cb_qp_offset: h.slice_cb_qp_offset.unwrap_or(0),
            slice_cr_qp_offset: h.slice_cr_qp_offset.unwrap_or(0),
            deblocking_filter_override_flag: h.deblocking_filter_override_flag.unwrap_or(false) as u32,
            slice_deblocking_filter_disabled_flag: h
                .slice_deblocking_filter_disabled_flag
                .unwrap_or(pps.pps_deblocking_filter_disabled_flag.unwrap_or(false)) as u32,
            slice_beta_offset_div2: h.slice_beta_offset_div2.unwrap_or(pps.pps_beta_offset_div2.unwrap_or(0)),
            slice_tc_offset_div2: h.slice_tc_offset_div2.unwrap_or(pps.pps_tc_offset_div2.unwrap_or(0)),
            slice_loop_filter_across_slices_enabled_flag: h
                .slice_loop_filter_across_slices_enabled_flag
                .unwrap_or(pps.pps_loop_filter_across_slices_enabled_flag) as u32,
            num_entry_point_offsets: h.num_entry_point_offsets,
            entry_point_offset_minus1: [0; HEIC_MAX_ENTRY_POINTS],
            slice_data_byte_offset,
            substream_offset: [0; HEIC_MAX_ENTRY_POINTS + 1],
        };
        // escaped position of the slice data start: every dropped byte at or before it shifts it up by one
        let mut boundary = slice_data_byte_offset as u64;
        for &p in epb {
            if (p as u64) <= boundary { boundary += 1 } else { break }
        }
        let n = (h.num_entry_point_offsets as usize).min(HEIC_MAX_ENTRY_POINTS);
        for k in 0..n {
            o.entry_point_offset_minus1[k] = h.entry_point_offsets[k];
            boundary += h.entry_point_offsets[k] as u64 + 1;  // escaped position where substream k + 1 starts
            let removed = epb.partition_point(|&p| (p as u64) < boundary) as u64;
            o.substream_offset[k + 1] = (boundary - removed - slice_data_byte_offset as u64) as u32;
        }
        o
    }
}

#[repr(C)]
pub struct heic_tile_desc {
    pub rbsp: *const u8,
    pub rbsp_len: u32,
    pub nal_unit_type: u32,
    /// 0: `rbsp` is un-escaped; 1: raw NAL payload, offsets in raw byte counts (un-escaped on the GPU)
    pub escaped: u32,
    pub header: heic_slice_header,
}

#[repr(C)]
pub struct heic_image_desc {
    pub sps: heic_sps,
    pub pps: heic_pps,
    pub grid_rows: u32,
    pub grid_cols: u32,
    pub output_width: u32,
    pub output_height: u32,
    pub rotation_ccw_quarter_turns: u32,
    pub n_tiles: u32,
    pub tiles: *const heic_tile_desc,
}

/// Output geometry of one image: the crop of the canvas, then `orientation & 3` anticlockwise quarter turns, then a
/// left<->right mirror when `orientation & 4`.
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct heic_image_transform {
    pub crop_x: u32,
    pub crop_y: u32,
    pub crop_w: u32,
    pub crop_h: u32,
    pub orientation: u32,
}

/// Output size and filter (`HEIC_RESAMPLE_*`) of a resize; all zero: no resize.
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct heic_resize {
    pub width: u32,
    pub height: u32,
    pub filter: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct heic_tile_status {
    pub code: i32,
    pub bins_decoded: u32,
    pub ctus_decoded: u32,
    pub reserved: u32,
}

/// Container metadata the reference's integration test pins (tests/libheif_comparison.rs:102-111).
#[repr(C)]
#[derive(Clone, Copy, Default)]
pub struct heic_file_info {
    pub primary_item_id: u32,
    pub ispe_width: u32,
    pub ispe_height: u32,
    pub rotation_ccw_quarter_turns: u32,
    pub rotated_width: u32,
    pub rotated_height: u32,
    pub luma_bits: u32,
    pub chroma_bits: u32,
    pub thumbnail_count: u32,
    pub item_count: u32,
    pub is_grid: u32,
}

/// Host copies of one tile's intermediate buffers (per-stage parity tests); any pointer may be null.
#[repr(C)]
pub struct heic_tile_dump {
    pub tu_map: *mut u32,
    pub tu_map_len: u32,
    pub coeff: [*mut i16; 3],
    pub coeff_len: [u32; 3],
    pub qp_map: *mut u8,
    pub qp_map_len: u32,
    pub sao: *mut u32,
    pub sao_len: u32,
    pub plane: [*mut u8; 3],
    pub plane_len: [u32; 3],
}

#[repr(C)]
pub struct heic_b200_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct heic_b200_file {
    _private: [u8; 0],
}
#[repr(C)]
pub struct heic_b200_job {
    _private: [u8; 0],
}
#[repr(C)]
pub struct heic_b200_batch {
    _private: [u8; 0],
}

extern "C" {
    pub fn heic_b200_abi_version() -> i32;
    pub fn heic_b200_last_error() -> *const c_char;
    pub fn heic_b200_create(device: i32, out_ctx: *mut *mut heic_b200_ctx) -> i32;
    pub fn heic_b200_destroy(ctx: *mut heic_b200_ctx);
    pub fn heic_b200_launch_count(ctx: *const heic_b200_ctx) -> u64;
    // ---- host-side restatement of the reference's parse layer ----
    pub fn heic_b200_remove_emulation_prevention(
        data: *const u8, len: usize, out: *mut u8, epb_pos: *mut u32, epb_cap: usize, n_epb: *mut usize,
    ) -> i64;
    pub fn heic_b200_rbsp_read_ue(data: *const u8, len: usize, bit_pos: *mut usize, out: *mut u32) -> i32;
    pub fn heic_b200_rbsp_read_se(data: *const u8, len: usize, bit_pos: *mut usize, out: *mut i32) -> i32;
    pub fn heic_b200_parse_sps(rbsp: *const u8, len: usize, out: *mut heic_sps) -> i32;
    pub fn heic_b200_parse_pps(rbsp: *const u8, len: usize, out: *mut heic_pps) -> i32;
    pub fn heic_b200_parse_slice_header(
        rbsp: *const u8, len: usize, nal_unit_type: u32, sps: *const heic_sps, pps: *const heic_pps,
        epb_pos: *const u32, n_epb: usize, out: *mut heic_slice_header,
    ) -> i32;
    pub fn heic_b200_parse_slice_header_raw(
        nal_payload: *const u8, len: usize, nal_unit_type: u32, sps: *const heic_sps, pps: *const heic_pps,
        out: *mut heic_slice_header,
    ) -> i32;
    // ---- HeifReader / HeicDecoder item walk ----
    pub fn heic_b200_file_open(data: *const u8, len: usize, out: *mut *mut heic_b200_file) -> i32;
    pub fn heic_b200_file_close(f: *mut heic_b200_file);
    pub fn heic_b200_file_primary_image(f: *const heic_b200_file) -> *const heic_image_desc;
    pub fn heic_b200_file_aux_image_count(f: *const heic_b200_file) -> u32;
    pub fn heic_b200_file_aux_image(f: *const heic_b200_file, i: u32) -> *const heic_image_desc;
    pub fn heic_b200_file_primary_image_raw(f: *const heic_b200_file) -> *const heic_image_desc;
    pub fn heic_b200_file_aux_image_raw(f: *const heic_b200_file, i: u32) -> *const heic_image_desc;
    pub fn heic_b200_file_parameter_set_nal(
        f: *const heic_b200_file, image: i32, nal_unit_type: u32, data: *mut *const u8, len: *mut usize,
    ) -> i32;
    pub fn heic_b200_file_tile_nal(
        f: *const heic_b200_file, image: i32, tile: u32, data: *mut *const u8, len: *mut usize,
    ) -> i32;
    pub fn heic_b200_file_info(f: *const heic_b200_file, out: *mut heic_file_info) -> i32;
    pub fn heic_b200_file_image_transform(f: *const heic_b200_file, image: i32, out: *mut heic_image_transform) -> i32;
    // ---- the hot path ----
    pub fn heic_b200_decode_grids(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, n_imgs: u32, rgb_out: *mut u8, pitch: usize,
        image_stride: usize, apply_transforms: c_int, status: *mut heic_tile_status,
    ) -> i32;
    pub fn heic_b200_decode_grids_submit(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, n_imgs: u32, rgb_out: *mut u8, pitch: usize,
        image_stride: usize, apply_transforms: c_int, status: *mut heic_tile_status, out_job: *mut *mut heic_b200_job,
    ) -> i32;
    pub fn heic_b200_job_wait(job: *mut heic_b200_job) -> i32;
    pub fn heic_b200_decode_grids_transformed(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, n_imgs: u32,
        rgb_out: *mut u8, pitch: usize, image_stride: usize, status: *mut heic_tile_status,
    ) -> i32;
    pub fn heic_b200_decode_grids_submit_transformed(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, n_imgs: u32,
        rgb_out: *mut u8, pitch: usize, image_stride: usize, status: *mut heic_tile_status, out_job: *mut *mut heic_b200_job,
    ) -> i32;
    pub fn heic_b200_decode_grids_reduced(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, reduce: *const u32,
        n_imgs: u32, rgb_out: *mut u8, pitch: usize, image_stride: usize, status: *mut heic_tile_status,
    ) -> i32;
    pub fn heic_b200_decode_grids_submit_reduced(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, reduce: *const u32,
        n_imgs: u32, rgb_out: *mut u8, pitch: usize, image_stride: usize, status: *mut heic_tile_status,
        out_job: *mut *mut heic_b200_job,
    ) -> i32;
    pub fn heic_b200_decode_grids_resized(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, reduce: *const u32,
        resize: *const heic_resize, n_imgs: u32, rgb_out: *mut u8, pitch: usize, image_stride: usize,
        status: *mut heic_tile_status,
    ) -> i32;
    pub fn heic_b200_decode_grids_submit_resized(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, reduce: *const u32,
        resize: *const heic_resize, n_imgs: u32, rgb_out: *mut u8, pitch: usize, image_stride: usize,
        status: *mut heic_tile_status, out_job: *mut *mut heic_b200_job,
    ) -> i32;
    pub fn heic_b200_resample_coeffs(
        n_in: u32, n_out: u32, filter: u32, bounds: *mut i32, coeffs: *mut i32, coeffs_cap: usize,
    ) -> i64;
    pub fn heic_b200_decode_grids_yuv(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, n_imgs: u32, y_out: *mut u8, cb_out: *mut u8,
        cr_out: *mut u8, status: *mut heic_tile_status,
    ) -> i32;
    pub fn heic_b200_decode_file(
        ctx: *mut heic_b200_ctx, data: *const u8, len: usize, rgb_out: *mut u8, pitch: usize, apply_transforms: c_int,
    ) -> i32;
    // ---- resident batches ----
    pub fn heic_b200_batch_create(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, n_imgs: u32, out: *mut *mut heic_b200_batch,
    ) -> i32;
    pub fn heic_b200_batch_create_ex(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, n_imgs: u32, apply_transforms: i32, out: *mut *mut heic_b200_batch,
    ) -> i32;
    pub fn heic_b200_batch_create_transformed(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, n_imgs: u32,
        out: *mut *mut heic_b200_batch,
    ) -> i32;
    pub fn heic_b200_batch_create_reduced(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, reduce: *const u32,
        n_imgs: u32, out: *mut *mut heic_b200_batch,
    ) -> i32;
    pub fn heic_b200_batch_create_resized(
        ctx: *mut heic_b200_ctx, imgs: *const heic_image_desc, xforms: *const heic_image_transform, reduce: *const u32,
        resize: *const heic_resize, n_imgs: u32, out: *mut *mut heic_b200_batch,
    ) -> i32;
    pub fn heic_b200_batch_destroy(b: *mut heic_b200_batch);
    pub fn heic_b200_batch_decode(b: *mut heic_b200_batch) -> i32;
    pub fn heic_b200_batch_run_stages(b: *mut heic_b200_batch, stage_mask: u32) -> i32;
    pub fn heic_b200_batch_sync(b: *mut heic_b200_batch) -> i32;
    pub fn heic_b200_batch_stream(b: *mut heic_b200_batch) -> *mut c_void;
    pub fn heic_b200_batch_rgb(
        b: *mut heic_b200_batch, dev_ptr: *mut *mut c_void, pitch: *mut usize, image_stride: *mut usize,
    ) -> i32;
    pub fn heic_b200_batch_download_rgb(b: *mut heic_b200_batch, rgb_out: *mut u8, pitch: usize, image_stride: usize) -> i32;
    pub fn heic_b200_batch_status(b: *mut heic_b200_batch, status: *mut heic_tile_status) -> i32;
    pub fn heic_b200_batch_download_image(b: *mut heic_b200_batch, image_index: u32, rgb_out: *mut u8, pitch: usize) -> i32;
    pub fn heic_b200_batch_tile_count(b: *const heic_b200_batch) -> u32;
    pub fn heic_b200_batch_cabac_order(b: *const heic_b200_batch, out: *mut u32, cap: usize, tiles_per_group: *mut u32) -> usize;
    pub fn heic_b200_batch_dump_tile(b: *mut heic_b200_batch, tile_index: u32, dump: *mut heic_tile_dump) -> i32;
    // ---- stand-alone stages on caller-owned buffers ----
    pub fn heic_b200_unescape(
        ctx: *mut heic_b200_ctx, nal_payload: *const u8, len: usize, slice_data_byte_offset: u32,
        substream_offset: *const u32, n_substreams: u32, rbsp_out: *mut u8, rbsp_len: *mut usize,
        slice_data_byte_offset_out: *mut u32, substream_offset_out: *mut u32,
    ) -> i32;
    pub fn heic_b200_color_stitch(
        ctx: *mut heic_b200_ctx, dev_planes: *const c_void, n_images: u32, grid_rows: u32, grid_cols: u32, tile_w: u32,
        tile_h: u32, out_w: u32, out_h: u32, full_range: u32, matrix_coeffs: u32, dev_rgb: *mut c_void, pitch: usize,
        image_stride: usize,
    ) -> i32;
}

/// One decoder = one CUDA stream on one device.  Not `Sync`: use one per thread.
pub struct B200Decoder(*mut heic_b200_ctx);

impl B200Decoder {
    pub fn new(device: i32) -> Result<Self, String> {
        let mut ctx = std::ptr::null_mut();
        let rc = unsafe { heic_b200_create(device, &mut ctx) };
        if rc < 0 { Err(last_error()) } else { Ok(Self(ctx)) }
    }

    /// Replacement for the reference's tile loop: all tiles of all images in one call; returns interleaved RGB8.
    pub fn decode_grids(&mut self, imgs: &[heic_image_desc], width: usize, height: usize) -> Result<Vec<u8>, String> {
        let mut rgb = vec![0u8; imgs.len() * width * height * 3];
        let rc = unsafe {
            heic_b200_decode_grids(self.0, imgs.as_ptr(), imgs.len() as u32, rgb.as_mut_ptr(), width * 3,
                                   width * height * 3, 0, std::ptr::null_mut())
        };
        if rc < 0 { Err(last_error()) } else { Ok(rgb) }
    }
}

/// A submitted `decode_grids` call (the asynchronous form, INTEGRATION.md section 4).  The output buffer is owned by the
/// job until `wait` hands it back, so it cannot be read or dropped while the device still writes it.
pub struct B200Job {
    job: *mut heic_b200_job,
    rgb: Vec<u8>,
}

impl B200Job {
    /// Blocks until the RGB of this call is complete and returns it.
    pub fn wait(mut self) -> Result<Vec<u8>, String> {
        let rc = unsafe { heic_b200_job_wait(self.job) };
        self.job = std::ptr::null_mut();
        let rgb = std::mem::take(&mut self.rgb);
        if rc < 0 { Err(last_error()) } else { Ok(rgb) }
    }
}

impl Drop for B200Job {
    fn drop(&mut self) {
        if !self.job.is_null() {
            unsafe { heic_b200_job_wait(self.job) }; // the buffer must outlive the copies
        }
    }
}

impl B200Decoder {
    /// Queues all copies and kernels of one call and returns; submit the next call before waiting for this one to
    /// overlap its host->device copy and kernels with this call's device->host copy.
    pub fn submit_grids(&mut self, imgs: &[heic_image_desc], width: usize, height: usize) -> Result<B200Job, String> {
        let mut rgb = vec![0u8; imgs.len() * width * height * 3];
        let mut job = std::ptr::null_mut();
        let rc = unsafe {
            heic_b200_decode_grids_submit(self.0, imgs.as_ptr(), imgs.len() as u32, rgb.as_mut_ptr(), width * 3,
                                          width * height * 3, 0, std::ptr::null_mut(), &mut job)
        };
        if rc < 0 { Err(last_error()) } else { Ok(B200Job { job, rgb }) }
    }

    /// `HeicDecoder::decode(&[u8])` that returns the image (decoder.rs:12 returns `()`): (width, height, RGB8).
    pub fn decode_file(&mut self, data: &[u8]) -> Result<(u32, u32, Vec<u8>), String> {
        let mut f = std::ptr::null_mut();
        if unsafe { heic_b200_file_open(data.as_ptr(), data.len(), &mut f) } < 0 {
            return Err(last_error());
        }
        let mut info = heic_file_info::default();
        let rc = unsafe { heic_b200_file_info(f, &mut info) };
        unsafe { heic_b200_file_close(f) };
        if rc < 0 {
            return Err(last_error());
        }
        let (w, h) = (info.ispe_width as usize, info.ispe_height as usize);
        let mut rgb = vec![0u8; w * h * 3];
        let rc = unsafe { heic_b200_decode_file(self.0, data.as_ptr(), data.len(), rgb.as_mut_ptr(), w * 3, 0) };
        if rc < 0 { Err(last_error()) } else { Ok((info.ispe_width, info.ispe_height, rgb)) }
    }
}

impl Drop for B200Decoder {
    fn drop(&mut self) {
        unsafe { heic_b200_destroy(self.0) }
    }
}

fn last_error() -> String {
    unsafe { std::ffi::CStr::from_ptr(heic_b200_last_error()).to_string_lossy().into_owned() }
}
