/*
 * heic_b200.h — C ABI of the B200-native HEIC image-reconstruction path.
 *
 * This is the drop-in boundary for friendlymatthew/heif's decode path.  The
 * reference has no FFI of its own; the seam this ABI replaces is
 *
 *     SliceSegmentReader::read_data(&mut self) -> Result<()>     src/hevc/slice.rs:206
 *     called per grid tile from HeicDecoder::decode               src/heic/decoder.rs:114-119
 *
 * i.e. "everything from slice data onward".  The host side (container, VPS/SPS/PPS,
 * slice-segment header) stays on the CPU and hands this library plain-old-data
 * descriptors; the library runs CABAC, dequant + inverse transform, intra
 * prediction, deblocking, SAO and YCbCr->RGB + grid stitch as sm_100a CUDA kernels.
 * There is no CPU fallback: every compute entry point returns HEIC_E_NO_DEVICE when
 * no CUDA device is usable.
 *
 * Conventions: all functions return 0 on success or a negative heic_status code;
 * heic_b200_last_error() returns a thread-local, NUL-terminated description of the last
 * failure on the calling thread.  Nothing unwinds or aborts across this boundary (the
 * reference's todo!/unimplemented!/assert! sites become error codes).  The caller owns
 * every buffer it passes in.  One heic_b200_ctx per host thread / CUDA stream.
 */
#ifndef HEIC_B200_H
#define HEIC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HEIC_B200_ABI_VERSION 1

typedef enum heic_status {
  HEIC_OK = 0,
  HEIC_E_INVALID_ARG = -1,
  HEIC_E_UNSUPPORTED = -2,   /* legal HEVC/HEIF the path does not implement (PCM, tiles, 4:4:4, >8 bit ...) */
  HEIC_E_BITSTREAM = -3,     /* malformed container / parameter set / slice data                          */
  HEIC_E_NO_DEVICE = -4,     /* no CUDA device; this library has no CPU path                              */
  HEIC_E_CUDA = -5,          /* CUDA runtime error (message in heic_b200_last_error)                      */
  HEIC_E_NOMEM = -6,
} heic_status;

/* ------------------------------------------------------------------------------------------------
 * Parameter sets as plain data.
 *   heic_sps mirrors SequenceParameterSet   (reference src/hevc/grammar.rs:388-428)
 *   heic_pps mirrors PictureParameterSet    (reference src/hevc/grammar.rs:511-548)
 *   heic_slice_header mirrors SliceSegmentHeader (reference src/hevc/grammar.rs:551-572)
 * Option<T> fields of the reference are flattened to their inferred values.  Fields the
 * reference parses and drops but the reconstruction needs are added and marked [+].
 * ---------------------------------------------------------------------------------------------- */

typedef struct heic_scaling_list {
  /* ScalingList[sizeId][matrixId][i] in up-right diagonal scan order as coded (7.3.4);
   * sizeId 0: 16 entries used, sizeId 1..3: 64.  sizeId 3 uses matrixId 0 and 3 only. */
  uint8_t list[4][6][64];
  uint8_t dc[2][6];          /* scaling_list_dc_coef_minus8 + 8 for sizeId 2,3 */
} heic_scaling_list;

typedef struct heic_sps {
  uint32_t sps_video_parameter_set_id;
  uint32_t sps_max_sub_layers_minus1;
  uint32_t sps_temporal_id_nesting_flag;
  uint32_t sps_seq_parameter_set_id;
  uint32_t chroma_format_idc;                 /* ChromaFormat */
  uint32_t separate_colour_plane_flag;
  uint32_t pic_width_in_luma_samples;
  uint32_t pic_height_in_luma_samples;
  uint32_t conformance_window_flag;
  uint32_t conf_win_left_offset, conf_win_right_offset, conf_win_top_offset, conf_win_bottom_offset;
  uint32_t bit_depth_luma_minus8, bit_depth_chroma_minus8;
  uint32_t log2_max_pic_order_cnt_lsb_minus4;
  uint32_t log2_min_luma_coding_block_size_minus3;
  uint32_t log2_diff_max_min_luma_coding_block_size;
  uint32_t log2_min_luma_transform_block_size_minus2;
  uint32_t log2_diff_max_min_luma_transform_block_size;
  uint32_t max_transform_hierarchy_depth_inter;
  uint32_t max_transform_hierarchy_depth_intra;
  uint32_t scaling_list_enabled_flag;
  uint32_t sps_scaling_list_data_present_flag; /* [+] */
  uint32_t amp_enabled_flag;
  uint32_t sample_adaptive_offset_enabled_flag;
  uint32_t pcm_enabled_flag;
  uint32_t pcm_sample_bit_depth_luma_minus1, pcm_sample_bit_depth_chroma_minus1;
  uint32_t log2_min_pcm_luma_coding_block_size_minus3, log2_diff_max_min_pcm_luma_coding_block_size;
  uint32_t pcm_loop_filter_disabled_flag;
  uint32_t num_short_term_ref_pic_sets;
  uint32_t long_term_ref_pics_present_flag;
  uint32_t sps_temporal_mvp_enabled_flag;
  uint32_t strong_intra_smoothing_enabled_flag;
  uint32_t vui_parameters_present_flag;
  uint32_t video_full_range_flag;             /* [+] read and dropped at parameter_set_reader.rs:281 */
  uint32_t colour_primaries, transfer_characteristics, matrix_coeffs; /* 2 = unspecified when absent */
  heic_scaling_list scaling_list;             /* [+] valid when sps_scaling_list_data_present_flag */
} heic_sps;

typedef struct heic_pps {
  uint32_t pps_pic_parameter_set_id, pps_seq_parameter_set_id;
  uint32_t dependent_slice_segments_enabled_flag;
  uint32_t output_flag_present_flag;
  uint32_t num_extra_slice_header_bits;
  uint32_t sign_data_hiding_enabled_flag;
  uint32_t cabac_init_present_flag;
  uint32_t num_ref_idx_l0_default_active_minus1, num_ref_idx_l1_default_active_minus1;
  int32_t  init_qp_minus26;
  uint32_t constrained_intra_pred_flag;
  uint32_t transform_skip_enabled_flag;
  uint32_t cu_qp_delta_enabled_flag;
  uint32_t diff_cu_qp_delta_depth;
  int32_t  pps_cb_qp_offset, pps_cr_qp_offset;
  uint32_t pps_slice_chroma_qp_offsets_present_flag;
  uint32_t weighted_pred_flag, weighted_bipred_flag;
  uint32_t transquant_bypass_enabled_flag;
  uint32_t tiles_enabled_flag;
  uint32_t entropy_coding_sync_enabled_flag;
  uint32_t num_tile_columns_minus1, num_tile_rows_minus1, uniform_spacing_flag;
  uint32_t loop_filter_across_tiles_enabled_flag;
  uint32_t pps_loop_filter_across_slices_enabled_flag;
  uint32_t deblocking_filter_control_present_flag;
  uint32_t deblocking_filter_override_enabled_flag;
  uint32_t pps_deblocking_filter_disabled_flag;
  int32_t  pps_beta_offset_div2, pps_tc_offset_div2;
  uint32_t pps_scaling_list_data_present_flag;
  uint32_t lists_modification_present_flag;
  uint32_t log2_parallel_merge_level_minus2;
  uint32_t slice_segment_header_extension_present_flag;
  heic_scaling_list scaling_list;             /* [+] valid when pps_scaling_list_data_present_flag */
} heic_pps;

#define HEIC_MAX_ENTRY_POINTS 255

typedef struct heic_slice_header {
  uint32_t first_slice_segment_in_pic_flag;
  uint32_t no_output_of_prior_pics_flag;
  uint32_t slice_pic_parameter_set_id;
  uint32_t slice_type;                        /* SliceKind: 0 B, 1 P, 2 I; only I is decodable */
  uint32_t slice_sao_luma_flag, slice_sao_chroma_flag;
  int32_t  slice_qp_delta;
  int32_t  slice_cb_qp_offset, slice_cr_qp_offset;
  uint32_t deblocking_filter_override_flag;
  uint32_t slice_deblocking_filter_disabled_flag;
  int32_t  slice_beta_offset_div2, slice_tc_offset_div2;
  uint32_t slice_loop_filter_across_slices_enabled_flag;
  uint32_t num_entry_point_offsets;
  /* entry_point_offset_minus1[i] exactly as coded: byte counts in the ESCAPED NAL
   * (reference keeps them raw at slice.rs:155-171).  */
  uint32_t entry_point_offset_minus1[HEIC_MAX_ENTRY_POINTS];
  /* [+] what the reference cannot expose after slice.rs:29-33 moves the reader: */
  uint32_t slice_data_byte_offset;            /* first byte of slice_segment_data() in the un-escaped RBSP */
  /* [+] substream start offsets in the UN-ESCAPED RBSP, relative to slice_data_byte_offset;
   * substream_offset[0] == 0; n = num_entry_point_offsets + 1 entries are valid. */
  uint32_t substream_offset[HEIC_MAX_ENTRY_POINTS + 1];
} heic_slice_header;

/* One coded picture = one HEIF grid tile (or a single hvc1 item). */
typedef struct heic_tile_desc {
  const uint8_t* rbsp;        /* un-escaped slice-segment RBSP (after the 2-byte NAL header), host memory */
  uint32_t rbsp_len;
  uint32_t nal_unit_type;     /* must be an IRAP type; the reference insists on IDR_N_LP (decoder.rs:109-112) */
  /* [+] 0: `rbsp` is the un-escaped RBSP (what RbspReader::remove_emulation_prevention returns, rbsp_reader.rs:11-39)
   *        and the header's offsets count un-escaped bytes;
   *     1: `rbsp` is the raw NAL payload, emulation prevention bytes still in place, and header.slice_data_byte_offset /
   *        header.substream_offset[] count raw bytes (the way entry_point_offset_minus1 does, 7.4.7.1) — see
   *        heic_b200_parse_slice_header_raw.  The library then removes the emulation prevention bytes and re-bases
   *        the offsets on the GPU, and the host never touches the slice data. */
  uint32_t escaped;
  heic_slice_header header;
} heic_tile_desc;

/* One HEIF image item: a grid of tiles (rows*cols pictures sharing SPS/PPS) or a single picture
 * (rows = cols = 1). */
typedef struct heic_image_desc {
  heic_sps sps;
  heic_pps pps;
  uint32_t grid_rows, grid_cols;
  uint32_t output_width, output_height;  /* grid canvas size before rotation (HEIF 6.6.2.3); crop of the tile mosaic */
  uint32_t rotation_ccw_quarter_turns;   /* irot.angle; applied to the RGB output when apply_transforms != 0 */
  uint32_t n_tiles;                      /* == grid_rows * grid_cols */
  const heic_tile_desc* tiles;           /* row-major */
} heic_image_desc;

/* Output geometry of one image, carried beside its heic_image_desc (whose layout is fixed by the ABI version):
 *   out = canvas[crop_y : crop_y + crop_h, crop_x : crop_x + crop_w], then rotated anticlockwise by
 *   (orientation & 3) quarter turns, then, when orientation & 4, mirrored left <-> right.
 * The canvas is the output_width x output_height grid canvas.  This normal form covers every sequence of the
 * HEIF transformative properties clap, irot and imir (heic_b200_file_image_transform composes them).
 * The identity is {0, 0, output_width, output_height, 0}. */
typedef struct heic_image_transform {
  uint32_t crop_x, crop_y, crop_w, crop_h;  /* canvas coordinates, before the orientation */
  uint32_t orientation;                     /* bits 0-1: ccw quarter turns; bit 2: then mirror left<->right */
} heic_image_transform;

typedef struct heic_tile_status {
  int32_t code;               /* heic_status for this tile; one bad tile does not poison a batch */
  uint32_t bins_decoded;      /* CABAC bins (decision + bypass + terminate) consumed */
  uint32_t ctus_decoded;
  uint32_t reserved;
} heic_tile_status;

typedef struct heic_b200_ctx heic_b200_ctx;

/* ---- library / context -------------------------------------------------------------------- */
int32_t heic_b200_abi_version(void);
const char* heic_b200_last_error(void);
/* device < 0 selects the current CUDA device. */
int32_t heic_b200_create(int32_t device, heic_b200_ctx** out_ctx);
void    heic_b200_destroy(heic_b200_ctx* ctx);
/* Number of kernel launches issued by this context since creation (for launch accounting). */
uint64_t heic_b200_launch_count(const heic_b200_ctx* ctx);

/* ---- host-side restatement of the reference's parse layer (C++ behind a C ABI) ------------- */
/* RbspReader::remove_emulation_prevention                       src/hevc/rbsp_reader.rs:11-39
 * out must hold len bytes; returns the un-escaped length (>= 0).  If epb_pos != NULL it receives up
 * to epb_cap positions (in the escaped input) of every removed 0x03 byte; *n_epb gets the count. */
int64_t heic_b200_remove_emulation_prevention(const uint8_t* data, size_t len, uint8_t* out,
                                              uint32_t* epb_pos, size_t epb_cap, size_t* n_epb);
/* RbspReader::read_ue / read_se                                  src/hevc/rbsp_reader.rs:87,101
 * Reads one Exp-Golomb code starting at bit *bit_pos of data (MSB first) and advances *bit_pos. */
int32_t heic_b200_rbsp_read_ue(const uint8_t* data, size_t len, size_t* bit_pos, uint32_t* out);
int32_t heic_b200_rbsp_read_se(const uint8_t* data, size_t len, size_t* bit_pos, int32_t* out);
/* video/sequence/picture_parameter_set_rbsp                     src/hevc/parameter_set_reader.rs:7,36,351
 * Input is the un-escaped RBSP without the 2-byte NAL header. */
int32_t heic_b200_parse_sps(const uint8_t* rbsp, size_t len, heic_sps* out);
int32_t heic_b200_parse_pps(const uint8_t* rbsp, size_t len, heic_pps* out);
/* SliceSegmentReader::read_header                                src/hevc/slice.rs:44-204
 * rbsp is un-escaped; epb_pos/n_epb (from remove_emulation_prevention, positions relative to the
 * escaped payload after the NAL header) convert entry points to un-escaped substream offsets. */
int32_t heic_b200_parse_slice_header(const uint8_t* rbsp, size_t len, uint32_t nal_unit_type,
                                     const heic_sps* sps, const heic_pps* pps,
                                     const uint32_t* epb_pos, size_t n_epb, heic_slice_header* out);
/* [+] The same header read straight from a raw NAL payload (emulation prevention bytes in place; only the first
 * bytes are un-escaped, the slice data is not touched): slice_data_byte_offset is the raw position of
 * slice_segment_data() and substream_offset[k] the running sum of entry_point_offset_minus1 + 1, i.e. raw byte counts.
 * For heic_tile_desc::escaped = 1. */
int32_t heic_b200_parse_slice_header_raw(const uint8_t* nal_payload, size_t len, uint32_t nal_unit_type,
                                         const heic_sps* sps, const heic_pps* pps, heic_slice_header* out);

/* HeifReader::{new, read, get_item_data} + HeicDecoder::decode's item walk
 *                                                               src/heif/reader.rs:25,59,33; src/heic/decoder.rs:12-112
 * Parses a HEIC file and builds the image descriptor of the primary item (grid or single hvc1).
 * The returned handle owns all storage the descriptor points into. */
typedef struct heic_b200_file heic_b200_file;
int32_t heic_b200_file_open(const uint8_t* data, size_t len, heic_b200_file** out);
void    heic_b200_file_close(heic_b200_file* f);
const heic_image_desc* heic_b200_file_primary_image(const heic_b200_file* f);
/* Auxiliary images (e.g. the Apple HDR gain map, `auxl` reference to the primary item). */
uint32_t heic_b200_file_aux_image_count(const heic_b200_file* f);
const heic_image_desc* heic_b200_file_aux_image(const heic_b200_file* f, uint32_t i);
/* The same images with raw tile payloads (heic_tile_desc::escaped = 1): the bytes of the NAL units as they lie in
 * `mdat`, minus the 2-byte NAL header. */
const heic_image_desc* heic_b200_file_primary_image_raw(const heic_b200_file* f);
const heic_image_desc* heic_b200_file_aux_image_raw(const heic_b200_file* f, uint32_t i);
/* Escaped NAL units (2-byte header included) as stored in the file, e.g. to feed an external decoder.
 * image = -1 selects the primary image, >= 0 an auxiliary image.  nal_unit_type: 32 VPS, 33 SPS, 34 PPS.
 * The pointers stay valid until heic_b200_file_close. */
int32_t heic_b200_file_parameter_set_nal(const heic_b200_file* f, int32_t image, uint32_t nal_unit_type,
                                         const uint8_t** data, size_t* len);
int32_t heic_b200_file_tile_nal(const heic_b200_file* f, int32_t image, uint32_t tile, const uint8_t** data, size_t* len);
/* Container metadata checked by the reference's integration test (tests/libheif_comparison.rs:102-111). */
typedef struct heic_file_info {
  uint32_t primary_item_id;
  uint32_t ispe_width, ispe_height;       /* ispe associated with the primary item */
  uint32_t rotation_ccw_quarter_turns;    /* irot.angle */
  uint32_t rotated_width, rotated_height; /* size after every transformative property (clap, irot, imir) */
  uint32_t luma_bits, chroma_bits;
  uint32_t thumbnail_count;
  uint32_t item_count;
  uint32_t is_grid;
} heic_file_info;
int32_t heic_b200_file_info(const heic_b200_file* f, heic_file_info* out);
/* The clap / irot / imir properties of an image item (image = -1: primary, >= 0: auxiliary), taken in the order its
 * ipma lists them and reduced to the normal form of heic_image_transform.  Properties of grid tile items are not applied. */
int32_t heic_b200_file_image_transform(const heic_b200_file* f, int32_t image, heic_image_transform* out);

/* ---- the hot path ------------------------------------------------------------------------- */
/* Replacement for the tile loop + SliceSegmentReader::read_data (decoder.rs:114-119, slice.rs:206):
 * decodes n_imgs images (all tiles of all images form one batch) from HOST descriptors and writes
 * interleaved RGB8 to HOST memory: image i at rgb_out + i*image_stride, rows of `pitch` bytes.
 * With apply_transforms = 0 the output is the output_width x output_height canvas; with 1 the irot
 * rotation is applied (width/height swap for odd quarter turns).  status (n_total_tiles entries,
 * images concatenated) may be NULL. */
int32_t heic_b200_decode_grids(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs,
                               uint8_t* rgb_out, size_t pitch, size_t image_stride,
                               int32_t apply_transforms, heic_tile_status* status);

/* Asynchronous form of the same call, for double-buffered serving loops: submit queues the host->device copies, the
 * kernels and the device->host copies of all chunks and returns; heic_b200_job_wait blocks until the RGB and the status
 * of that call are complete, returns its result (0 / HEIC_E_BITSTREAM) and frees the job.  Descriptors and bitstreams are
 * consumed before submit returns; rgb_out and status must stay valid until the wait.  Several jobs may be in flight on
 * one context (same thread); a later job's host->device copy and kernels overlap an earlier job's device->host copy. */
typedef struct heic_b200_job heic_b200_job;
int32_t heic_b200_decode_grids_submit(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs,
                                      uint8_t* rgb_out, size_t pitch, size_t image_stride,
                                      int32_t apply_transforms, heic_tile_status* status, heic_b200_job** out_job);
int32_t heic_b200_job_wait(heic_b200_job* job);

/* decode_grids / decode_grids_submit with an output geometry per image (xforms: n_imgs entries): image i is written as
 * heic_image_transform describes, crop_w x crop_h, or crop_h x crop_w for odd quarter turns.  A transform whose crop
 * does not lie inside its canvas, or whose orientation is above 7, fails the whole call with HEIC_E_INVALID_ARG before
 * anything is queued.  The calls without xforms are these with {whole canvas, rotation_ccw_quarter_turns & 3} per image
 * when apply_transforms != 0, and with the identity otherwise. */
int32_t heic_b200_decode_grids_transformed(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                           uint32_t n_imgs, uint8_t* rgb_out, size_t pitch, size_t image_stride,
                                           heic_tile_status* status);
int32_t heic_b200_decode_grids_submit_transformed(heic_b200_ctx* ctx, const heic_image_desc* imgs,
                                                  const heic_image_transform* xforms, uint32_t n_imgs, uint8_t* rgb_out,
                                                  size_t pitch, size_t image_stride, heic_tile_status* status,
                                                  heic_b200_job** out_job);

/* decode_grids_transformed / decode_grids_submit_transformed with a box reduction per image (reduce: n_imgs factors,
 * 1..16): image i is PIL.Image.fromarray(T).reduce(reduce[i]) of the RGB8 image T that the _transformed call writes for
 * xforms[i].  Its size is ceil(w / k) x ceil(h / k) for the w x h of T and k = reduce[i].  Each output pixel and channel
 * comes from the block of n = rows x cols pixels of T it covers (k x k, fewer in the last output row and column), with
 * channel sum S:
 *     out = (((S + n / 2) * M(n)) mod 2^32) >> 24,   M(n) = trunc(float32(2^32) / float32(256 * n))
 * (Pillow's fixed-point division; it differs from the rounded mean (S + n / 2) / n at some ties when n is not a power of
 * two).  Decoding is unchanged; only the colour stage and the output shrink.  Factors of 1 give the _transformed output
 * (those calls are these with every factor 1); factors may differ between images.  A factor of 0 or above 16 fails the
 * whole call with HEIC_E_INVALID_ARG before anything is queued. */
int32_t heic_b200_decode_grids_reduced(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                       const uint32_t* reduce, uint32_t n_imgs, uint8_t* rgb_out, size_t pitch,
                                       size_t image_stride, heic_tile_status* status);
int32_t heic_b200_decode_grids_submit_reduced(heic_b200_ctx* ctx, const heic_image_desc* imgs,
                                              const heic_image_transform* xforms, const uint32_t* reduce, uint32_t n_imgs,
                                              uint8_t* rgb_out, size_t pitch, size_t image_stride, heic_tile_status* status,
                                              heic_b200_job** out_job);

/* Same, planar YCbCr out (tile mosaic cropped to the output canvas, no colour conversion): Y plane
 * output_width x output_height, then Cb, Cr at half resolution (rounded up), per image.  Tiles are stitched at their
 * conformance-window size; no transform is applied.  */
int32_t heic_b200_decode_grids_yuv(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs,
                                   uint8_t* y_out, uint8_t* cb_out, uint8_t* cr_out,
                                   heic_tile_status* status);

/* Convenience: HeicDecoder::decode(&[u8]) that actually returns the image (decoder.rs:12 returns ()).
 * With apply_transforms != 0 the file's own transform (heic_b200_file_image_transform) is applied.
 * Query the size first with heic_b200_file_info (rotated_* when apply_transforms, else ispe_*). */
int32_t heic_b200_decode_file(heic_b200_ctx* ctx, const uint8_t* data, size_t len, uint8_t* rgb_out,
                              size_t pitch, int32_t apply_transforms);

/* ---- resident batches: decode with everything already in HBM (what bench.py's `value` times) --- */
typedef struct heic_b200_batch heic_b200_batch;
/* Uploads bitstreams + descriptors of n_imgs images (identical geometry per image is NOT required)
 * and allocates all intermediate and output buffers on the device. */
int32_t heic_b200_batch_create(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs,
                               heic_b200_batch** out);
/* The same with apply_transforms != 0: the RGB output of every image is rotated by its irot (as heic_b200_decode_grids does). */
int32_t heic_b200_batch_create_ex(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs, int32_t apply_transforms,
                                  heic_b200_batch** out);
/* The same with an output geometry per image (see heic_b200_decode_grids_transformed). */
int32_t heic_b200_batch_create_transformed(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                           uint32_t n_imgs, heic_b200_batch** out);
/* The same with a box reduction factor per image (1..16; see heic_b200_decode_grids_reduced for the definition): the
 * batch's RGB output, its pitch and its image stride are those of the reduced images. */
int32_t heic_b200_batch_create_reduced(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                       const uint32_t* reduce, uint32_t n_imgs, heic_b200_batch** out);
void    heic_b200_batch_destroy(heic_b200_batch* b);
/* Runs slice data -> RGB for the whole batch on the context's stream; does not synchronise. */
int32_t heic_b200_batch_decode(heic_b200_batch* b);
/* Stage selection for per-stage timing/parity: bitmask of HEIC_STAGE_*; stages run in pipeline order. */
enum {
  HEIC_STAGE_CABAC = 1, HEIC_STAGE_TRANSFORM = 2, HEIC_STAGE_INTRA = 4, HEIC_STAGE_DEBLOCK = 8,
  HEIC_STAGE_SAO = 16, HEIC_STAGE_COLOR = 32, HEIC_STAGE_ALL = 63
};
int32_t heic_b200_batch_run_stages(heic_b200_batch* b, uint32_t stage_mask);
int32_t heic_b200_batch_sync(heic_b200_batch* b);
/* CUDA stream (cudaStream_t) the batch launches on, for event timing by the caller. */
void*   heic_b200_batch_stream(heic_b200_batch* b);
/* Device pointer + layout of the RGB output (image i at base + i*image_stride). */
int32_t heic_b200_batch_rgb(heic_b200_batch* b, void** dev_ptr, size_t* pitch, size_t* image_stride);
int32_t heic_b200_batch_download_rgb(heic_b200_batch* b, uint8_t* rgb_out, size_t pitch, size_t image_stride);
/* RGB of one image of the batch (rows of rot_w*3 bytes, `pitch` apart) to host memory; synchronises the batch's stream. */
int32_t heic_b200_batch_download_image(heic_b200_batch* b, uint32_t image_index, uint8_t* rgb_out, size_t pitch);
int32_t heic_b200_batch_status(heic_b200_batch* b, heic_tile_status* status /* n_total_tiles */);
uint32_t heic_b200_batch_tile_count(const heic_b200_batch* b);
/* CABAC launch order of a resident batch (tools / bench.py): tile indices, *tiles_per_group (32 or 1) per CTA, 0xffffffff =
 * idle lane.  Returns the number of entries and copies at most `cap` of them; `out` / `tiles_per_group` may be NULL. */
size_t   heic_b200_batch_cabac_order(const heic_b200_batch* b, uint32_t* out, size_t cap, uint32_t* tiles_per_group);

/* Intermediate buffers of one tile, copied to host, for per-stage parity tests.  Layouts are
 * documented in DESIGN.md ("Data layout in HBM").  Any pointer may be NULL.  The coefficient buffers hold levels
 * after the CABAC stage, residuals after the transform stage, and zeros once the intra stage has consumed them. */
typedef struct heic_tile_dump {
  uint32_t* tu_map;      uint32_t tu_map_len;     /* one word per 4x4 luma block, CTB-major z-order  */
  int16_t*  coeff[3];    uint32_t coeff_len[3];   /* levels (after CABAC) or residual (after TRANSFORM) */
  uint8_t*  qp_map;      uint32_t qp_map_len;     /* QpY per 8x8 luma block, raster                   */
  uint32_t* sao;         uint32_t sao_len;        /* 4 words per CTB                                  */
  uint8_t*  plane[3];    uint32_t plane_len[3];   /* current picture planes (recon / deblocked / SAO) */
} heic_tile_dump;
int32_t heic_b200_batch_dump_tile(heic_b200_batch* b, uint32_t tile_index, heic_tile_dump* dump);

/* ---- stand-alone stage entry point on caller-owned DEVICE buffers (config 2 of the survey) ---- */
/* [+] RbspReader::remove_emulation_prevention on the GPU                    src/hevc/rbsp_reader.rs:11-39
 * One raw NAL payload (after the 2-byte header) in, its RBSP out (rbsp_out holds `len` bytes), plus the slice data
 * offset and the substream offsets re-based from raw to un-escaped byte counts — the stage heic_b200_decode_grids
 * runs for heic_tile_desc::escaped tiles, exposed for parity tests against the host function. */
int32_t heic_b200_unescape(heic_b200_ctx* ctx, const uint8_t* nal_payload, size_t len, uint32_t slice_data_byte_offset,
                           const uint32_t* substream_offset, uint32_t n_substreams, uint8_t* rbsp_out, size_t* rbsp_len,
                           uint32_t* slice_data_byte_offset_out, uint32_t* substream_offset_out);

/* YCbCr 4:2:0 -> RGB8 + grid stitch + crop.  planes: n_tiles tiles, each tile_w*tile_h Y followed by
 * Cb and Cr at (tile_w/2)*(tile_h/2), contiguous per tile (tile stride = tile_w*tile_h*3/2).
 * full_range/matrix_coeffs select the integer matrix (DESIGN.md, "Colour definition"). */
int32_t heic_b200_color_stitch(heic_b200_ctx* ctx, const void* dev_planes, uint32_t n_images,
                               uint32_t grid_rows, uint32_t grid_cols, uint32_t tile_w, uint32_t tile_h,
                               uint32_t out_w, uint32_t out_h, uint32_t full_range, uint32_t matrix_coeffs,
                               void* dev_rgb, size_t pitch, size_t image_stride);

#ifdef __cplusplus
}
#endif
#endif /* HEIC_B200_H */
