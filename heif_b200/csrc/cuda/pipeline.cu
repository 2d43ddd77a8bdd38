// Host side of the GPU path: resident batches (bitstreams + descriptors + every intermediate in HBM),
// stage sequencing on one CUDA stream, and the C ABI of include/heic_b200.h for everything that touches
// the device.  This is the replacement for the tile loop of HeicDecoder::decode
// (reference src/heic/decoder.rs:98-119) and SliceSegmentReader::read_data (src/hevc/slice.rs:206).
// There is no CPU fallback: without a usable CUDA device every entry point fails with HEIC_E_NO_DEVICE.
#include <cuda_runtime.h>

#include <chrono>
#include <cstdio>
#include <cstdlib>

#include <algorithm>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "../host/capi_common.h"
#include "../host/heic_decoder.h"
#include "../host/resample.h"
#include "cabac_tables.h"
#include "host_params.h"
#include "kernels.h"

using namespace heic;
using namespace heic::dev;

namespace {

[[noreturn]] void cuda_fail(cudaError_t e, const char* what) {
  int code = (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver || e == cudaErrorInvalidDevice) ? HEIC_E_NO_DEVICE
             : (e == cudaErrorMemoryAllocation)                                                          ? HEIC_E_NOMEM
                                                                                                         : HEIC_E_CUDA;
  bail(code, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(call)                               \
  do {                                         \
    cudaError_t e__ = (call);                  \
    if (e__ != cudaSuccess) cuda_fail(e__, #call); \
  } while (0)

// Growable device / pinned-host buffers: decode_grids re-uses one scratch batch per context, so steady
// state calls do not allocate.
struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  void ensure(size_t n) {
    if (n <= cap) return;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 256;
    CU(cudaMalloc(&p, want));
    cap = want;
  }
  ~DevBuf() {
    if (p) cudaFree(p);
  }
};
struct PinnedBuf {
  void* p = nullptr;
  size_t cap = 0;
  void ensure(size_t n) {
    if (n <= cap) return;
    if (p) cudaFreeHost(p);
    p = nullptr;
    cap = 0;
    size_t want = n + n / 8 + 256;
    CU(cudaMallocHost(&p, want));
    cap = want;
  }
  ~PinnedBuf() {
    if (p) cudaFreeHost(p);
  }
};

size_t up(size_t v, size_t a) { return (v + a - 1) / a * a; }

int env_int(const char* name, int dflt) {
  const char* s = std::getenv(name);
  return (s && *s) ? std::atoi(s) : dflt;
}

}  // namespace

// One submitted decode_grids call: its chunks are in flight on the context's pipeline slots until it is waited for.
struct heic_b200_job {
  heic_b200_ctx* ctx = nullptr;
  heic_tile_status* status = nullptr;     // caller's array, or `local`
  std::vector<heic_tile_status> local;
  size_t n_tiles = 0;
};

struct PipePending {
  heic_b200_job* job = nullptr;  // null: slot idle
  size_t tile0 = 0, n_tiles = 0;
  // HEIC_B200_TRACE=2: device timeline of the chunk (events: queued, slice data on the device, CABAC done, kernels done, RGB on the host)
  cudaEvent_t ev[5] = {};
  double host_ms = 0;  // host time at which the chunk was queued
};

struct heic_b200_ctx {
  int device = 0;
  int n_sm = 148;
  cudaStream_t stream = nullptr;
  CabacTabs* d_tabs = nullptr;
  uint64_t launches = 0;
  int cabac_tiles_per_cta = 32;  // 32: thread per substream, 1: warp per substream
  int cabac_slots = 0;           // 0: derive from the picture geometry
  int low_latency_tiles = 384;   // loads of at most this many tiles use the warp-per-substream CABAC mapping
  int intra_slots = 0;           // 0: automatic (wavefront for small batches, one warp per picture for large)
  int intra_single_warp_tiles = 2048;
  int cabac_plain_sort = 0;      // measurement knob: plain size sort, copies of a slice may share a warp (bench.py's upper bound)
  int cabac_resident = 0;        // persistent CABAC CTAs to launch; 0: as many as are resident at once (tests use 2)
  int cabac_persistent = 1;      // large batches: CABAC CTAs take group after group, warp by warp (no ramp-up / drain per group)
  int fuse_sao = 1;              // full decodes to RGB apply SAO inside the colour kernel (no `final` planes round trip)
  // decode_grids pipeline: chunks of `pipe_chunk` images rotate over up to kPipe slots, each with its own stream and
  // scratch batch, so the H2D copy, the kernels and the D2H copy of different chunks overlap
  static constexpr int kPipe = 16;
  int pipe_chunk = 0;   // images per chunk; 0: automatic (see submit_grids)
  int pipe_slots = 0;   // chunks in flight; 0: automatic
  cudaEvent_t trace_base = nullptr;  // HEIC_B200_TRACE=2: time zero of the chunk timelines
  int pipe_order = 1;                // chunks in flight keep their order on the device (HEIC_B200_PIPE_ORDER=0: A/B)
  cudaEvent_t ev_cabac = nullptr, ev_d2h = nullptr;  // end of the last queued chunk's CABAC stage / device->host copies
  bool d2h_recorded = false;
  cudaStream_t pipe_stream[kPipe] = {};
  std::unique_ptr<heic_b200_batch> pipe_batch[kPipe];
  PipePending pipe_pending[kPipe];
  uint32_t pipe_next = 0;  // round-robin slot cursor, continues across calls so that jobs in flight interleave
  ~heic_b200_ctx();
};

// One image of a batch.  Everything but first_tile, pic and src_slot is planned before the batch is loaded (plan_image).
struct ImageInfo {
  uint32_t first_tile, n_tiles, pic;
  uint32_t grid_rows, grid_cols, canvas_w, canvas_h;        // canvas: output_width x output_height of the descriptor
  uint32_t tile_w, tile_h, win_x, win_y;                    // conformance window of every tile (luma samples)
  uint32_t crop_x, crop_y, crop_w, crop_h, orientation;     // heic_image_transform
  uint32_t reduce;                                          // box reduction factor (1: none)
  uint32_t color_w, color_h;                                // size of the colour stage's output (oriented, reduced)
  uint32_t rgb_w, rgb_h;                                    // the RGB output (oriented, reduced, resized)
  uint32_t filter;                                          // resize filter (HEIC_RESAMPLE_*); 0: rgb_w x rgb_h = color_w x color_h
  uint32_t src_slot;                                        // resized images: index in the batch's source arena
  uint32_t full_range, matrix_coeffs;
};

// What one image's RGB output is: the crop and turn of its canvas, then the box reduction, then the resize.
struct OutputSpec {
  heic_image_transform xf;
  uint32_t reduce;
  heic_resize resize;
};

// An image planned and validated before anything is queued: its ImageInfo and the parameters of its decoded pictures.
struct ImagePlan {
  ImageInfo info;
  PicParams pp;
};

namespace {

// The part of a decoded picture that a grid stitches: its conformance window, in luma samples.
struct TileWindow {
  uint32_t x, y, w, h;
};

// Decoded picture, conformance window and output canvas of an image descriptor; throws for a window or a canvas that
// the tiles do not cover.
void image_geometry(const heic_image_desc& im, PicParams& pp, TileWindow& tw, uint32_t& canvas_w, uint32_t& canvas_h) {
  if (!im.tiles || im.n_tiles == 0 || im.n_tiles != im.grid_rows * im.grid_cols)
    bail(HEIC_E_INVALID_ARG, "image descriptor: n_tiles must equal grid_rows * grid_cols");
  make_pic_params(im.sps, im.pps, pp);
  tw = {0, 0, (uint32_t)pp.w, (uint32_t)pp.h};
  if (im.sps.conformance_window_flag) {
    const uint64_t sub = pp.chroma ? 2 : 1;  // SubWidthC = SubHeightC: 4:2:0 or 4:0:0 (make_pic_params rejects the rest)
    const uint64_t l = sub * im.sps.conf_win_left_offset, r = sub * im.sps.conf_win_right_offset;
    const uint64_t t = sub * im.sps.conf_win_top_offset, b = sub * im.sps.conf_win_bottom_offset;
    if (l + r >= (uint64_t)pp.w || t + b >= (uint64_t)pp.h) bail(HEIC_E_BITSTREAM, "conformance window is empty");
    tw = {(uint32_t)l, (uint32_t)t, (uint32_t)(pp.w - l - r), (uint32_t)(pp.h - t - b)};
  }
  const uint64_t mosaic_w = (uint64_t)im.grid_cols * tw.w, mosaic_h = (uint64_t)im.grid_rows * tw.h;
  const uint64_t ow = im.output_width ? im.output_width : mosaic_w, oh = im.output_height ? im.output_height : mosaic_h;
  if (ow > mosaic_w || oh > mosaic_h) bail(HEIC_E_BITSTREAM, "grid canvas is larger than the tile mosaic");
  canvas_w = (uint32_t)ow;
  canvas_h = (uint32_t)oh;
}

void check_transform(const heic_image_transform& x, uint32_t canvas_w, uint32_t canvas_h) {
  if (x.orientation > 7 || !x.crop_w || !x.crop_h || (uint64_t)x.crop_x + x.crop_w > canvas_w || (uint64_t)x.crop_y + x.crop_h > canvas_h)
    bail(HEIC_E_INVALID_ARG, "image transform: crop rectangle not inside the canvas, or orientation above 7");
}

void check_reduce(uint32_t k) {
  if (k < 1 || k > 16) bail(HEIC_E_INVALID_ARG, "reduction factor outside 1..16");
}

void check_resize(const heic_resize& r) {
  if ((r.width == 0) != (r.height == 0) || r.width > kResampleMaxSide || r.height > kResampleMaxSide ||
      (r.width && (r.filter < HEIC_RESAMPLE_LANCZOS || r.filter > HEIC_RESAMPLE_HAMMING)))
    bail(HEIC_E_INVALID_ARG, "resize: exactly one side 0, a side above 32768, or a filter outside 1..5");
}

// One OutputSpec per image from the caller's arrays of n_imgs entries.  A null array is the default: the whole canvas,
// turned by irot when apply_transforms is set; factor 1; no resize.  (A public call that takes an array rejects a null one
// before it gets here.)
std::vector<OutputSpec> output_specs(const heic_image_desc* imgs, uint32_t n_imgs, const heic_image_transform* xforms,
                                     const uint32_t* reduce, const heic_resize* resize, int32_t apply_transforms) {
  if (!imgs) bail(HEIC_E_INVALID_ARG, "null argument");
  std::vector<OutputSpec> specs(n_imgs);
  for (uint32_t i = 0; i < n_imgs; i++) {
    OutputSpec& s = specs[i];
    if (xforms) {
      s.xf = xforms[i];
    } else {
      PicParams pp;
      TileWindow tw;
      uint32_t cw, ch;
      image_geometry(imgs[i], pp, tw, cw, ch);
      s.xf = {0, 0, cw, ch, apply_transforms ? (imgs[i].rotation_ccw_quarter_turns & 3u) : 0u};
    }
    s.reduce = reduce ? reduce[i] : 1u;
    s.resize = resize ? resize[i] : heic_resize{0, 0, 0};
  }
  return specs;
}

// Plans one image: throws for an invalid descriptor or spec, checking in this order the descriptor and its canvas, the
// transform, the factor, the resize and every tile's slice header.  Without RGB output (with_rgb = false) no resize runs.
ImagePlan plan_image(const heic_image_desc& im, const OutputSpec& s, bool with_rgb) {
  ImagePlan p;
  ImageInfo& info = p.info;
  TileWindow win;
  image_geometry(im, p.pp, win, info.canvas_w, info.canvas_h);
  check_transform(s.xf, info.canvas_w, info.canvas_h);
  check_reduce(s.reduce);
  check_resize(s.resize);
  TileParams tp;
  for (uint32_t t = 0; t < im.n_tiles; t++) make_tile_params(p.pp, im.pps, im.tiles[t], tp);
  info.first_tile = info.pic = info.src_slot = 0;  // set by load()
  info.n_tiles = im.n_tiles;
  info.grid_rows = im.grid_rows;
  info.grid_cols = im.grid_cols;
  info.tile_w = win.w;
  info.tile_h = win.h;
  info.win_x = win.x;
  info.win_y = win.y;
  info.crop_x = s.xf.crop_x;
  info.crop_y = s.xf.crop_y;
  info.crop_w = s.xf.crop_w;
  info.crop_h = s.xf.crop_h;
  info.orientation = s.xf.orientation;
  info.reduce = s.reduce;
  // the crop, turned for odd quarter turns, then ceil(w / k) x ceil(h / k)
  const bool turned = s.xf.orientation & 1u;
  info.color_w = ((turned ? s.xf.crop_h : s.xf.crop_w) + s.reduce - 1) / s.reduce;
  info.color_h = ((turned ? s.xf.crop_w : s.xf.crop_h) + s.reduce - 1) / s.reduce;
  info.rgb_w = with_rgb && s.resize.width ? s.resize.width : info.color_w;
  info.rgb_h = with_rgb && s.resize.width ? s.resize.height : info.color_h;
  // a resize to the size it already has is Pillow's copy(): the colour stage writes the output
  info.filter = info.rgb_w != info.color_w || info.rgb_h != info.color_h ? s.resize.filter : 0u;
  info.full_range = im.sps.vui_parameters_present_flag ? im.sps.video_full_range_flag : 0u;
  info.matrix_coeffs = im.sps.vui_parameters_present_flag ? im.sps.matrix_coeffs : 2u;
  return p;
}

}  // namespace

// One distinct coefficient table of a load: its device layout sits in heic_b200_batch::rs_tables at these int32 offsets.
struct ResampleTableRef {
  ResampleAxis ax;              // the pointers are filled in by run()
  size_t o_out, o_band, o_coef;
  uint32_t row0, row_end;       // as a vertical table: the first and one past the last source row it reads
};

// Images in a row of a batch with equal (source size, target size, filter): one launch per resampling pass.
struct ResampleRun {
  uint32_t first, count;      // images
  int h_table, v_table;       // index into heic_b200_batch::rs_axes; -1: that pass does not run
  uint32_t row0, rows;        // horizontal pass: source rows it reads (the vertical pass's first and last used rows)
  size_t tmp_off, tmp_pitch, tmp_stride;  // uint8 intermediate of the two-pass case
};

struct CabacClass {  // tiles launched together: same wavefront shape
  int n_slots, hctb;
  uint32_t order_off, n_groups, n_tiles;
};

struct heic_b200_batch {
  heic_b200_ctx* ctx = nullptr;
  cudaStream_t stream = nullptr;  // ctx->stream for explicit batches, a pipeline stream for decode_grids chunks
  int tiles_per_cta = 32;         // CABAC mapping of this load: 32 (throughput) or 1 (lowest latency, small loads)
  std::vector<PicParams> pics;
  std::vector<ScalingSet> scaling;
  std::vector<TileParams> tiles;
  std::vector<ImageInfo> images;
  std::vector<uint32_t> substreams, order, heavy_first;
  std::vector<CabacClass> classes;
  std::vector<ResampleRun> rs_runs;
  std::vector<ResampleTableRef> rs_axes;
  std::vector<int32_t> rs_tables;     // device layout of every distinct table of the load (ResampleAxis)
  size_t src_pitch = 0, src_image_stride = 0, n_src = 0, tmp_bytes = 0;
  size_t src_off = 0, tmp_off = 0;  // byte offsets of the source arena and the intermediate inside d_rgb's allocation
  size_t raw_bytes = 0;       // raw NAL payloads of the tiles shipped with emulation prevention bytes in place
  bool any_plain = false;
  size_t bs_bytes = 0, tu_words = 0, coeff_elems = 0, plane_bytes = 0, map4_bytes = 0, map8_bytes = 0, sao_words = 0, wpp_bytes = 0;
  size_t rgb_pitch = 0, rgb_image_stride = 0;
  uint32_t max_tu = 0, max_w = 0, max_h = 0, max_pitch = 0;
  int max_log2_ctb = 4, max_log2_tb = 2, intra_slots = 1, max_hctb = 1;
  uint32_t stages_run = 0;
  bool final_stale = false;   // SAO ran fused into the colour kernel: the `final` planes were not written (dump_tile refreshes them)
  bool coeff_clean = false;   // the coefficient arena is all-zero (fresh memset, or the last intra stage cleared it)
  PinnedBuf h_bitstream, h_status, h_params;
  // inside the parameter blob
  size_t off_sub = 0, off_order = 0, off_heavy = 0, off_pics = 0, off_tiles = 0, off_scaling = 0, off_resample = 0;
  // d_rgb's allocation also holds, after the RGB output, the source arena (the colour stage's output of the resized
  // images; the output then holds the resized ones) and the uint8 rows of the horizontal pass of the two-pass images: one
  // allocation, so a context that alternates resized and unresized calls keeps the larger of the two layouts, not both.
  DevBuf d_bitstream, d_params, d_tu, d_coeff, d_recon, d_final, d_ipm, d_ctd,
      d_qp, d_sao, d_wpp, d_status, d_rgb, d_list, d_list_count, d_raw, d_counters;
  PinnedBuf h_raw;
  uint32_t list_off[LIST_CLASSES] = {};
  Arenas arenas() const {
    Arenas a;
    a.bitstream = (const uint8_t*)d_bitstream.p;
    a.raw = (const uint8_t*)d_raw.p;
    const uint8_t* pb = (const uint8_t*)d_params.p;
    a.substreams = (const uint32_t*)(pb + off_sub);
    a.pics = (const PicParams*)(pb + off_pics);
    a.tiles = (const TileParams*)(pb + off_tiles);
    a.scaling = (const ScalingSet*)(pb + off_scaling);
    a.tu_map = (uint32_t*)d_tu.p;
    a.coeff = (int16_t*)d_coeff.p;
    a.recon = (uint8_t*)d_recon.p;
    a.final_ = (uint8_t*)d_final.p;
    a.ipm = (uint8_t*)d_ipm.p;
    a.ct_depth = (uint8_t*)d_ctd.p;
    a.qp_map = (uint8_t*)d_qp.p;
    a.sao = (uint32_t*)d_sao.p;
    a.wpp_save = (uint8_t*)d_wpp.p;
    a.status = (TileStatusDev*)d_status.p;
    a.n_tiles = (uint32_t)tiles.size();
    a.tu_list = (uint2_t*)d_list.p;
    a.list_count = (uint32_t*)d_list_count.p;
    for (int k = 0; k < LIST_CLASSES; k++) a.list_off[k] = list_off[k];
    return a;
  }
  void load(const heic_image_desc* imgs, const ImagePlan* plans, uint32_t n_imgs, bool with_rgb);
  void layout_tiles(const heic_image_desc* imgs, const ImagePlan* plans, uint32_t n_imgs);
  void plan_resample();
  void plan_cabac(const heic_image_desc* imgs, uint32_t n_imgs);
  void upload(const heic_image_desc* imgs, uint32_t n_imgs, bool with_rgb);
  void run(uint32_t mask);
};

heic_b200_ctx::~heic_b200_ctx() {
  if (trace_base) cudaEventDestroy(trace_base);
  if (ev_cabac) cudaEventDestroy(ev_cabac);
  if (ev_d2h) cudaEventDestroy(ev_d2h);
  for (int i = 0; i < kPipe; i++) {
    for (cudaEvent_t e : pipe_pending[i].ev)
      if (e) cudaEventDestroy(e);
    pipe_batch[i].reset();
    if (pipe_stream[i]) cudaStreamDestroy(pipe_stream[i]);
  }
  if (d_tabs) cudaFree(d_tabs);
  if (stream) cudaStreamDestroy(stream);
}

// ---- batch construction --------------------------------------------------------------------------------
// Loads planned images: arena layout, resampling, CABAC launch classes, then the uploads on the batch's stream.
void heic_b200_batch::load(const heic_image_desc* imgs, const ImagePlan* plans, uint32_t n_imgs, bool with_rgb) {
  layout_tiles(imgs, plans, n_imgs);
  plan_resample();
  if (tiles.size() >= (1u << 24)) bail(HEIC_E_UNSUPPORTED, "more than 2^24 tiles in one batch (the transform lists keep the tile index in 24 bits)");
  plan_cabac(imgs, n_imgs);
  upload(imgs, n_imgs, with_rgb);
}

// Per-tile parameters and the offsets of every tile's slice of the per-batch arenas; the RGB output's layout.
void heic_b200_batch::layout_tiles(const heic_image_desc* imgs, const ImagePlan* plans, uint32_t n_imgs) {
  pics.clear();
  scaling.clear();
  tiles.clear();
  images.clear();
  substreams.clear();
  raw_bytes = 0;
  any_plain = false;
  bs_bytes = tu_words = coeff_elems = plane_bytes = map4_bytes = map8_bytes = sao_words = wpp_bytes = 0;
  max_tu = max_w = max_h = max_pitch = 0;
  max_log2_ctb = 4;
  max_log2_tb = 2;
  intra_slots = 1;
  max_hctb = 1;
  stages_run = 0;
  size_t max_rgb_rows = 0, max_rgb_pitch = 0;
  for (uint32_t i = 0; i < n_imgs; i++) {
    const heic_image_desc& im = imgs[i];
    PicParams pp = plans[i].pp;
    ScalingSet ss;
    build_scaling_set(im.sps, im.pps, ss);
    size_t s = 0;
    for (; s < scaling.size(); s++)
      if (!std::memcmp(&scaling[s], &ss, sizeof ss)) break;
    if (s == scaling.size()) scaling.push_back(ss);
    pp.scaling_set = (int)s;
    // consecutive images with identical parameters share one PicParams entry
    if (pics.empty() || std::memcmp(&pics.back(), &pp, sizeof pp)) pics.push_back(pp);
    const uint32_t pic = (uint32_t)pics.size() - 1;
    ImageInfo info = plans[i].info;
    info.first_tile = (uint32_t)tiles.size();
    info.pic = pic;
    images.push_back(info);
    max_rgb_pitch = std::max(max_rgb_pitch, up((size_t)info.rgb_w * 3, 16));
    max_rgb_rows = std::max(max_rgb_rows, (size_t)info.rgb_h);
    for (uint32_t t = 0; t < im.n_tiles; t++) {
      TileParams tp;
      std::memset(&tp, 0, sizeof tp);
      make_tile_params(pp, im.pps, im.tiles[t], tp);
      tp.pic = pic;
      tp.image = i;
      tp.tile_in_image = t;
      tp.bs_off = (uint32_t)bs_bytes;
      bs_bytes = up(bs_bytes + tp.bs_len + 8, 16);
      tp.escaped = im.tiles[t].escaped ? 1u : 0u;
      if (tp.escaped) {
        tp.raw_off = raw_bytes;
        raw_bytes = up(raw_bytes + tp.bs_len + 8, 16);
      } else {
        any_plain = true;
      }
      if (bs_bytes > 0xfff00000ull) bail(HEIC_E_UNSUPPORTED, "more than 4 GiB of slice data in one batch");
      tp.sub_first = (uint32_t)substreams.size();
      for (uint32_t k = 0; k < tp.n_sub; k++) substreams.push_back(im.tiles[t].header.substream_offset[k]);
      tp.tu_off = tu_words;
      tu_words += (size_t)pp.n_tu;
      tp.coeff_off[0] = coeff_elems;
      tp.coeff_off[1] = tp.coeff_off[0] + (size_t)pp.n_tu * 16;
      tp.coeff_off[2] = tp.coeff_off[1] + (size_t)pp.n_tu * 4;
      coeff_elems = tp.coeff_off[2] + (size_t)pp.n_tu * 4;
      // planes cover whole CTBs so the intra kernel never needs a store mask beyond the picture size
      const size_t ysz = (size_t)pp.pitch_y * (size_t)pp.h, csz = (size_t)pp.pitch_c * (size_t)(pp.h >> 1);
      tp.plane_off[0] = plane_bytes;
      tp.plane_off[1] = tp.plane_off[0] + ysz;
      tp.plane_off[2] = tp.plane_off[1] + csz;
      plane_bytes = up(tp.plane_off[2] + csz, 256);
      tp.map4_off = map4_bytes;
      map4_bytes = up(map4_bytes + (size_t)pp.w4 * pp.h4, 64);
      tp.map8_off = map8_bytes;
      map8_bytes = up(map8_bytes + (size_t)pp.w8 * pp.h8, 64);
      tp.sao_off = sao_words;
      sao_words += (size_t)pp.wctb * pp.hctb * 4;
      tp.wpp_off = wpp_bytes;
      wpp_bytes += (size_t)pp.hctb * NUM_CTX_PAD;
      tiles.push_back(tp);
    }
    max_tu = std::max(max_tu, (uint32_t)pp.n_tu);
    max_w = std::max(max_w, (uint32_t)pp.w);
    max_h = std::max(max_h, (uint32_t)pp.h);
    max_pitch = std::max(max_pitch, (uint32_t)pp.pitch_y);
    max_log2_ctb = std::max(max_log2_ctb, pp.log2_ctb);
    max_log2_tb = std::max(max_log2_tb, pp.log2_max_tb);
    max_hctb = std::max(max_hctb, pp.hctb);
    intra_slots = std::max(intra_slots, std::min(8, std::min(pp.hctb, (pp.wctb + 1) / 2 + 1)));
  }
  rgb_pitch = max_rgb_pitch;
  // every image is written at the widest pitch: the stride holds the tallest image at that pitch
  rgb_image_stride = up(max_rgb_pitch * max_rgb_rows, 256);
}

// CABAC launch classes: tiles with the same wavefront shape, heaviest first, tiles_per_cta per CTA; and the intra
// kernel's launch order.
void heic_b200_batch::plan_cabac(const heic_image_desc* imgs, uint32_t n_imgs) {
  order.clear();
  heavy_first.clear();
  classes.clear();
  // few tiles: a warp per substream finishes a 12 MP image in about half the time of the 32-tiles-per-CTA mapping
  // (the GPU is mostly empty either way); many tiles: thread per substream is 11x the throughput
  tiles_per_cta = (ctx->cabac_tiles_per_cta == 32 && tiles.size() > (size_t)ctx->low_latency_tiles) ? 32 : 1;
  const int tpc = tiles_per_cta;
  // content fingerprint of every slice (four 8-byte samples): equal length + equal fingerprint = "the same picture again"
  std::vector<uint64_t> fingerprint(tiles.size(), 0);
  {
    size_t t = 0;
    for (uint32_t i = 0; i < n_imgs; i++)
      for (uint32_t k = 0; k < imgs[i].n_tiles; k++, t++) {
        const uint8_t* p = imgs[i].tiles[k].rbsp;
        const size_t len = imgs[i].tiles[k].rbsp_len;
        uint64_t h = 0x9e3779b97f4a7c15ull ^ len;
        if (len >= 8)
          for (int q = 0; q < 4; q++) {
            uint64_t w8;
            std::memcpy(&w8, p + (len - 8) * q / 3, 8);
            h = (h ^ w8) * 0xbf58476d1ce4e5b9ull;
            h ^= h >> 29;
          }
        fingerprint[t] = h;
      }
  }
  std::map<std::tuple<int, int, int, int>, std::vector<uint32_t>> by_shape;
  for (uint32_t t = 0; t < tiles.size(); t++) {
    const PicParams& pp = pics[tiles[t].pic];
    by_shape[std::make_tuple(pp.wpp, pp.wctb, pp.hctb, pp.log2_ctb)].push_back(t);
  }
  for (auto& kv : by_shape) {
    std::vector<uint32_t>& v = kv.second;
    std::stable_sort(v.begin(), v.end(), [&](uint32_t a, uint32_t b) {
      return tiles[a].bs_len != tiles[b].bs_len ? tiles[a].bs_len > tiles[b].bs_len : fingerprint[a] < fingerprint[b];
    });
    const int wpp = std::get<0>(kv.first), wctb = std::get<1>(kv.first), hctb = std::get<2>(kv.first);
    CabacClass c;
    // with the two-CTU WPP lag at most ceil(wctb / 2) rows of a picture are in flight
    c.n_slots = wpp ? std::max(1, std::min(hctb, (wctb + 1) / 2)) : 1;
    if (ctx->cabac_slots > 0 && wpp) c.n_slots = std::min(hctb, ctx->cabac_slots);
    c.n_slots = std::min(c.n_slots, tpc == 32 ? 8 : 16);
    c.order_off = (uint32_t)order.size();
    // Tiles stay sorted by slice size so that the lanes of a warp carry similar statistics: measured on a B200,
    // dealing heavy and light tiles round-robin into the same warp is 3.5x slower (the light lanes idle while one
    // heavy lane runs at single-thread latency).  Groups of about equal slice bytes and a byte cap on the heaviest
    // groups (fewer lanes for them) measured slower too, see DESIGN.md.
    c.n_groups = 0;
    if (tpc == 1) {
      for (uint32_t t : v) order.push_back(t);
      c.n_groups = (uint32_t)v.size();
    } else {
      // Groups of 32 tiles of neighbouring slice size, NO TWO OF THEM BYTE-IDENTICAL.  The sorted list is seen as runs of
      // identical slices (same length and same content fingerprint; a batch of distinct pictures has runs of one, and the
      // groups are then simply consecutive blocks of the sorted list).  A group takes one tile from each of the first 32
      // runs that still have one, so copies of a picture -- which would run converged in one warp and flatter the
      // throughput, as a benchmark batch built from few distinct tiles does -- always land in different warps, while the
      // lanes of a warp stay as similar in size as the input allows.
      struct Run {
        size_t first, left;
      };
      std::vector<Run> runs;
      for (size_t i = 0; i < v.size();) {
        size_t j = i + 1;
        while (!ctx->cabac_plain_sort && j < v.size() && tiles[v[j]].bs_len == tiles[v[i]].bs_len && fingerprint[v[j]] == fingerprint[v[i]]) j++;
        runs.push_back({i, j - i});
        i = j;
      }
      size_t head = 0;  // runs before `head` are exhausted
      while (head < runs.size()) {
        int n = 0;
        for (size_t r = head; r < runs.size() && n < tpc; r++) {
          if (!runs[r].left) continue;
          order.push_back(v[runs[r].first++]);
          runs[r].left--;
          n++;
        }
        while (head < runs.size() && !runs[head].left) head++;
        for (; n < tpc; n++) order.push_back(0xffffffffu);
        c.n_groups++;
      }
    }
    c.hctb = hctb;
    c.n_tiles = (uint32_t)v.size();
    classes.push_back(c);
  }

  // every tile once, largest slice first: launch order of the one-CTA-per-picture intra kernel (the heaviest pictures
  // must not be the last ones to start)
  heavy_first.resize(tiles.size());
  for (uint32_t t = 0; t < tiles.size(); t++) heavy_first[t] = t;
  std::stable_sort(heavy_first.begin(), heavy_first.end(), [&](uint32_t a, uint32_t b) { return tiles[a].bs_len > tiles[b].bs_len; });
}

// Device memory and uploads: one pinned blob for all parameter tables, one for the slice data.
void heic_b200_batch::upload(const heic_image_desc* imgs, uint32_t n_imgs, bool with_rgb) {
  cudaStream_t st = stream;
  if (any_plain) h_bitstream.ensure(bs_bytes + 16);
  if (raw_bytes) h_raw.ensure(raw_bytes + 16);
  {
    size_t t = 0;
    uint8_t* hb = (uint8_t*)h_bitstream.p;
    uint8_t* hr = (uint8_t*)h_raw.p;
    for (uint32_t i = 0; i < n_imgs; i++)
      for (uint32_t k = 0; k < imgs[i].n_tiles; k++, t++) {
        const size_t len = imgs[i].tiles[k].rbsp_len;
        if (tiles[t].escaped) {  // raw NAL payload: un-escaped on the device into its bitstream slot
          std::memcpy(hr + tiles[t].raw_off, imgs[i].tiles[k].rbsp, len);
          std::memset(hr + tiles[t].raw_off + len, 0, up(len + 8, 16) - len);
          continue;
        }
        std::memcpy(hb + tiles[t].bs_off, imgs[i].tiles[k].rbsp, len);
        const size_t end = tiles[t].bs_off + len;
        const size_t next = t + 1 < tiles.size() ? tiles[t + 1].bs_off : bs_bytes + 16;
        std::memset(hb + end, 0, next - end);
      }
  }
  off_sub = 0;
  off_order = up(off_sub + substreams.size() * 4, 256);
  off_heavy = up(off_order + order.size() * 4, 256);
  off_pics = up(off_heavy + heavy_first.size() * 4, 256);
  off_tiles = up(off_pics + pics.size() * sizeof(PicParams), 256);
  off_scaling = up(off_tiles + tiles.size() * sizeof(TileParams), 256);
  off_resample = up(off_scaling + scaling.size() * sizeof(ScalingSet), 256);
  const size_t params_bytes = up(off_resample + rs_tables.size() * sizeof(int32_t), 256);
  h_params.ensure(params_bytes);
  {
    uint8_t* hp = (uint8_t*)h_params.p;
    std::memcpy(hp + off_sub, substreams.data(), substreams.size() * 4);
    std::memcpy(hp + off_order, order.data(), order.size() * 4);
    std::memcpy(hp + off_heavy, heavy_first.data(), heavy_first.size() * 4);
    std::memcpy(hp + off_pics, pics.data(), pics.size() * sizeof(PicParams));
    std::memcpy(hp + off_tiles, tiles.data(), tiles.size() * sizeof(TileParams));
    std::memcpy(hp + off_scaling, scaling.data(), scaling.size() * sizeof(ScalingSet));
    std::memcpy(hp + off_resample, rs_tables.data(), rs_tables.size() * sizeof(int32_t));
  }
  d_bitstream.ensure(bs_bytes + 16);
  d_params.ensure(params_bytes);
  d_tu.ensure(tu_words * 4);
  if (tu_words >= (1ull << 31)) bail(HEIC_E_UNSUPPORTED, "batch too large: more than 2^31 4x4 blocks in one load");
  d_list.ensure(transform_list_layout(tu_words, list_off) * sizeof(uint2_t));
  d_list_count.ensure(LIST_CLASSES * LIST_COUNT_STRIDE * sizeof(uint32_t));
  if (coeff_elems * 2 > d_coeff.cap) coeff_clean = false;  // a fresh allocation is not zero
  d_coeff.ensure(coeff_elems * 2);
  d_recon.ensure(plane_bytes);
  d_final.ensure(plane_bytes);
  d_ipm.ensure(map4_bytes);
  d_ctd.ensure(map8_bytes);
  d_qp.ensure(map8_bytes);
  d_sao.ensure(sao_words * 4);
  d_wpp.ensure(wpp_bytes);
  d_status.ensure(tiles.size() * sizeof(TileStatusDev));
  h_status.ensure(tiles.size() * sizeof(TileStatusDev));
  if (with_rgb) {
    src_off = up(rgb_image_stride * images.size(), 256);
    tmp_off = up(src_off + src_image_stride * n_src, 256);
    d_rgb.ensure(tmp_off + tmp_bytes);
  }
  d_raw.ensure(raw_bytes ? raw_bytes + 16 : 0);
  if (any_plain) CU(cudaMemcpyAsync(d_bitstream.p, h_bitstream.p, bs_bytes + 16, cudaMemcpyHostToDevice, st));
  if (raw_bytes) CU(cudaMemcpyAsync(d_raw.p, h_raw.p, raw_bytes + 16, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d_params.p, h_params.p, params_bytes, cudaMemcpyHostToDevice, st));
}

// Source arena, coefficient tables and launch runs of the resized images of a load.  The colour stage writes a resized
// image into the source arena at its full (oriented, reduced) size, and the resampling passes write d_rgb.  Tables are
// shared by every image and axis with the same (input size, output size, filter).
void heic_b200_batch::plan_resample() {
  rs_runs.clear();
  rs_axes.clear();
  rs_tables.clear();
  src_pitch = src_image_stride = n_src = tmp_bytes = 0;
  size_t max_rows = 0;
  for (ImageInfo& im : images) {
    if (!im.filter) continue;
    im.src_slot = (uint32_t)n_src++;
    src_pitch = std::max(src_pitch, up((size_t)im.color_w * 3, 16));
    max_rows = std::max(max_rows, (size_t)im.color_h);
  }
  if (!n_src) return;
  src_image_stride = up(src_pitch * max_rows, 256);
  std::map<std::tuple<uint32_t, uint32_t, uint32_t>, int> by_key;
  auto table = [&](uint32_t n_in, uint32_t n_out, uint32_t filter) -> int {
    const auto key = std::make_tuple(n_in, n_out, filter);
    const auto it = by_key.find(key);
    if (it != by_key.end()) return it->second;
    ResampleTable t;
    resample_coeffs(n_in, n_out, filter, t);
    ResampleTableRef ref;
    std::memset(&ref, 0, sizeof ref);
    ref.ax.n_out = n_out;
    ref.ax.n_bands = (n_out + kResampleBand - 1) / kResampleBand;
    ref.row0 = (uint32_t)t.xmin[0];
    ref.row_end = (uint32_t)(t.xmin[n_out - 1] + t.n[n_out - 1]);
    // every part is a multiple of 4 words: the int4 entries and the coefficient bands start at 16-byte boundaries
    ref.o_out = rs_tables.size();
    ref.o_band = ref.o_out + 4 * (size_t)n_out;
    ref.o_coef = ref.o_band + 4 * (size_t)ref.ax.n_bands;
    rs_tables.resize(ref.o_coef, 0);
    for (uint32_t b = 0; b < ref.ax.n_bands; b++) {
      const uint32_t j0 = b * kResampleBand, j1 = std::min(n_out, j0 + kResampleBand);
      int32_t taps = 0, end = 0;
      for (uint32_t j = j0; j < j1; j++) taps = std::max(taps, t.n[j]), end = std::max(end, t.xmin[j] + t.n[j]);
      const size_t cb = rs_tables.size();
      rs_tables.resize(cb + (size_t)taps * kResampleBand, 0);
      for (uint32_t j = j0; j < j1; j++) {
        for (int32_t x = 0; x < t.n[j]; x++) rs_tables[cb + (size_t)x * kResampleBand + (j - j0)] = t.coeffs[t.off[j] + x];
        int32_t* e = &rs_tables[ref.o_out + 4 * (size_t)j];
        e[0] = t.xmin[j];
        e[1] = t.n[j];
        e[2] = (int32_t)(cb - ref.o_coef + (j - j0));
      }
      const int32_t x0 = t.xmin[j0];
      int32_t* e = &rs_tables[ref.o_band + 4 * (size_t)b];
      e[0] = x0;
      e[1] = end - x0;
      e[2] = taps;
      e[3] = (int32_t)(cb - ref.o_coef);
      ref.ax.max_taps = std::max(ref.ax.max_taps, (uint32_t)taps);
      // resample_h_kernel's row buffer holds the span from its 16-byte aligned start, and the band's last output reads
      // `taps` pixels from its xmin
      const size_t lead = (3u * (uint32_t)x0) & 15u;
      const size_t need = std::max(lead + 3 * (size_t)(t.xmin[j1 - 1] - x0 + taps), lead + 3 * (size_t)(end - x0) + 15);
      ref.ax.max_row_bytes = std::max(ref.ax.max_row_bytes, (uint32_t)up(need, 16));
    }
    rs_axes.push_back(ref);
    return by_key[key] = (int)rs_axes.size() - 1;
  };
  for (size_t i = 0; i < images.size();) {
    if (!images[i].filter) {
      i++;
      continue;
    }
    const ImageInfo& im = images[i];
    size_t j = i + 1;
    while (j < images.size() && images[j].filter == im.filter && images[j].color_w == im.color_w &&
           images[j].color_h == im.color_h && images[j].rgb_w == im.rgb_w && images[j].rgb_h == im.rgb_h)
      j++;
    ResampleRun r;
    r.first = (uint32_t)i;
    r.count = (uint32_t)(j - i);
    r.h_table = im.rgb_w != im.color_w ? table(im.color_w, im.rgb_w, im.filter) : -1;
    r.v_table = im.rgb_h != im.color_h ? table(im.color_h, im.rgb_h, im.filter) : -1;
    r.row0 = 0;
    r.rows = im.color_h;
    if (r.v_table >= 0) r.row0 = rs_axes[r.v_table].row0, r.rows = rs_axes[r.v_table].row_end - r.row0;
    r.tmp_off = tmp_bytes;
    r.tmp_pitch = up((size_t)im.rgb_w * 3, 16);
    r.tmp_stride = up(r.tmp_pitch * r.rows, 256);
    if (r.h_table >= 0 && r.v_table >= 0) tmp_bytes += r.tmp_stride * r.count;
    rs_runs.push_back(r);
    i = j;
  }
}

// ---- stage sequencing ----------------------------------------------------------------------------------
void heic_b200_batch::run(uint32_t mask) {
  cudaStream_t st = stream;
  const Arenas A = arenas();
  if (!A.n_tiles) return;
  if (mask & HEIC_STAGE_CABAC) {
    // tu_map must be zero outside transform-unit origins, levels zero outside significant coefficients
    CU(cudaMemsetAsync(d_tu.p, 0, tu_words * 4, st));
    if (!coeff_clean) CU(cudaMemsetAsync(d_coeff.p, 0, coeff_elems * 2, st));
    coeff_clean = false;
    CU(cudaMemsetAsync(d_status.p, 0, tiles.size() * sizeof(TileStatusDev), st));
    CU(cudaMemsetAsync(d_sao.p, 0, sao_words * 4, st));  // slices without SAO parse no parameters
    if (raw_bytes) {  // tiles shipped raw: emulation-prevention removal + entry-point re-basing (a no-op once done)
      uint8_t* pb = (uint8_t*)d_params.p;
      CU(launch_unescape(A, (TileParams*)(pb + off_tiles), (uint32_t*)(pb + off_sub), st));
      ctx->launches++;
    }
    constexpr size_t kCounters = 64;  // one group counter per launch class (persistent CABAC CTAs)
    d_counters.ensure(kCounters * sizeof(uint32_t));
    const bool persistent = ctx->cabac_persistent && classes.size() <= kCounters;
    if (persistent) CU(cudaMemsetAsync(d_counters.p, 0, kCounters * sizeof(uint32_t), st));
    size_t ci = 0;
    for (const CabacClass& c : classes) {
      CU(launch_cabac(A, ctx->d_tabs, (const uint32_t*)((const uint8_t*)d_params.p + off_order) + c.order_off, c.n_groups, tiles_per_cta,
                      c.n_slots, (persistent && c.hctb > c.n_slots) ? (uint32_t*)d_counters.p + ci : nullptr, ctx->n_sm, ctx->cabac_resident, st));
      ctx->launches++;
      ci++;
    }
  }
  if (mask & HEIC_STAGE_TRANSFORM) {
    CU(launch_transform(A, max_tu, max_log2_tb, ctx->n_sm, st));
    ctx->launches += transform_launches(max_log2_tb);
  }
  if (mask & HEIC_STAGE_INTRA) {
    // enough pictures to fill the GPU with one warp each: drop the intra-picture wavefront (no waiting at all)
    int slots = tiles.size() >= (size_t)ctx->intra_single_warp_tiles ? 1 : intra_slots;
    if (ctx->intra_slots > 0) slots = std::min(ctx->intra_slots, std::max(1, max_hctb));
    CU(launch_intra(A, (const uint32_t*)((const uint8_t*)d_params.p + off_heavy), max_log2_ctb, max_hctb, slots, true, st));
    coeff_clean = true;
    ctx->launches++;
  }
  if (mask & HEIC_STAGE_DEBLOCK) {
    CU(launch_deblock(A, max_w, max_h, st));
    ctx->launches += 2;  // luma + chroma
  }
  const bool fuse = ctx->fuse_sao && (mask & HEIC_STAGE_SAO) && (mask & HEIC_STAGE_COLOR) && d_rgb.p;
  if ((mask & HEIC_STAGE_SAO) && !fuse) {
    CU(launch_sao(A, max_pitch, max_h, st));
    final_stale = false;
    ctx->launches++;
  }
  if (fuse) {
    // SAO for the few CTBs that have it on, into the final arena; the colour kernel picks per CTB and component
    CU(launch_sao_sparse(A, max_hctb, st));
    ctx->launches++;
    final_stale = true;
  }
  if ((mask & HEIC_STAGE_COLOR) && d_rgb.p) {
    // consecutive images of identical geometry go out in one launch
    size_t i = 0;
    while (i < images.size()) {
      size_t j = i + 1;
      auto same = [&](const ImageInfo& a, const ImageInfo& b) {
        return a.pic == b.pic && a.n_tiles == b.n_tiles && a.grid_cols == b.grid_cols && a.canvas_w == b.canvas_w &&
               a.canvas_h == b.canvas_h && a.tile_w == b.tile_w && a.tile_h == b.tile_h && a.win_x == b.win_x && a.win_y == b.win_y &&
               a.crop_x == b.crop_x && a.crop_y == b.crop_y && a.crop_w == b.crop_w && a.crop_h == b.crop_h &&
               a.orientation == b.orientation && a.full_range == b.full_range && a.matrix_coeffs == b.matrix_coeffs &&
               a.reduce == b.reduce && (a.filter != 0) == (b.filter != 0);
      };
      while (j < images.size() && same(images[i], images[j])) j++;
      const ImageInfo& im = images[i];
      const PicParams& pp = pics[im.pic];
      const TileParams& t0 = tiles[im.first_tile];
      ColorJob job;
      job.planes = (const uint8_t*)(fuse ? d_recon.p : d_final.p) + t0.plane_off[0];
      job.fused = fuse ? 1u : 0u;
      job.planes_sao = (const uint8_t*)d_final.p + t0.plane_off[0];
      job.sao = A.sao + t0.sao_off;
      job.sao_stride = (uint32_t)((size_t)pp.wctb * pp.hctb * 4);
      job.log2_ctb = (uint32_t)pp.log2_ctb;
      job.wctb = (uint32_t)pp.wctb;
      job.tile_stride = im.n_tiles > 1 || j - i > 1
                            ? (size_t)(tiles[std::min<size_t>(im.first_tile + 1, tiles.size() - 1)].plane_off[0] - t0.plane_off[0])
                            : 0;
      job.cb_off = t0.plane_off[1] - t0.plane_off[0];
      job.cr_off = t0.plane_off[2] - t0.plane_off[0];
      job.pitch_y = (uint32_t)pp.pitch_y;
      job.pitch_c = (uint32_t)pp.pitch_c;
      job.tile_w = im.tile_w;
      job.tile_h = im.tile_h;
      job.grid_cols = im.grid_cols;
      job.grid_rows = im.grid_rows;
      job.out_w = im.canvas_w;
      job.out_h = im.canvas_h;
      job.n_images = (uint32_t)(j - i);
      job.chroma = (uint32_t)pp.chroma;
      job.full_range = im.full_range;
      job.matrix_coeffs = im.matrix_coeffs;
      job.orientation = im.orientation;
      if (im.filter) {  // resized: the source arena, where consecutive resized images have consecutive slots
        job.rgb = (uint8_t*)d_rgb.p + src_off + (size_t)im.src_slot * src_image_stride;
        job.pitch = src_pitch;
        job.image_stride = src_image_stride;
      } else {
        job.rgb = (uint8_t*)d_rgb.p + i * rgb_image_stride;
        job.pitch = rgb_pitch;
        job.image_stride = rgb_image_stride;
      }
      const ColorWindow win = {im.crop_x, im.crop_y, im.crop_w, im.crop_h, im.win_x, im.win_y};
      CU(launch_color(job, win, im.reduce, st));
      ctx->launches++;
      i = j;
    }
    // resampling: horizontal pass first (into the intermediate when the vertical pass follows), then vertical, per run of images
    const uint8_t* tabs = (const uint8_t*)d_params.p + off_resample;
    auto axis = [&](int t) {
      ResampleAxis a = rs_axes[t].ax;
      a.out = (const int4*)(tabs + rs_axes[t].o_out * 4);
      a.band = (const int4*)(tabs + rs_axes[t].o_band * 4);
      a.coeffs = (const int32_t*)(tabs + rs_axes[t].o_coef * 4);
      return a;
    };
    for (const ResampleRun& r : rs_runs) {
      const ImageInfo& im = images[r.first];
      ResampleJob rj;
      rj.src = (const uint8_t*)d_rgb.p + src_off + (size_t)im.src_slot * src_image_stride;
      rj.src_pitch = src_pitch;
      rj.src_image_stride = src_image_stride;
      rj.n_images = r.count;
      rj.out_w = im.rgb_w;
      uint8_t* out = (uint8_t*)d_rgb.p + (size_t)r.first * rgb_image_stride;
      const bool two = r.h_table >= 0 && r.v_table >= 0;
      if (r.h_table >= 0) {
        rj.dst = two ? (uint8_t*)d_rgb.p + tmp_off + r.tmp_off : out;
        rj.dst_pitch = two ? r.tmp_pitch : rgb_pitch;
        rj.dst_image_stride = two ? r.tmp_stride : rgb_image_stride;
        rj.rows = r.rows;
        rj.row0 = r.row0;
        CU(launch_resample_h(rj, axis(r.h_table), st));
        ctx->launches++;
      }
      if (r.v_table >= 0) {
        if (two) {  // the intermediate starts at the first used row: the vertical bounds shift by it
          rj.src = rj.dst;
          rj.src_pitch = rj.dst_pitch;
          rj.src_image_stride = rj.dst_image_stride;
        }
        rj.dst = out;
        rj.dst_pitch = rgb_pitch;
        rj.dst_image_stride = rgb_image_stride;
        rj.rows = im.rgb_h;
        rj.row0 = two ? r.row0 : 0;
        CU(launch_resample_v(rj, axis(r.v_table), st));
        ctx->launches++;
      }
    }
  }
  stages_run |= mask;
}

// ---- C ABI ---------------------------------------------------------------------------------------------
namespace {

// The host copy of the device status of n tiles in the C ABI's form.
void convert_status(const TileStatusDev* s, size_t n, heic_tile_status* out) {
  for (size_t i = 0; i < n; i++) {
    out[i].code = s[i].code;
    out[i].bins_decoded = s[i].bins;
    out[i].ctus_decoded = s[i].ctus;
    out[i].reserved = 0;
  }
}

void collect_status(heic_b200_batch* b, heic_tile_status* status) {
  cudaStream_t st = b->stream;
  const size_t n = b->tiles.size();
  CU(cudaMemcpyAsync(b->h_status.p, b->d_status.p, n * sizeof(TileStatusDev), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  convert_status((const TileStatusDev*)b->h_status.p, n, status);
}

// The caller's RGB layout for one of n_imgs images: rows of at least rgb_w * 3 bytes and, with more than one image, an
// image stride that holds its rows.
void check_rgb_layout(const ImageInfo& im, size_t pitch, size_t image_stride, size_t n_imgs) {
  if (pitch < (size_t)im.rgb_w * 3) bail(HEIC_E_INVALID_ARG, "output pitch smaller than a row of RGB");
  if (n_imgs > 1 && (size_t)im.rgb_h * pitch > image_stride) bail(HEIC_E_INVALID_ARG, "image_stride smaller than one image (rows x pitch)");
}

// Queues on the batch's stream the device->host copy of the RGB of images [first, first + n) to dst, image i at
// dst + (i - first) * image_stride.  When the caller's layout is the batch's and leaves no padding, that is one copy.
void queue_rgb_download(const heic_b200_batch* b, size_t first, size_t n, uint8_t* dst, size_t pitch, size_t image_stride) {
  const uint8_t* src = (const uint8_t*)b->d_rgb.p + first * b->rgb_image_stride;
  bool one_copy = image_stride == b->rgb_image_stride && pitch == b->rgb_pitch;
  for (size_t i = first; i < first + n && one_copy; i++)
    one_copy = (size_t)b->images[i].rgb_w * 3 == pitch && (size_t)b->images[i].rgb_h * pitch == image_stride;
  if (one_copy) {
    CU(cudaMemcpyAsync(dst, src, n * image_stride, cudaMemcpyDeviceToHost, b->stream));
    return;
  }
  for (size_t i = first; i < first + n; i++) {
    const ImageInfo& im = b->images[i];
    CU(cudaMemcpy2DAsync(dst + (i - first) * image_stride, pitch, src + (i - first) * b->rgb_image_stride, b->rgb_pitch,
                         (size_t)im.rgb_w * 3, im.rgb_h, cudaMemcpyDeviceToHost, b->stream));
  }
}

}  // namespace

extern "C" {

int32_t heic_b200_create(int32_t device, heic_b200_ctx** out_ctx) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!out_ctx) bail(HEIC_E_INVALID_ARG, "null argument");
    *out_ctx = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
      bail(HEIC_E_NO_DEVICE, std::string("no CUDA device (this library has no CPU path): ") + cudaGetErrorString(e));
    auto c = std::make_unique<heic_b200_ctx>();
    if (device < 0) CU(cudaGetDevice(&c->device));
    else c->device = device;
    CU(cudaSetDevice(c->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, c->device));
    if (prop.major < 10)
      bail(HEIC_E_NO_DEVICE, std::string("device '") + prop.name + "' is not sm_100 class; the kernels are built for sm_100a only");
    CU(cudaDeviceGetAttribute(&c->n_sm, cudaDevAttrMultiProcessorCount, c->device));
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    static CabacTabs tabs;
    build_cabac_tabs(tabs);
    CU(cudaMalloc((void**)&c->d_tabs, sizeof(CabacTabs)));
    CU(cudaMemcpy(c->d_tabs, &tabs, sizeof tabs, cudaMemcpyHostToDevice));
    c->cabac_tiles_per_cta = env_int("HEIC_B200_CABAC_TILES_PER_CTA", 32) == 1 ? 1 : 32;
    c->cabac_slots = env_int("HEIC_B200_CABAC_SLOTS", 0);
    c->intra_slots = std::min(8, env_int("HEIC_B200_INTRA_SLOTS", 0));
    c->pipe_chunk = std::max(0, env_int("HEIC_B200_PIPE_CHUNK", 0));
    c->low_latency_tiles = env_int("HEIC_B200_LOW_LATENCY_TILES", 384);
    c->fuse_sao = env_int("HEIC_B200_FUSE_SAO", 1) != 0;
    c->cabac_persistent = env_int("HEIC_B200_CABAC_PERSISTENT", 1) != 0;
    c->cabac_resident = std::max(0, env_int("HEIC_B200_CABAC_RESIDENT", 0));
    c->cabac_plain_sort = env_int("HEIC_B200_CABAC_PLAIN_SORT", 0) != 0;
    c->pipe_slots = std::min((int)heic_b200_ctx::kPipe, std::max(0, env_int("HEIC_B200_PIPE_SLOTS", 0)));
    c->pipe_order = env_int("HEIC_B200_PIPE_ORDER", 1) != 0;
    *out_ctx = c.release();
    return 0;
  }));
}

void heic_b200_destroy(heic_b200_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  if (ctx->stream) cudaStreamSynchronize(ctx->stream);
  delete ctx;
}

uint64_t heic_b200_launch_count(const heic_b200_ctx* ctx) { return ctx ? ctx->launches : 0; }

int32_t heic_b200_batch_create(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs, heic_b200_batch** out) {
  return heic_b200_batch_create_ex(ctx, imgs, n_imgs, 0, out);
}

static int64_t batch_create(heic_b200_ctx* ctx, const heic_image_desc* imgs, const OutputSpec* specs, uint32_t n_imgs,
                            heic_b200_batch** out) {
  if (!ctx || !imgs || !out || !n_imgs) bail(HEIC_E_INVALID_ARG, "null argument");
  *out = nullptr;
  CU(cudaSetDevice(ctx->device));
  std::vector<ImagePlan> plans(n_imgs);
  for (uint32_t i = 0; i < n_imgs; i++) plans[i] = plan_image(imgs[i], specs[i], true);
  auto b = std::make_unique<heic_b200_batch>();
  b->ctx = ctx;
  b->stream = ctx->stream;
  b->load(imgs, plans.data(), n_imgs, true);
  CU(cudaStreamSynchronize(ctx->stream));
  *out = b.release();
  return 0;
}

int32_t heic_b200_batch_create_ex(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs, int32_t apply_transforms,
                                  heic_b200_batch** out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!ctx || !imgs || !out || !n_imgs) bail(HEIC_E_INVALID_ARG, "null argument");
    *out = nullptr;
    return batch_create(ctx, imgs, output_specs(imgs, n_imgs, nullptr, nullptr, nullptr, apply_transforms).data(), n_imgs, out);
  }));
}

int32_t heic_b200_batch_create_transformed(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                           uint32_t n_imgs, heic_b200_batch** out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!xforms) bail(HEIC_E_INVALID_ARG, "null argument");
    return batch_create(ctx, imgs, output_specs(imgs, n_imgs, xforms, nullptr, nullptr, 0).data(), n_imgs, out);
  }));
}

int32_t heic_b200_batch_create_reduced(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                       const uint32_t* reduce, uint32_t n_imgs, heic_b200_batch** out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!xforms || !reduce) bail(HEIC_E_INVALID_ARG, "null argument");
    return batch_create(ctx, imgs, output_specs(imgs, n_imgs, xforms, reduce, nullptr, 0).data(), n_imgs, out);
  }));
}

int32_t heic_b200_batch_create_resized(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                       const uint32_t* reduce, const heic_resize* resize, uint32_t n_imgs, heic_b200_batch** out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!xforms || !reduce || !resize) bail(HEIC_E_INVALID_ARG, "null argument");
    return batch_create(ctx, imgs, output_specs(imgs, n_imgs, xforms, reduce, resize, 0).data(), n_imgs, out);
  }));
}

void heic_b200_batch_destroy(heic_b200_batch* b) {
  if (!b) return;
  cudaSetDevice(b->ctx->device);
  cudaStreamSynchronize(b->stream);
  delete b;
}

int32_t heic_b200_batch_run_stages(heic_b200_batch* b, uint32_t stage_mask) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!b) bail(HEIC_E_INVALID_ARG, "null batch");
    CU(cudaSetDevice(b->ctx->device));
    b->run(stage_mask & HEIC_STAGE_ALL);
    return 0;
  }));
}

int32_t heic_b200_batch_decode(heic_b200_batch* b) { return heic_b200_batch_run_stages(b, HEIC_STAGE_ALL); }

int32_t heic_b200_batch_sync(heic_b200_batch* b) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!b) bail(HEIC_E_INVALID_ARG, "null batch");
    CU(cudaStreamSynchronize(b->stream));
    return 0;
  }));
}

void* heic_b200_batch_stream(heic_b200_batch* b) { return b ? (void*)b->stream : nullptr; }

int32_t heic_b200_batch_rgb(heic_b200_batch* b, void** dev_ptr, size_t* pitch, size_t* image_stride) {
  if (!b) {
    set_last_error("null batch");
    return HEIC_E_INVALID_ARG;
  }
  if (dev_ptr) *dev_ptr = b->d_rgb.p;
  if (pitch) *pitch = b->rgb_pitch;
  if (image_stride) *image_stride = b->rgb_image_stride;
  return 0;
}

int32_t heic_b200_batch_download_rgb(heic_b200_batch* b, uint8_t* rgb_out, size_t pitch, size_t image_stride) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!b || !rgb_out) bail(HEIC_E_INVALID_ARG, "null argument");
    CU(cudaSetDevice(b->ctx->device));
    // validate the whole layout before the first copy is queued
    for (const ImageInfo& im : b->images) check_rgb_layout(im, pitch, image_stride, b->images.size());
    queue_rgb_download(b, 0, b->images.size(), rgb_out, pitch, image_stride);
    CU(cudaStreamSynchronize(b->stream));
    return 0;
  }));
}

// One image of a resident batch (bench.py / tools: pixel checks at batch sizes whose whole RGB output would not fit the host).
int32_t heic_b200_batch_download_image(heic_b200_batch* b, uint32_t image_index, uint8_t* rgb_out, size_t pitch) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!b || !rgb_out || image_index >= b->images.size()) bail(HEIC_E_INVALID_ARG, "invalid argument");
    if (!b->d_rgb.p) bail(HEIC_E_INVALID_ARG, "the batch has no RGB output");
    CU(cudaSetDevice(b->ctx->device));
    check_rgb_layout(b->images[image_index], pitch, 0, 1);
    queue_rgb_download(b, image_index, 1, rgb_out, pitch, 0);
    CU(cudaStreamSynchronize(b->stream));
    return 0;
  }));
}

int32_t heic_b200_batch_status(heic_b200_batch* b, heic_tile_status* status) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!b || !status) bail(HEIC_E_INVALID_ARG, "null argument");
    CU(cudaSetDevice(b->ctx->device));
    collect_status(b, status);
    return 0;
  }));
}

uint32_t heic_b200_batch_tile_count(const heic_b200_batch* b) { return b ? (uint32_t)b->tiles.size() : 0; }

// CABAC launch order of a resident batch: tile indices, 32 per warp-group in the thread-per-substream mapping
// (0xffffffff = idle lane).  Returns the number of entries; copies at most `cap` of them.  For tools and bench.py, which
// checks that no warp holds two copies of one tile.
size_t heic_b200_batch_cabac_order(const heic_b200_batch* b, uint32_t* out, size_t cap, uint32_t* tiles_per_group) {
  if (!b) return 0;
  if (tiles_per_group) *tiles_per_group = (uint32_t)b->tiles_per_cta;
  if (out)
    for (size_t i = 0; i < b->order.size() && i < cap; i++) out[i] = b->order[i];
  return b->order.size();
}

int32_t heic_b200_batch_dump_tile(heic_b200_batch* b, uint32_t tile_index, heic_tile_dump* dump) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!b || !dump || tile_index >= b->tiles.size()) bail(HEIC_E_INVALID_ARG, "invalid argument");
    CU(cudaSetDevice(b->ctx->device));
    cudaStream_t st = b->stream;
    CU(cudaStreamSynchronize(st));
    const TileParams& tp = b->tiles[tile_index];
    const PicParams& pp = b->pics[tp.pic];
    if (dump->tu_map) {
      if (dump->tu_map_len < (uint32_t)pp.n_tu) bail(HEIC_E_INVALID_ARG, "tu_map buffer too small");
      CU(cudaMemcpy(dump->tu_map, (const uint32_t*)b->d_tu.p + tp.tu_off, (size_t)pp.n_tu * 4, cudaMemcpyDeviceToHost));
    }
    for (int c = 0; c < (pp.chroma ? 3 : 1); c++)
      if (dump->coeff[c]) {
        const size_t n = (size_t)pp.n_tu * (c ? 4 : 16);
        if (dump->coeff_len[c] < n) bail(HEIC_E_INVALID_ARG, "coefficient buffer too small");
        CU(cudaMemcpy(dump->coeff[c], (const int16_t*)b->d_coeff.p + tp.coeff_off[c], n * 2, cudaMemcpyDeviceToHost));
      }
    if (dump->qp_map) {
      const size_t wq = (size_t)pp.w >> 3, hq = (size_t)pp.h >> 3;
      if (dump->qp_map_len < wq * hq) bail(HEIC_E_INVALID_ARG, "qp_map buffer too small");
      CU(cudaMemcpy2D(dump->qp_map, wq, (const uint8_t*)b->d_qp.p + tp.map8_off, (size_t)pp.w8, wq, hq, cudaMemcpyDeviceToHost));
    }
    if (dump->sao) {
      const size_t n = (size_t)pp.wctb * pp.hctb * 4;
      if (dump->sao_len < n) bail(HEIC_E_INVALID_ARG, "sao buffer too small");
      CU(cudaMemcpy(dump->sao, (const uint32_t*)b->d_sao.p + tp.sao_off, n * 4, cudaMemcpyDeviceToHost));
    }
    if ((b->stages_run & HEIC_STAGE_SAO) && b->final_stale) {  // SAO was applied inside the colour kernel: write the planes now
      CU(launch_sao(b->arenas(), b->max_pitch, b->max_h, b->stream));
      CU(cudaStreamSynchronize(b->stream));
      b->final_stale = false;
    }
    const uint8_t* src = (const uint8_t*)((b->stages_run & HEIC_STAGE_SAO) ? b->d_final.p : b->d_recon.p);
    for (int c = 0; c < (pp.chroma ? 3 : 1); c++)
      if (dump->plane[c]) {
        const size_t w = (size_t)pp.w >> (c ? 1 : 0), h = (size_t)pp.h >> (c ? 1 : 0);
        if (dump->plane_len[c] < w * h) bail(HEIC_E_INVALID_ARG, "plane buffer too small");
        CU(cudaMemcpy2D(dump->plane[c], w, src + tp.plane_off[c], (size_t)(c ? pp.pitch_c : pp.pitch_y), w, h,
                        cudaMemcpyDeviceToHost));
      }
    return 0;
  }));
}

// HOST in / HOST out: the reference-facing call (replaces the tile loop of decoder.rs:98-119).
// The images are processed in chunks that rotate over kPipe (stream, scratch batch) slots: while chunk k's RGB
// travels to the host, chunk k+1 runs its kernels and chunk k+2's slice data travels to the device.  Output buffers
// should be pinned host memory; pageable memory works but its copies are staged synchronously.
static void harvest_slot(heic_b200_ctx* ctx, int slot) {
  PipePending& pd = ctx->pipe_pending[slot];
  if (!pd.job) return;
  heic_b200_batch* b = ctx->pipe_batch[slot].get();
  CU(cudaStreamSynchronize(b->stream));
  if (pd.ev[0] && ctx->trace_base) {
    float t[5];
    for (int k = 0; k < 5; k++) cudaEventElapsedTime(&t[k], ctx->trace_base, pd.ev[k]);
    std::fprintf(stderr, "[heic_b200] chunk slot %2d tiles %6zu: queued %8.1f  h2d %8.1f  cabac %8.1f  kernels %8.1f  d2h %8.1f ms\n", slot,
                 pd.n_tiles, t[0], t[1], t[2], t[3], t[4]);
  }
  convert_status((const TileStatusDev*)b->h_status.p, pd.n_tiles, pd.job->status + pd.tile0);
  pd.job = nullptr;
}

// specs: one output per image (RGB output; the planar output applies no transform)
static heic_b200_job* submit_grids(heic_b200_ctx* ctx, const heic_image_desc* imgs, const OutputSpec* specs, uint32_t n_imgs,
                                   uint8_t* rgb_out, size_t pitch, size_t image_stride, uint8_t* y_out, uint8_t* cb_out,
                                   uint8_t* cr_out, heic_tile_status* status) {
  if (!ctx || !imgs || !n_imgs) bail(HEIC_E_INVALID_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  // plan every image, and check the caller's buffer layout for it, before any work is queued, so a bad image rejects the
  // call as a whole
  std::vector<ImagePlan> plans(n_imgs);
  std::vector<size_t> first_tile(n_imgs + 1, 0), y_off(n_imgs + 1, 0), c_off(n_imgs + 1, 0);
  for (uint32_t i = 0; i < n_imgs; i++) {
    plans[i] = plan_image(imgs[i], specs[i], rgb_out != nullptr);
    const ImageInfo& im = plans[i].info;
    if (rgb_out) check_rgb_layout(im, pitch, image_stride, n_imgs);
    const size_t cw = im.canvas_w, ch = im.canvas_h;
    first_tile[i + 1] = first_tile[i] + im.n_tiles;
    y_off[i + 1] = y_off[i] + cw * ch;
    c_off[i + 1] = c_off[i] + ((cw + 1) / 2) * ((ch + 1) / 2);
  }
  static const bool trace = std::getenv("HEIC_B200_TRACE") != nullptr;  // host-side phase times of a submit, to stderr
  static const bool trace2 = trace && std::atoi(std::getenv("HEIC_B200_TRACE")) >= 2;  // + the device timeline of every chunk
  using clk = std::chrono::steady_clock;
  auto ms_since = [](clk::time_point t0) { return std::chrono::duration<double, std::milli>(clk::now() - t0).count(); };
  const clk::time_point t_call = clk::now();
  double t_wait = 0, t_load = 0, t_run = 0;
  auto job = std::make_unique<heic_b200_job>();
  job->ctx = ctx;
  job->n_tiles = first_tile[n_imgs];
  job->status = status;
  if (!job->status) {
    job->local.resize(job->n_tiles);
    job->status = job->local.data();
  }
  // equal chunks (a ramp of small first chunks was measured slower: every chunk pays the CABAC latency floor of its
  // heaviest tiles while holding a pipeline slot)
  // Chunk size.  The CABAC stage is latency-bound per 32-tile group (a group lasts as long as its heaviest tile's critical
  // path, ~100 ms for a 70 KB slice), so a chunk only uses the machine when it brings about as many groups as CTAs are
  // resident (444 groups = 296 images of 48 tiles): measured on B200, eight 32-image chunks in flight decode at 10.4 K MP/s,
  // one 256-image chunk per call, double-buffered, at the speed of a resident 256-image batch.  So by default a call is cut
  // into equal chunks of at most 296 images, and three such chunks rotate: one in its kernels, one in its D2H copy and one
  // being staged by the host (with two, the GPU idled while the host staged the next chunk behind a finished copy);
  // HEIC_B200_PIPE_CHUNK / _SLOTS override.
  uint32_t chunk = (uint32_t)std::max(0, ctx->pipe_chunk);
  if (chunk == 0) {
    const uint32_t parts = (n_imgs + 295u) / 296u;
    chunk = (n_imgs + parts - 1) / parts;
  }
  const uint32_t n_slots_use = ctx->pipe_slots > 0 ? (uint32_t)ctx->pipe_slots : std::min(8u, std::max(3u, 900u / chunk));
  std::vector<uint32_t> chunk_start;
  for (uint32_t i = 0; i < n_imgs; i += chunk) chunk_start.push_back(i);
  chunk_start.push_back(n_imgs);
  const uint32_t n_chunks = (uint32_t)chunk_start.size() - 1;
  try {
  for (uint32_t k = 0; k < n_chunks; k++) {
    const int slot = (int)(ctx->pipe_next++ % n_slots_use);
    const uint32_t i0 = chunk_start[k], cnt = chunk_start[k + 1] - i0;
    if (!ctx->pipe_stream[slot]) CU(cudaStreamCreateWithFlags(&ctx->pipe_stream[slot], cudaStreamNonBlocking));
    if (!ctx->pipe_batch[slot]) {
      ctx->pipe_batch[slot] = std::make_unique<heic_b200_batch>();
      ctx->pipe_batch[slot]->ctx = ctx;
      ctx->pipe_batch[slot]->stream = ctx->pipe_stream[slot];
    }
    clk::time_point t0 = clk::now();
    harvest_slot(ctx, slot);  // the slot's previous chunk (kernels, copies, status) is complete before its buffers are reused
    t_wait += ms_since(t0);
    heic_b200_batch* b = ctx->pipe_batch[slot].get();
    cudaStream_t st = b->stream;
    t0 = clk::now();
    b->load(imgs + i0, plans.data() + i0, cnt, rgb_out != nullptr);
    t_load += ms_since(t0);
    t0 = clk::now();
    PipePending& pend = ctx->pipe_pending[slot];
    if (trace2) {
      if (!ctx->trace_base) {
        CU(cudaEventCreate(&ctx->trace_base));
        CU(cudaEventRecord(ctx->trace_base, st));
      }
      for (int e = 0; e < 5; e++)
        if (!pend.ev[e]) CU(cudaEventCreate(&pend.ev[e]));
      // (the H2D copies were queued by load(): "queued" is recorded behind them, so h2d - queued is not their duration;
      // the columns that matter are when CABAC, the other kernels and the D2H copy of this chunk END)
      CU(cudaEventRecord(pend.ev[0], st));
      CU(cudaEventRecord(pend.ev[1], st));
    }
    // Chunks in flight are kept in order on the device: a chunk's CABAC stage starts when the previous chunk's has ended
    // (so CABAC of chunk k+1 shares the GPU with the throughput kernels of chunk k, not with another latency-bound CABAC
    // stage), and its device->host copy starts when the previous chunk's has ended (each copy gets the whole link).  Left to
    // the hardware scheduler, the first chunk of a run took 390 ms to reach its copy instead of 140 (three chunks' kernels
    // interleaved) and the copy engine idled that long.
    if (ctx->pipe_order) {
      if (!ctx->ev_cabac) {
        CU(cudaEventCreateWithFlags(&ctx->ev_cabac, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&ctx->ev_d2h, cudaEventDisableTiming));
      } else {
        CU(cudaStreamWaitEvent(st, ctx->ev_cabac, 0));
      }
    }
    b->run(HEIC_STAGE_CABAC);
    if (ctx->pipe_order) CU(cudaEventRecord(ctx->ev_cabac, st));
    if (trace2) CU(cudaEventRecord(pend.ev[2], st));
    b->run((rgb_out ? HEIC_STAGE_ALL : (HEIC_STAGE_ALL & ~HEIC_STAGE_COLOR)) & ~HEIC_STAGE_CABAC);
    if (trace2) CU(cudaEventRecord(pend.ev[3], st));
    if (ctx->pipe_order && ctx->d2h_recorded) CU(cudaStreamWaitEvent(st, ctx->ev_d2h, 0));
    t_run += ms_since(t0);
    if (rgb_out) {
      queue_rgb_download(b, 0, cnt, rgb_out + (size_t)i0 * image_stride, pitch, image_stride);
    } else {
      // planar output: tile mosaic (each tile's conformance window) cropped to the canvas, images back to back
      for (size_t i = 0; i < b->images.size(); i++) {
        const ImageInfo& im = b->images[i];
        const PicParams& pp = b->pics[im.pic];
        const size_t yo = y_off[i0 + i], co = c_off[i0 + i];
        const size_t cw = (im.canvas_w + 1) / 2, chh = (im.canvas_h + 1) / 2;
        const uint8_t* fin = (const uint8_t*)b->d_final.p;
        for (uint32_t t = 0; t < im.n_tiles; t++) {
          const TileParams& tp = b->tiles[im.first_tile + t];
          const size_t tx = (size_t)(t % im.grid_cols) * im.tile_w, ty = (size_t)(t / im.grid_cols) * im.tile_h;
          if (tx >= im.canvas_w || ty >= im.canvas_h) continue;
          const size_t w = std::min<size_t>(im.tile_w, im.canvas_w - tx), h = std::min<size_t>(im.tile_h, im.canvas_h - ty);
          CU(cudaMemcpy2DAsync(y_out + yo + ty * im.canvas_w + tx, im.canvas_w,
                               fin + tp.plane_off[0] + (size_t)im.win_y * pp.pitch_y + im.win_x, pp.pitch_y, w, h,
                               cudaMemcpyDeviceToHost, st));
          if (pp.chroma && cb_out && cr_out) {  // 4:2:0: the window's offsets and sizes are even
            const size_t wc = std::min<size_t>(im.tile_w / 2, cw - tx / 2), hc = std::min<size_t>(im.tile_h / 2, chh - ty / 2);
            const size_t wo = (size_t)(im.win_y / 2) * pp.pitch_c + im.win_x / 2;
            CU(cudaMemcpy2DAsync(cb_out + co + (ty / 2) * cw + tx / 2, cw, fin + tp.plane_off[1] + wo, pp.pitch_c, wc, hc,
                                 cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpy2DAsync(cr_out + co + (ty / 2) * cw + tx / 2, cw, fin + tp.plane_off[2] + wo, pp.pitch_c, wc, hc,
                                 cudaMemcpyDeviceToHost, st));
          }
        }
      }
    }
    CU(cudaMemcpyAsync(b->h_status.p, b->d_status.p, b->tiles.size() * sizeof(TileStatusDev), cudaMemcpyDeviceToHost, st));
    if (ctx->pipe_order) {
      CU(cudaEventRecord(ctx->ev_d2h, st));
      ctx->d2h_recorded = true;
    }
    if (trace2) CU(cudaEventRecord(pend.ev[4], st));
    ctx->pipe_pending[slot].job = job.get();
    ctx->pipe_pending[slot].tile0 = first_tile[i0];
    ctx->pipe_pending[slot].n_tiles = b->tiles.size();
  }
  } catch (...) {
    // a chunk could not be queued: retire the chunks of this job that are already in flight, then report
    // (the failing chunk's slot has no pending entry yet but may already have copies queued into the caller's buffer:
    // drain every idle slot's stream as well)
    for (int slot = 0; slot < heic_b200_ctx::kPipe; slot++) {
      if (!ctx->pipe_stream[slot]) continue;
      if (ctx->pipe_pending[slot].job == job.get() || !ctx->pipe_pending[slot].job) cudaStreamSynchronize(ctx->pipe_stream[slot]);
      if (ctx->pipe_pending[slot].job == job.get()) ctx->pipe_pending[slot].job = nullptr;
    }
    throw;
  }
  if (trace)
    std::fprintf(stderr, "[heic_b200] submit %u images: %.1f ms on the host (slot wait %.1f, load %.1f, launch %.1f)\n", n_imgs,
                 ms_since(t_call), t_wait, t_load, t_run);
  return job.release();
}

static int64_t job_wait(heic_b200_job* job) {
  std::unique_ptr<heic_b200_job> owner(job);
  heic_b200_ctx* ctx = job->ctx;
  CU(cudaSetDevice(ctx->device));
  for (int slot = 0; slot < heic_b200_ctx::kPipe; slot++)
    if (ctx->pipe_pending[slot].job == job) harvest_slot(ctx, slot);
  size_t bad = 0;
  for (size_t i = 0; i < job->n_tiles; i++)
    if (job->status[i].code != 0) bad++;
  if (bad) {
    set_last_error(std::to_string(bad) + " tile(s) failed to decode (malformed slice data); see the per-tile status");
    return HEIC_E_BITSTREAM;
  }
  return 0;
}

static int64_t decode_grids_impl(heic_b200_ctx* ctx, const heic_image_desc* imgs, const OutputSpec* specs, uint32_t n_imgs,
                                 uint8_t* rgb_out, size_t pitch, size_t image_stride, uint8_t* y_out, uint8_t* cb_out,
                                 uint8_t* cr_out, heic_tile_status* status) {
  return job_wait(submit_grids(ctx, imgs, specs, n_imgs, rgb_out, pitch, image_stride, y_out, cb_out, cr_out, status));
}

int32_t heic_b200_decode_grids(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs, uint8_t* rgb_out,
                               size_t pitch, size_t image_stride, int32_t apply_transforms, heic_tile_status* status) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!ctx || !rgb_out) bail(HEIC_E_INVALID_ARG, "null argument");
    return decode_grids_impl(ctx, imgs, output_specs(imgs, n_imgs, nullptr, nullptr, nullptr, apply_transforms).data(), n_imgs,
                             rgb_out, pitch, image_stride, nullptr, nullptr, nullptr, status);
  }));
}

int32_t heic_b200_decode_grids_transformed(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                           uint32_t n_imgs, uint8_t* rgb_out, size_t pitch, size_t image_stride,
                                           heic_tile_status* status) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rgb_out) bail(HEIC_E_INVALID_ARG, "null output buffer");
    if (!xforms) bail(HEIC_E_INVALID_ARG, "null argument");
    return decode_grids_impl(ctx, imgs, output_specs(imgs, n_imgs, xforms, nullptr, nullptr, 0).data(), n_imgs, rgb_out, pitch,
                             image_stride, nullptr, nullptr, nullptr, status);
  }));
}

int32_t heic_b200_decode_grids_reduced(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                       const uint32_t* reduce, uint32_t n_imgs, uint8_t* rgb_out, size_t pitch, size_t image_stride,
                                       heic_tile_status* status) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rgb_out) bail(HEIC_E_INVALID_ARG, "null output buffer");
    if (!xforms || !reduce) bail(HEIC_E_INVALID_ARG, "null argument");
    return decode_grids_impl(ctx, imgs, output_specs(imgs, n_imgs, xforms, reduce, nullptr, 0).data(), n_imgs, rgb_out, pitch,
                             image_stride, nullptr, nullptr, nullptr, status);
  }));
}

int32_t heic_b200_decode_grids_resized(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                       const uint32_t* reduce, const heic_resize* resize, uint32_t n_imgs, uint8_t* rgb_out,
                                       size_t pitch, size_t image_stride, heic_tile_status* status) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rgb_out) bail(HEIC_E_INVALID_ARG, "null output buffer");
    if (!xforms || !reduce || !resize) bail(HEIC_E_INVALID_ARG, "null argument");
    return decode_grids_impl(ctx, imgs, output_specs(imgs, n_imgs, xforms, reduce, resize, 0).data(), n_imgs, rgb_out, pitch,
                             image_stride, nullptr, nullptr, nullptr, status);
  }));
}

int32_t heic_b200_decode_grids_submit(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs, uint8_t* rgb_out,
                                      size_t pitch, size_t image_stride, int32_t apply_transforms, heic_tile_status* status,
                                      heic_b200_job** out_job) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!ctx || !rgb_out || !out_job) bail(HEIC_E_INVALID_ARG, "null argument");
    *out_job = submit_grids(ctx, imgs, output_specs(imgs, n_imgs, nullptr, nullptr, nullptr, apply_transforms).data(), n_imgs,
                            rgb_out, pitch, image_stride, nullptr, nullptr, nullptr, status);
    return 0;
  }));
}

int32_t heic_b200_decode_grids_submit_transformed(heic_b200_ctx* ctx, const heic_image_desc* imgs,
                                                  const heic_image_transform* xforms, uint32_t n_imgs, uint8_t* rgb_out,
                                                  size_t pitch, size_t image_stride, heic_tile_status* status,
                                                  heic_b200_job** out_job) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rgb_out || !out_job || !xforms) bail(HEIC_E_INVALID_ARG, "null argument");
    *out_job = submit_grids(ctx, imgs, output_specs(imgs, n_imgs, xforms, nullptr, nullptr, 0).data(), n_imgs, rgb_out, pitch,
                            image_stride, nullptr, nullptr, nullptr, status);
    return 0;
  }));
}

int32_t heic_b200_decode_grids_submit_reduced(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                              const uint32_t* reduce, uint32_t n_imgs, uint8_t* rgb_out, size_t pitch,
                                              size_t image_stride, heic_tile_status* status, heic_b200_job** out_job) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rgb_out || !out_job || !xforms || !reduce) bail(HEIC_E_INVALID_ARG, "null argument");
    *out_job = submit_grids(ctx, imgs, output_specs(imgs, n_imgs, xforms, reduce, nullptr, 0).data(), n_imgs, rgb_out, pitch,
                            image_stride, nullptr, nullptr, nullptr, status);
    return 0;
  }));
}

int32_t heic_b200_decode_grids_submit_resized(heic_b200_ctx* ctx, const heic_image_desc* imgs, const heic_image_transform* xforms,
                                              const uint32_t* reduce, const heic_resize* resize, uint32_t n_imgs, uint8_t* rgb_out,
                                              size_t pitch, size_t image_stride, heic_tile_status* status, heic_b200_job** out_job) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!rgb_out || !out_job || !xforms || !reduce || !resize) bail(HEIC_E_INVALID_ARG, "null argument");
    *out_job = submit_grids(ctx, imgs, output_specs(imgs, n_imgs, xforms, reduce, resize, 0).data(), n_imgs, rgb_out, pitch,
                            image_stride, nullptr, nullptr, nullptr, status);
    return 0;
  }));
}

int32_t heic_b200_job_wait(heic_b200_job* job) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!job) bail(HEIC_E_INVALID_ARG, "null job");
    return job_wait(job);
  }));
}

int32_t heic_b200_decode_grids_yuv(heic_b200_ctx* ctx, const heic_image_desc* imgs, uint32_t n_imgs, uint8_t* y_out,
                                   uint8_t* cb_out, uint8_t* cr_out, heic_tile_status* status) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!ctx || !y_out) bail(HEIC_E_INVALID_ARG, "null argument");
    return decode_grids_impl(ctx, imgs, output_specs(imgs, n_imgs, nullptr, nullptr, nullptr, 0).data(), n_imgs, nullptr, 0, 0,
                             y_out, cb_out, cr_out, status);
  }));
}

int32_t heic_b200_decode_file(heic_b200_ctx* ctx, const uint8_t* data, size_t len, uint8_t* rgb_out, size_t pitch,
                              int32_t apply_transforms) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!ctx || !data || !rgb_out) bail(HEIC_E_INVALID_ARG, "null argument");
    std::unique_ptr<HeicFile> f = HeicDecoder::open(data, len);
    const heic_image_transform* xf = apply_transforms ? &f->primary.transform : nullptr;
    return decode_grids_impl(ctx, &f->primary.desc, output_specs(&f->primary.desc, 1, xf, nullptr, nullptr, 0).data(), 1, rgb_out,
                             pitch, 0, nullptr, nullptr, nullptr, nullptr);
  }));
}

// Stand-alone emulation-prevention removal + entry-point re-basing of one raw NAL payload on the GPU (the stage
// decode_grids runs for heic_tile_desc::escaped tiles): the device twin of heic_b200_remove_emulation_prevention.
int32_t heic_b200_unescape(heic_b200_ctx* ctx, const uint8_t* nal_payload, size_t len, uint32_t slice_data_byte_offset,
                           const uint32_t* substream_offset, uint32_t n_substreams, uint8_t* rbsp_out, size_t* rbsp_len,
                           uint32_t* slice_data_byte_offset_out, uint32_t* substream_offset_out) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!ctx || !nal_payload || !rbsp_out || !rbsp_len || (n_substreams && (!substream_offset || !substream_offset_out)))
      bail(HEIC_E_INVALID_ARG, "null argument");
    if (len > 0x7fffffffu || slice_data_byte_offset > len) bail(HEIC_E_INVALID_ARG, "payload too large or data offset outside it");
    CU(cudaSetDevice(ctx->device));
    const size_t padded = up(len + 8, 16) + 16;
    DevBuf d_raw, d_out, d_tile, d_sub, d_status;
    d_raw.ensure(padded);
    d_out.ensure(padded);
    d_tile.ensure(sizeof(TileParams));
    d_sub.ensure((size_t)std::max(1u, n_substreams) * 4);
    d_status.ensure(sizeof(TileStatusDev));
    TileParams tp;
    std::memset(&tp, 0, sizeof tp);
    tp.bs_len = (uint32_t)len;
    tp.data_off = slice_data_byte_offset;
    tp.n_sub = n_substreams;
    tp.escaped = 1;
    cudaStream_t st = ctx->stream;
    CU(cudaMemsetAsync(d_raw.p, 0, padded, st));
    CU(cudaMemsetAsync(d_status.p, 0, sizeof(TileStatusDev), st));
    CU(cudaMemcpyAsync(d_raw.p, nal_payload, len, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_tile.p, &tp, sizeof tp, cudaMemcpyHostToDevice, st));
    if (n_substreams) CU(cudaMemcpyAsync(d_sub.p, substream_offset, (size_t)n_substreams * 4, cudaMemcpyHostToDevice, st));
    Arenas A;
    std::memset(&A, 0, sizeof A);
    A.raw = (const uint8_t*)d_raw.p;
    A.bitstream = (const uint8_t*)d_out.p;
    A.status = (TileStatusDev*)d_status.p;
    A.n_tiles = 1;
    CU(launch_unescape(A, (TileParams*)d_tile.p, (uint32_t*)d_sub.p, st));
    ctx->launches++;
    TileStatusDev sd;
    CU(cudaMemcpyAsync(&tp, d_tile.p, sizeof tp, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(&sd, d_status.p, sizeof sd, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (sd.code != 0) bail(HEIC_E_BITSTREAM, "more emulation prevention bytes in one NAL unit than the GPU path handles");
    *rbsp_len = tp.bs_len;
    if (slice_data_byte_offset_out) *slice_data_byte_offset_out = tp.data_off;
    CU(cudaMemcpy(rbsp_out, d_out.p, tp.bs_len, cudaMemcpyDeviceToHost));
    if (n_substreams) CU(cudaMemcpy(substream_offset_out, d_sub.p, (size_t)n_substreams * 4, cudaMemcpyDeviceToHost));
    return 0;
  }));
}

int32_t heic_b200_color_stitch(heic_b200_ctx* ctx, const void* dev_planes, uint32_t n_images, uint32_t grid_rows,
                               uint32_t grid_cols, uint32_t tile_w, uint32_t tile_h, uint32_t out_w, uint32_t out_h,
                               uint32_t full_range, uint32_t matrix_coeffs, void* dev_rgb, size_t pitch,
                               size_t image_stride) {
  return static_cast<int32_t>(guard([&]() -> int64_t {
    if (!ctx || !dev_planes || !dev_rgb) bail(HEIC_E_INVALID_ARG, "null argument");
    if (!n_images || !grid_rows || !grid_cols || (tile_w & 7) || (tile_h & 1) || !tile_w || !tile_h)
      bail(HEIC_E_INVALID_ARG, "tile width must be a multiple of 8 and tile height even");
    if (out_w > grid_cols * tile_w || out_h > grid_rows * tile_h || pitch < (size_t)out_w * 3)
      bail(HEIC_E_INVALID_ARG, "canvas larger than the tile mosaic, or pitch too small");
    CU(cudaSetDevice(ctx->device));
    ColorJob job;
    job.planes = (const uint8_t*)dev_planes;
    job.fused = 0;
    job.planes_sao = nullptr;
    job.sao = nullptr;
    job.sao_stride = 0;
    job.log2_ctb = job.wctb = 0;
    job.tile_stride = (size_t)tile_w * tile_h * 3 / 2;
    job.cb_off = (size_t)tile_w * tile_h;
    job.cr_off = job.cb_off + (size_t)(tile_w / 2) * (tile_h / 2);
    job.pitch_y = tile_w;
    job.pitch_c = tile_w / 2;
    job.tile_w = tile_w;
    job.tile_h = tile_h;
    job.grid_cols = grid_cols;
    job.grid_rows = grid_rows;
    job.out_w = out_w;
    job.out_h = out_h;
    job.n_images = n_images;
    job.chroma = 1;
    job.full_range = full_range;
    job.matrix_coeffs = matrix_coeffs;
    job.orientation = 0;
    job.rgb = (uint8_t*)dev_rgb;
    job.pitch = pitch;
    job.image_stride = image_stride;
    CU(launch_color(job, ColorWindow{0, 0, out_w, out_h, 0, 0}, 1, ctx->stream));
    ctx->launches++;
    CU(cudaStreamSynchronize(ctx->stream));
    return 0;
  }));
}

}  // extern "C"
