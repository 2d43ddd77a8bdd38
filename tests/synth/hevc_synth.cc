// TEST INFRASTRUCTURE ONLY — a small deterministic HEVC Main-Still-Picture intra *bitstream generator*.
//
// BASELINE.json asks for "synthetic HEVC Main-Still-Picture intra bitstreams from a small deterministic in-repo
// CABAC encoder" because the only real input is halfmoonbay.heic.  This is that encoder.  It does not compress an
// image: it drives the repo's own syntax walker (heif_b200/csrc/cuda/cabac_parse.cuh, compiled for the host) with an
// arithmetic *encoder* in place of the decoder engine.  Every bin the walker asks for is drawn from a seeded RNG
// according to the context's own probability estimate, encoded (H.265 9.3.4.x encoding process: EncodeDecision,
// EncodeBypass, EncodeTerminate, EncodeFlush, PutBit with outstanding bits) and returned, so the walker's control
// flow guarantees a syntactically valid slice that exercises whatever the parameter sets enable (CTB 16/32/64,
// transform hierarchy, transform skip, sign data hiding, cu_qp_delta, SAO, WPP on/off, scaling lists, 4:0:0, picture
// sizes that are not CTB multiples, escape-coded levels up to 32767 on request).  VPS/SPS/PPS/slice-header writers (7.3.1-7.3.6) and emulation prevention
// make it a complete Annex-B-able stream, so FFmpeg — not just this repo's oracle — can decode it.
// Never linked into libheic_b200.so.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../heif_b200/csrc/cuda/cabac_tables.h"
#include "../../heif_b200/csrc/cuda/host_params.h"

using namespace heic;
using namespace heic::dev;

namespace {

struct Rng {  // splitmix64
  uint64_t s;
  uint64_t next() {
    uint64_t z = (s += 0x9e3779b97f4a7c15ull);
    z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
    z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
    return z ^ (z >> 31);
  }
  double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
};

struct BitWriter {
  std::vector<uint8_t> bytes;
  int nbits = 0;  // bits used in the last byte
  void put(uint32_t bit) {
    if (nbits == 0) bytes.push_back(0);
    bytes.back() |= (uint8_t)((bit & 1u) << (7 - nbits));
    nbits = (nbits + 1) & 7;
  }
  void u(uint32_t v, int n) {
    for (int i = n - 1; i >= 0; i--) put((v >> i) & 1u);
  }
  void ue(uint32_t v) {
    uint64_t x = (uint64_t)v + 1;
    int len = 0;
    while ((x >> len) > 1) len++;
    for (int i = 0; i < len; i++) put(0);
    for (int i = len; i >= 0; i--) put((uint32_t)(x >> i) & 1u);
  }
  void se(int32_t v) { ue(v > 0 ? (uint32_t)(2 * v - 1) : (uint32_t)(-2 * (int64_t)v)); }
  void trailing() {  // rbsp_trailing_bits / byte_alignment
    put(1);
    while (nbits) put(0);
  }
  bool aligned() const { return nbits == 0; }
};

// 9.3.3.11 binarization of coeff_abs_level_remaining: TR prefix (cMax 4 << cRiceParam) and, past it, an EG(k) escape with
// k = cRiceParam + 1 (unary prefix of ones, a zero, prefix + k suffix bits).  Appends the bins to `out`.
void level_remaining_bins(int rice, uint32_t v, std::vector<uint8_t>& out) {
  if (v < (4u << rice)) {
    for (uint32_t i = 0; i < (v >> rice); i++) out.push_back(1);
    out.push_back(0);
    for (int b = rice - 1; b >= 0; b--) out.push_back((uint8_t)((v >> b) & 1u));
    return;
  }
  for (int i = 0; i < 4; i++) out.push_back(1);
  uint32_t u = v - (4u << rice);
  int k = rice + 1, ones = 0;
  while (u >= (1u << k)) {
    u -= 1u << k;
    k++;
    ones++;
  }
  for (int i = 0; i < ones; i++) out.push_back(1);
  out.push_back(0);
  for (int b = k - 1; b >= 0; b--) out.push_back((uint8_t)((u >> b) & 1u));
}

// A coeff_abs_level_remaining value in [0, max_value]: the maximum, a value next to a change of the escape's prefix length
// (first value of a prefix length, +-1), or log-uniform over the range.
uint32_t large_level_target(Rng& rng, int rice, int max_value) {
  if (max_value <= 0) return 0;
  const uint32_t pick = (uint32_t)(rng.next() % 8);
  if (pick == 0) return (uint32_t)max_value;
  if (pick == 1) {
    uint32_t edges[24];
    int n = 0;
    for (int ones = 0; ones < 24; ones++) {
      const uint64_t first = (4ull << rice) + ((((1ull << ones) - 1ull)) << (rice + 1));
      if (first > (uint64_t)max_value) break;
      edges[n++] = (uint32_t)first;
    }
    if (n) {
      const int64_t v = (int64_t)edges[rng.next() % (uint64_t)n] + (int64_t)(rng.next() % 3) - 1;
      return (uint32_t)(v < 0 ? 0 : (v > max_value ? max_value : v));
    }
  }
  const double x = std::exp(rng.uniform() * std::log((double)max_value + 1.0)) - 1.0;
  const uint32_t v = (uint32_t)x;
  return v > (uint32_t)max_value ? (uint32_t)max_value : v;
}

// Encoder twin of dev::Engine (same member functions the Parser calls).
struct EncEngine {
  const uint8_t* data = nullptr;  // unused
  uint32_t bins = 0;
  Rng* rng = nullptr;
  double lps_gain = 1.0;          // > 1 makes LPS decisions more likely (busier streams)
  int max_bypass_ones = 6;        // caps unary / Exp-Golomb prefixes so values stay conformant
  // Optional overrides of P(bin = 1) for elements whose random-walk statistics are far from an encoder's choices
  // (< 0: off, the context's own probability is used and no extra number is drawn): real streams switch SAO on for a few
  // per cent of the CTBs and smooth pictures rarely split their coding units.  Few coded blocks (cbf_luma / cbf_cb /
  // cbf_cr) give smooth, prediction-dominated pictures, on which strong intra smoothing passes its flatness tests;
  // prev_intra_luma_pred_flag moves the luma modes between the most probable ones and the remaining 32.
  double sao_on_prob = -1.0, split_cu_prob = -1.0, cbf_prob = -1.0, prev_intra_prob = -1.0;
  // With this probability a coeff_abs_level_remaining takes a chosen value (large_level_target) instead of the random walk:
  // its bins are queued and served to the next bypass() calls without the ones cap.
  double big_level_prob = 0.0;
  int ctx_hint = -1;
  std::vector<uint8_t> queued;  // bypass bins still to serve, in order
  size_t queued_pos = 0;
  // arithmetic encoder state (9.3.4.x)
  uint32_t low = 0, range = 510;
  int first_bit = 1, outstanding = 0, ones_run = 0, next_term = 0;
  BitWriter* cur = nullptr;
  std::vector<BitWriter> substreams;

  void write_bit(uint32_t b) { cur->put(b); }
  void put_bit(uint32_t b) {
    if (first_bit) first_bit = 0;
    else write_bit(b);
    while (outstanding > 0) {
      write_bit(1 - b);
      outstanding--;
    }
  }
  void renorm() {
    while (range < 256) {
      if (low < 256) put_bit(0);
      else if (low >= 512) {
        low -= 512;
        put_bit(1);
      } else {
        low -= 256;
        outstanding++;
      }
      range <<= 1;
      low <<= 1;
    }
  }
  void encode_decision(const CabacTabs* T, uint32_t& s, int bin) {
    const uint32_t q = (range >> 6) & 3u;
    const uint32_t lps = (T->st[s].lps >> (q << 3)) & 0xffu;
    range -= lps;
    if (bin != (int)(s & 1u)) {
      low += range;
      range = lps;
      s = (T->st[s].next >> 8) & 0xffu;
    } else {
      s = T->st[s].next & 0xffu;
    }
    renorm();
  }
  void encode_bypass(int bin) {
    low <<= 1;
    if (bin) low += range;
    if (low >= 1024) {
      put_bit(1);
      low -= 1024;
    } else if (low < 512) {
      put_bit(0);
    } else {
      low -= 512;
      outstanding++;
    }
  }
  void flush() {
    range = 2;
    renorm();
    put_bit((low >> 9) & 1u);
    write_bit((low >> 8) & 1u);
    write_bit(1);  // ((low >> 7) & 3) | 1: the forced 1 is the rbsp stop bit / alignment_bit_equal_to_one
    while (!cur->aligned()) write_bit(0);
  }
  // ---- the interface Parser<> uses ------------------------------------------------------------------
  void init(const uint8_t*, uint32_t, uint32_t) {  // a new substream starts
    substreams.emplace_back();
    cur = &substreams.back();
    low = 0;
    range = 510;
    first_bit = 1;
    outstanding = 0;
    ones_run = 0;
  }
  bool offset_is_illegal() const { return false; }
  void expect_terminate(int v) { next_term = v; }
  void hint_ctx(int idx) { ctx_hint = idx; }
  void hint_level_remaining(int rice, int base_level) {
    if (big_level_prob <= 0.0 || rng->uniform() >= big_level_prob) return;  // no draw at all when off: streams stay as before
    level_remaining_bins(rice, large_level_target(*rng, rice, 32767 - base_level), queued);
    queued_pos = 0;
  }
  int decision(const CabacTabs* T, uint32_t& s) {
    double forced = -1.0;
    if (ctx_hint == CTX_SAO_TYPE) forced = sao_on_prob;
    else if (ctx_hint >= CTX_SPLIT_CU && ctx_hint < CTX_SPLIT_CU + 3) forced = split_cu_prob;
    else if (ctx_hint >= CTX_CBF_LUMA && ctx_hint < CTX_CBF_CHROMA + 4) forced = cbf_prob;  // CBF_CHROMA follows CBF_LUMA
    else if (ctx_hint == CTX_PREV_INTRA) forced = prev_intra_prob;
    ctx_hint = -1;
    if (forced >= 0.0) {
      const int bin = rng->uniform() < forced ? 1 : 0;
      encode_decision(T, s, bin);
      bins++;
      ones_run = 0;
      return bin;
    }
    // P(LPS) of pStateIdx p: 0.5 * alpha^p, alpha = (0.01875 / 0.5)^(1/63)
    const int p = (int)(s >> 1);
    double p_lps = 0.5;
    for (int i = 0; i < p; i++) p_lps *= 0.949217148;
    p_lps *= lps_gain;
    if (p_lps > 0.5) p_lps = 0.5;
    const int mps = (int)(s & 1u);
    const int bin = rng->uniform() < p_lps ? 1 - mps : mps;
    encode_decision(T, s, bin);
    bins++;
    ones_run = 0;
    return bin;
  }
  int bypass() {
    if (queued_pos < queued.size()) {
      const int bin = queued[queued_pos++];
      if (queued_pos == queued.size()) {
        queued.clear();
        queued_pos = 0;
      }
      ones_run = 0;
      encode_bypass(bin);
      bins++;
      return bin;
    }
    int bin = (int)(rng->next() >> 63);
    if (bin && ones_run >= max_bypass_ones) bin = 0;
    ones_run = bin ? ones_run + 1 : 0;
    encode_bypass(bin);
    bins++;
    return bin;
  }
  int terminate() {
    bins++;
    ones_run = 0;
    range -= 2;
    if (next_term) {
      low += range;
      flush();
      return 1;
    }
    renorm();
    return 0;
  }
  uint32_t fl_bypass(int n) {
    uint32_t v = 0;
    for (int i = 0; i < n; i++) v = (v << 1) | (uint32_t)bypass();
    return v;
  }
  uint32_t tr_bypass(uint32_t cmax) {
    uint32_t v = 0;
    while (v < cmax && bypass()) v++;
    return v;
  }
};

struct SeqSync {
  static constexpr int kSaveStride = 1;
  std::vector<uint8_t> save;
  SeqSync() : save(NUM_CTX_PAD) {}
  bool wait(int, int) { return true; }
  void publish(int, int) {}
  uint8_t* save_area(int) { return save.data(); }
  void abort(int) {}
};

// ---- parameter-set / header writers ------------------------------------------------------------------------
void profile_tier_level(BitWriter& w, int profile_idc) {
  w.u(0, 2);  // general_profile_space
  w.u(0, 1);  // general_tier_flag
  w.u((uint32_t)profile_idc, 5);
  for (int j = 0; j < 32; j++) w.u((j == profile_idc || (profile_idc == 3 && (j == 1 || j == 2))) ? 1 : 0, 1);
  w.u(1, 1);  // progressive_source
  w.u(0, 1);  // interlaced_source
  w.u(1, 1);  // non_packed_constraint
  w.u(1, 1);  // frame_only_constraint
  w.u(0, 32);
  w.u(0, 11);  // 43 reserved bits
  w.u(0, 1);   // general_inbld_flag / reserved
  w.u(120, 8); // general_level_idc (4.0)
}

void scaling_list_data(BitWriter& w, const heic_scaling_list& sl) {
  for (int size_id = 0; size_id < 4; size_id++)
    for (int m = 0; m < 6; m += (size_id == 3 ? 3 : 1)) {
      w.u(1, 1);  // scaling_list_pred_mode_flag: explicit
      const int n = size_id == 0 ? 16 : 64;
      int next = 8;
      if (size_id > 1) {
        const int dc = sl.dc[size_id - 2][m];
        w.se(dc - 8);
        next = dc;
      }
      for (int i = 0; i < n; i++) {
        int delta = (int)sl.list[size_id][m][i] - next;
        if (delta > 127) delta -= 256;
        if (delta < -128) delta += 256;
        w.se(delta);
        next = sl.list[size_id][m][i];
      }
    }
}

std::vector<uint8_t> escape(const std::vector<uint8_t>& rbsp) {  // 7.4.2: emulation prevention
  std::vector<uint8_t> out;
  int zeros = 0;
  for (uint8_t b : rbsp) {
    if (zeros >= 2 && b <= 3) {
      out.push_back(3);
      zeros = 0;
    }
    out.push_back(b);
    zeros = b == 0 ? zeros + 1 : 0;
  }
  return out;
}
size_t escaped_size(const std::vector<uint8_t>& v) { return escape(v).size(); }

std::vector<uint8_t> nal(int type, const std::vector<uint8_t>& rbsp) {
  std::vector<uint8_t> out = {(uint8_t)(type << 1), 1};  // forbidden_zero, type, layer 0, temporal_id_plus1 = 1
  std::vector<uint8_t> e = escape(rbsp);
  out.insert(out.end(), e.begin(), e.end());
  return out;
}

}  // namespace

extern "C" {

struct synth_config {
  uint32_t width, height;              // multiples of the minimum coding block size
  uint32_t chroma_format_idc;          // 0 or 1
  uint32_t log2_min_cb, log2_ctb;      // 3..6
  uint32_t log2_min_tb, log2_max_tb;   // 2..5
  uint32_t max_transform_hierarchy_depth_intra;
  uint32_t scaling_list_mode;          // 0 off, 1 default lists, 2 explicit lists in the SPS, 3 explicit lists in the PPS
  uint32_t sao, strong_intra_smoothing;
  uint32_t sign_data_hiding, transform_skip, cu_qp_delta, diff_cu_qp_delta_depth;
  int32_t init_qp_minus26, slice_qp_delta, cb_qp_offset, cr_qp_offset, slice_cb_qp_offset, slice_cr_qp_offset;
  uint32_t wpp;
  uint32_t deblocking_disabled;
  int32_t beta_offset_div2, tc_offset_div2;
  uint32_t slice_sao_luma, slice_sao_chroma;
  uint32_t full_range, matrix_coeffs;
  double lps_gain;                     // 1.0 = draw bins from the contexts' own probabilities
  uint32_t max_bypass_ones;
  double sao_on_prob, split_cu_prob;   // < 0: unbiased (see EncEngine)
  double big_level_prob;               // 0: every coeff_abs_level_remaining from the random walk (see EncEngine)
  uint32_t scaling_list_min, scaling_list_max;  // range of the explicit scaling-list entries (0, 0: 8..63)
  double cbf_prob, prev_intra_prob;    // < 0: unbiased (see EncEngine)
};

// Writes the four NAL units (2-byte header + escaped payload) of one IDR_N_LP picture.  Each out_* buffer has `cap`
// bytes; lens[4] receives the sizes (VPS, SPS, PPS, slice).  Returns 0, or a negative value when the buffers are too
// small (-1), the configuration is rejected (-2), or the random walk produced a non-conformant value (-3: retry with
// another seed).
int synth_encode_picture(const synth_config* cfg, uint64_t seed, uint8_t* out_vps, uint8_t* out_sps, uint8_t* out_pps,
                         uint8_t* out_slice, size_t cap, size_t* lens) {
  try {
    Rng rng{seed * 0x2545f4914f6cdd1dull + 0x1234567ull};
    heic_sps sps;
    heic_pps pps;
    std::memset(&sps, 0, sizeof sps);
    std::memset(&pps, 0, sizeof pps);
    sps.chroma_format_idc = cfg->chroma_format_idc;
    sps.pic_width_in_luma_samples = cfg->width;
    sps.pic_height_in_luma_samples = cfg->height;
    sps.log2_min_luma_coding_block_size_minus3 = cfg->log2_min_cb - 3;
    sps.log2_diff_max_min_luma_coding_block_size = cfg->log2_ctb - cfg->log2_min_cb;
    sps.log2_min_luma_transform_block_size_minus2 = cfg->log2_min_tb - 2;
    sps.log2_diff_max_min_luma_transform_block_size = cfg->log2_max_tb - cfg->log2_min_tb;
    sps.max_transform_hierarchy_depth_intra = cfg->max_transform_hierarchy_depth_intra;
    sps.max_transform_hierarchy_depth_inter = cfg->max_transform_hierarchy_depth_intra;
    sps.scaling_list_enabled_flag = cfg->scaling_list_mode != 0;
    sps.sps_scaling_list_data_present_flag = cfg->scaling_list_mode == 2;
    sps.sample_adaptive_offset_enabled_flag = cfg->sao;
    sps.strong_intra_smoothing_enabled_flag = cfg->strong_intra_smoothing;
    sps.vui_parameters_present_flag = 1;
    sps.video_full_range_flag = cfg->full_range;
    sps.colour_primaries = 2;
    sps.transfer_characteristics = 2;
    sps.matrix_coeffs = cfg->matrix_coeffs;
    pps.sign_data_hiding_enabled_flag = cfg->sign_data_hiding;
    pps.init_qp_minus26 = cfg->init_qp_minus26;
    pps.transform_skip_enabled_flag = cfg->transform_skip;
    pps.cu_qp_delta_enabled_flag = cfg->cu_qp_delta;
    pps.diff_cu_qp_delta_depth = cfg->cu_qp_delta ? cfg->diff_cu_qp_delta_depth : 0;
    pps.pps_cb_qp_offset = cfg->cb_qp_offset;
    pps.pps_cr_qp_offset = cfg->cr_qp_offset;
    pps.pps_slice_chroma_qp_offsets_present_flag = (cfg->slice_cb_qp_offset || cfg->slice_cr_qp_offset) ? 1 : 0;
    pps.entropy_coding_sync_enabled_flag = cfg->wpp;
    pps.deblocking_filter_control_present_flag = 1;
    pps.pps_deblocking_filter_disabled_flag = cfg->deblocking_disabled;
    pps.pps_beta_offset_div2 = cfg->beta_offset_div2;
    pps.pps_tc_offset_div2 = cfg->tc_offset_div2;
    pps.pps_scaling_list_data_present_flag = cfg->scaling_list_mode == 3;
    heic_scaling_list lists;
    default_scaling_list(lists);
    if (cfg->scaling_list_mode >= 2) {  // seeded explicit lists in [scaling_list_min, scaling_list_max]
      const uint32_t lo = cfg->scaling_list_min ? cfg->scaling_list_min : 8, hi = cfg->scaling_list_max ? cfg->scaling_list_max : 63;
      if (lo < 1 || hi > 255 || lo > hi) return -2;
      for (int s = 0; s < 4; s++)
        for (int m = 0; m < 6; m++) {
          for (int i = 0; i < 64; i++) lists.list[s][m][i] = (uint8_t)(lo + rng.next() % (hi - lo + 1));
          if (s >= 2) lists.dc[s - 2][m] = (uint8_t)(lo + rng.next() % (hi - lo + 1));
        }
      // sizeId 3 only codes matrixId 0 and 3; a decoder copies nothing else, so keep the chroma slots consistent with
      // what 7.3.4 infers for ChromaArrayType != 3 (not used for 4:2:0 intra 32x32, but keep the struct well defined)
      if (cfg->scaling_list_mode == 2) sps.scaling_list = lists;
      else pps.scaling_list = lists;
    }

    PicParams pp;
    make_pic_params(sps, pps, pp);

    // ---- slice data through the repo's syntax walker ----------------------------------------------------
    heic_tile_desc td;
    std::memset(&td, 0, sizeof td);
    static const uint8_t dummy[4] = {0, 0, 0, 0};
    td.rbsp = dummy;
    td.rbsp_len = 0;
    td.header.slice_type = 2;
    td.header.slice_qp_delta = cfg->slice_qp_delta;
    td.header.slice_cb_qp_offset = cfg->slice_cb_qp_offset;
    td.header.slice_cr_qp_offset = cfg->slice_cr_qp_offset;
    td.header.slice_sao_luma_flag = cfg->sao && cfg->slice_sao_luma;
    td.header.slice_sao_chroma_flag = cfg->sao && cfg->slice_sao_chroma && cfg->chroma_format_idc;
    td.header.slice_deblocking_filter_disabled_flag = cfg->deblocking_disabled;
    td.header.slice_beta_offset_div2 = cfg->beta_offset_div2;
    td.header.slice_tc_offset_div2 = cfg->tc_offset_div2;
    td.header.num_entry_point_offsets = cfg->wpp ? (uint32_t)pp.hctb - 1 : 0;
    if (td.header.num_entry_point_offsets > HEIC_MAX_ENTRY_POINTS) return -2;
    TileParams tp;
    std::memset(&tp, 0, sizeof tp);
    make_tile_params(pp, pps, td, tp);

    static const CabacTabs tabs = [] {  // built once (thread-safe: pool.py encodes from several threads)
      CabacTabs t;
      build_cabac_tabs(t);
      return t;
    }();
    std::vector<uint32_t> tu((size_t)pp.n_tu, 0), sao((size_t)pp.wctb * pp.hctb * 4, 0);
    std::vector<int16_t> l0((size_t)pp.n_tu * 16, 0), l1((size_t)pp.n_tu * 4, 0), l2((size_t)pp.n_tu * 4, 0);
    std::vector<uint8_t> ipm((size_t)pp.w4 * pp.h4, 0), ctd((size_t)pp.w8 * pp.h8, 0), qp((size_t)pp.w8 * pp.h8, 0), ctx(NUM_CTX_PAD);
    std::vector<uint32_t> sub_off((size_t)pp.hctb + 1, 0);
    Parser<1, EncEngine> P;
    P.e.rng = &rng;
    P.e.lps_gain = cfg->lps_gain > 0 ? cfg->lps_gain : 1.0;
    P.e.max_bypass_ones = cfg->max_bypass_ones ? (int)cfg->max_bypass_ones : 6;
    P.e.sao_on_prob = cfg->sao_on_prob;
    P.e.split_cu_prob = cfg->split_cu_prob;
    P.e.big_level_prob = cfg->big_level_prob;
    P.e.cbf_prob = cfg->cbf_prob;
    P.e.prev_intra_prob = cfg->prev_intra_prob;
    P.T = &tabs;
    P.ctx = ctx.data();
    P.pp = &pp;
    P.tp = &tp;
    P.tu_map = tu.data();
    P.coeff0 = l0.data();
    P.coeff1 = l1.data();
    P.coeff2 = l2.data();
    P.ipm = ipm.data();
    P.ct_depth = ctd.data();
    P.qp_map = qp.data();
    P.sao = sao.data();
    P.err = 0;
    SeqSync sync;
    parse_rows<1>(P, sub_off.data(), 0, 1, sync);
    if (P.err) return -3;

    // ---- slice segment header (7.3.6.1) + data -----------------------------------------------------------
    std::vector<BitWriter>& subs = P.e.substreams;
    BitWriter sh;
    sh.u(1, 1);                // first_slice_segment_in_pic_flag
    sh.u(0, 1);                // no_output_of_prior_pics_flag (IRAP)
    sh.ue(0);                  // slice_pic_parameter_set_id
    sh.ue(2);                  // slice_type I
    if (cfg->sao) {
      sh.u(td.header.slice_sao_luma_flag, 1);
      if (cfg->chroma_format_idc) sh.u(td.header.slice_sao_chroma_flag, 1);
    }
    sh.se(cfg->slice_qp_delta);
    if (pps.pps_slice_chroma_qp_offsets_present_flag) {
      sh.se(cfg->slice_cb_qp_offset);
      sh.se(cfg->slice_cr_qp_offset);
    }
    // deblocking_filter_override_enabled_flag = 0: no override syntax; pps_loop_filter_across_slices = 0
    if (cfg->wpp) {
      const uint32_t n = (uint32_t)subs.size() - 1;
      sh.ue(n);
      if (n) {
        uint32_t max_off = 1;
        std::vector<uint32_t> sizes;
        for (uint32_t k = 0; k < n; k++) {
          sizes.push_back((uint32_t)escaped_size(subs[k].bytes));
          if (sizes.back() > max_off) max_off = sizes.back();
        }
        int len = 1;
        while ((1ull << len) < (uint64_t)max_off) len++;  // entry_point_offset_minus1 < 2^len
        sh.ue((uint32_t)len - 1);
        for (uint32_t k = 0; k < n; k++) sh.u(sizes[k] - 1, len);
      }
    }
    sh.trailing();  // byte_alignment()
    std::vector<uint8_t> slice_rbsp = sh.bytes;
    for (const BitWriter& s : subs) slice_rbsp.insert(slice_rbsp.end(), s.bytes.begin(), s.bytes.end());

    // ---- VPS / SPS / PPS (7.3.2) ------------------------------------------------------------------------------
    const int profile = cfg->chroma_format_idc ? 3 : 4;  // Main Still Picture, or RExt for monochrome
    BitWriter v;
    v.u(0, 4);
    v.u(1, 1);
    v.u(1, 1);
    v.u(0, 6);
    v.u(0, 3);
    v.u(1, 1);
    v.u(0xffff, 16);
    profile_tier_level(v, profile);
    v.u(1, 1);  // vps_sub_layer_ordering_info_present_flag
    v.ue(0);
    v.ue(0);
    v.ue(0);
    v.u(0, 6);  // vps_max_layer_id
    v.ue(0);    // vps_num_layer_sets_minus1
    v.u(0, 1);  // vps_timing_info_present_flag
    v.u(0, 1);  // vps_extension_flag
    v.trailing();

    BitWriter s;
    s.u(0, 4);
    s.u(0, 3);
    s.u(1, 1);
    profile_tier_level(s, profile);
    s.ue(0);
    s.ue(cfg->chroma_format_idc);
    s.ue(cfg->width);
    s.ue(cfg->height);
    s.u(0, 1);  // conformance_window_flag
    s.ue(0);
    s.ue(0);    // bit depths
    s.ue(4);    // log2_max_pic_order_cnt_lsb_minus4
    s.u(1, 1);  // sps_sub_layer_ordering_info_present_flag
    s.ue(0);
    s.ue(0);
    s.ue(0);
    s.ue(sps.log2_min_luma_coding_block_size_minus3);
    s.ue(sps.log2_diff_max_min_luma_coding_block_size);
    s.ue(sps.log2_min_luma_transform_block_size_minus2);
    s.ue(sps.log2_diff_max_min_luma_transform_block_size);
    s.ue(sps.max_transform_hierarchy_depth_inter);
    s.ue(sps.max_transform_hierarchy_depth_intra);
    s.u(sps.scaling_list_enabled_flag, 1);
    if (sps.scaling_list_enabled_flag) {
      s.u(sps.sps_scaling_list_data_present_flag, 1);
      if (sps.sps_scaling_list_data_present_flag) scaling_list_data(s, lists);
    }
    s.u(0, 1);  // amp
    s.u(cfg->sao, 1);
    s.u(0, 1);  // pcm
    s.ue(0);    // num_short_term_ref_pic_sets
    s.u(0, 1);  // long_term_ref_pics_present
    s.u(0, 1);  // sps_temporal_mvp_enabled
    s.u(cfg->strong_intra_smoothing, 1);
    s.u(1, 1);  // vui_parameters_present_flag
    s.u(0, 1);  // aspect_ratio_info_present
    s.u(0, 1);  // overscan_info_present
    s.u(1, 1);  // video_signal_type_present
    s.u(5, 3);
    s.u(cfg->full_range, 1);
    s.u(1, 1);  // colour_description_present
    s.u(2, 8);
    s.u(2, 8);
    s.u(cfg->matrix_coeffs, 8);
    s.u(0, 1);  // chroma_loc_info_present
    s.u(0, 1);  // neutral_chroma_indication
    s.u(0, 1);  // field_seq
    s.u(0, 1);  // frame_field_info_present
    s.u(0, 1);  // default_display_window
    s.u(0, 1);  // vui_timing_info_present
    s.u(0, 1);  // bitstream_restriction
    s.u(0, 1);  // sps_extension_present
    s.trailing();

    BitWriter p;
    p.ue(0);
    p.ue(0);
    p.u(0, 1);  // dependent_slice_segments_enabled
    p.u(0, 1);  // output_flag_present
    p.u(0, 3);  // num_extra_slice_header_bits
    p.u(cfg->sign_data_hiding, 1);
    p.u(0, 1);  // cabac_init_present
    p.ue(0);
    p.ue(0);
    p.se(cfg->init_qp_minus26);
    p.u(0, 1);  // constrained_intra_pred
    p.u(cfg->transform_skip, 1);
    p.u(cfg->cu_qp_delta, 1);
    if (cfg->cu_qp_delta) p.ue(cfg->diff_cu_qp_delta_depth);
    p.se(cfg->cb_qp_offset);
    p.se(cfg->cr_qp_offset);
    p.u(pps.pps_slice_chroma_qp_offsets_present_flag, 1);
    p.u(0, 1);  // weighted_pred
    p.u(0, 1);  // weighted_bipred
    p.u(0, 1);  // transquant_bypass_enabled
    p.u(0, 1);  // tiles_enabled
    p.u(cfg->wpp, 1);
    p.u(0, 1);  // pps_loop_filter_across_slices_enabled
    p.u(1, 1);  // deblocking_filter_control_present
    p.u(0, 1);  // deblocking_filter_override_enabled
    p.u(cfg->deblocking_disabled, 1);
    if (!cfg->deblocking_disabled) {
      p.se(cfg->beta_offset_div2);
      p.se(cfg->tc_offset_div2);
    }
    p.u(pps.pps_scaling_list_data_present_flag, 1);
    if (pps.pps_scaling_list_data_present_flag) scaling_list_data(p, lists);
    p.u(0, 1);  // lists_modification_present
    p.ue(0);    // log2_parallel_merge_level_minus2
    p.u(0, 1);  // slice_segment_header_extension_present
    p.u(0, 1);  // pps_extension_present
    p.trailing();

    const std::vector<uint8_t> n_vps = nal(32, v.bytes), n_sps = nal(33, s.bytes), n_pps = nal(34, p.bytes),
                               n_slice = nal(20, slice_rbsp);
    const std::vector<uint8_t>* all[4] = {&n_vps, &n_sps, &n_pps, &n_slice};
    uint8_t* outs[4] = {out_vps, out_sps, out_pps, out_slice};
    for (int i = 0; i < 4; i++) {
      if (all[i]->size() > cap) return -1;
      std::memcpy(outs[i], all[i]->data(), all[i]->size());
      lens[i] = all[i]->size();
    }
    return 0;
  } catch (const Error&) {
    return -2;
  }
}

// Round trip of one coeff_abs_level_remaining through the arithmetic coder: `value` is encoded as bypass bins (the bins the
// generator queues) behind a seeded run of context-coded bins, which sets ivlCurrRange and the bit position, and the stream
// is placed at an even or odd byte offset (the engine's 16-bit refill phase).  The bins are then decoded twice: with
// dev::Engine::coeff_abs_level_remaining (the device routine: 7-bin division steps) and with the parser's bin-by-bin loop.
// out[0..4]: value and bins of the device routine, value and bins of the loop, bins the encoder wrote.  Returns 0; the
// `bad` flags of the two decodes (1: device routine, 2: loop) when one of them rejected the bins; -1 when the leading
// context-coded bins did not decode back.
int synth_level_remaining_roundtrip(int rice, uint32_t value, uint64_t seed, uint32_t* out) {
  static const CabacTabs tabs = [] {
    CabacTabs t;
    build_cabac_tabs(t);
    return t;
  }();
  Rng rng{seed * 0x9e3779b97f4a7c15ull + 0x51ed27ull};
  const int n_lead = (int)(rng.next() % 48), n_tail = 40;
  const int odd = (int)(rng.next() & 1u);
  std::vector<uint32_t> states;  // context state of each leading bin, drawn afresh per bin (both sides start from it)
  std::vector<uint8_t> lead;
  for (int i = 0; i < n_lead; i++) {
    states.push_back((uint32_t)(rng.next() % 126));
    lead.push_back((uint8_t)(rng.next() >> 63));
  }
  std::vector<uint8_t> bins;
  level_remaining_bins(rice, value, bins);
  EncEngine E;
  E.rng = &rng;
  E.init(nullptr, 0, 0);
  for (int i = 0; i < n_lead; i++) {
    uint32_t s = states[i];
    E.encode_decision(&tabs, s, lead[i]);
  }
  for (uint8_t b : bins) E.encode_bypass(b);
  for (int i = 0; i < n_tail; i++) E.encode_bypass((int)(rng.next() >> 63));
  E.range -= 2;  // end_of_slice_segment_flag = 1
  E.low += E.range;
  E.flush();
  std::vector<uint8_t> buf((size_t)odd, 0xa5);
  buf.insert(buf.end(), E.cur->bytes.begin(), E.cur->bytes.end());
  buf.resize(buf.size() + 8, 0);

  int flags = 0;
  uint32_t vals[2], used[2];
  for (int pass = 0; pass < 2; pass++) {
    Parser<1> P;
    P.err = 0;
    P.e.init(buf.data(), (uint32_t)odd, (uint32_t)buf.size());
    P.e.bins = 0;
    for (int i = 0; i < n_lead; i++) {
      uint32_t s = states[i];
      if (P.e.decision(&tabs, s) != lead[i]) return -1;  // the leading bins must come back unchanged
    }
    const uint32_t b0 = P.e.bins;
    int bad = 0;
    if (pass == 0) vals[0] = P.e.coeff_abs_level_remaining(rice, bad);
    else vals[1] = P.coeff_abs_level_remaining(rice, 0), bad = P.err != 0;
    used[pass] = P.e.bins - b0;
    if (bad) flags |= 1 << pass;
  }
  out[0] = vals[0];
  out[1] = used[0];
  out[2] = vals[1];
  out[3] = used[1];
  out[4] = (uint32_t)bins.size();
  return flags;
}

}  // extern "C"
