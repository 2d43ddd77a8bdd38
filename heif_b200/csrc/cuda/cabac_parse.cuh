// CABAC engine + slice_segment_data() syntax parser, written as per-thread code: one thread owns one
// substream (a WPP row of one HEIF grid tile) and carries the arithmetic decoder in registers, with
// its context table in shared memory.  The kernels in cabac_kernel.cu decide how threads map onto
// substreams; the same source also compiles for the host so the syntax logic can be unit-tested
// without a GPU (tests/emul/ — test infrastructure, never linked into the product library).
//
// Reference interfaces this replaces:
//   ArithmeticDecoderEngine::{try_new, decode_decision, decode_bypass, decode_terminate, try_renorm}
//                                                        src/cabac/arithmetic.rs:23-169
//   init_all_contexts / init_single_context              src/cabac/arithmetic.rs:40-78
//   SyntaxElement::init_values_i_slice                   src/cabac/syntax_element.rs:90-242
//   CabacDecoder binarisations                           src/cabac/decoder.rs:23-284
//   SliceSegmentReader::read_data / read_coding_tree_unit / sao / coding_quadtree
//                                                        src/hevc/slice.rs:206-255 (the last two are todo!())
// Syntax the reference does not implement follows ITU-T H.265 7.3.8 / 9.3 (clauses cited inline).
#pragma once
#include "dev_types.h"

namespace heic {
namespace dev {

// Tables the parser indexes dynamically; copied to shared memory at kernel start.
struct CabacTabs {
  // per context state s = pStateIdx<<1|valMps: .x = rangeTabLps[p][0..3] as 4 bytes (Table 9-46),
  // .y = next state after an MPS | next state after an LPS << 8 (Table 9-45, valMps flip folded in)
  struct alignas(8) State {
    uint32_t lps;   // rangeTabLps[p][0..3], one byte each
    uint32_t next;  // next state after an MPS | next state after an LPS << 8
  } st[128];        // one 8-byte entry per state: a single 64-bit shared-memory load per bin
  uint8_t diag4[16];      // 6.5.3 up-right diagonal, 4x4: scan pos -> x | y << 2
  uint8_t diag8[64];      // 8x8: x | y << 3
  uint8_t diag2[4];       // 2x2: x | y << 1
  uint8_t inv_diag4[16];  // y << 2 | x -> scan pos
  uint8_t inv_diag8[64];
  uint8_t inv_diag2[4];
  uint8_t sig_map4[16];   // ctxIdxMap of 9.3.4.2.5 for 4x4 blocks
  uint8_t sig_pat[4][16]; // sigCtx by prevCsbf pattern and yP << 2 | xP (9.3.4.2.5)
  // sigCtx of the 16 scan positions of a sub-block as nibbles (nibble k = scan position k), before the size / colour
  // offsets: [scanIdx] for 4x4 blocks (ctxIdxMap), [3 + scanIdx * 4 + prevCsbf] for larger ones
  uint64_t sig_nib[15];
  uint8_t init_value[NUM_CTX_PAD];
};
// Layout of the CABAC kernels' dynamic shared memory as far as the parser addresses it: the tables at offset 0, then a copy
// of the batch's arena pointers (cabac_kernel.cu puts them there; Parser::arenas()).
constexpr uint32_t kSmemArenasOff = (uint32_t)((sizeof(CabacTabs) + 15) & ~(size_t)15);

#if defined(__CUDA_ARCH__)
#define HEIC_NO_UNROLL _Pragma("unroll 1")
#else
#define HEIC_NO_UNROLL
#endif
#if defined(__CUDA_ARCH__)
#define HEIC_CLZ(x) __clz(x)
#define HEIC_POPC(x) __popc(x)
#else
#define HEIC_CLZ(x) ((x) ? __builtin_clz(x) : 32)
#define HEIC_POPC(x) __builtin_popcount(x)
#endif

HEIC_HD int clip3i(int lo, int hi, int v) { return v < lo ? lo : (v > hi ? hi : v); }
HEIC_HD uint32_t compact1by1(uint32_t v) {  // even bits of an 8-bit z-order index -> 4-bit coordinate
  v &= 0x55u;
  v = (v | (v >> 1)) & 0x33u;
  v = (v | (v >> 2)) & 0x0fu;
  return v;
}

#if defined(__CUDA_ARCH__)
// All dynamically indexed parser state (tables, context tables) lives in the kernel's dynamic shared memory.  The parser
// reaches it through 32-bit shared-window addresses it carries in registers (Parser::sm, ctx_off, cold_off), turned into
// pointers with smem_ptr(): the compiler still sees the shared address space and emits LDS/STS, but no longer forms the
// address of the shared-memory symbol -- on sm_90+ that is S2UR SR_CgaCtaId + ULEA at the head of every out-of-line
// routine, in front of its first load (3 % of the kernel's stall samples, 80 places).
extern __shared__ __align__(16) unsigned char heic_cabac_smem[];
template <class T>
__device__ __forceinline__ T* smem_ptr(uint32_t addr) {
  return reinterpret_cast<T*>(__cvta_shared_to_generic(addr));
}
#endif

// ------------------------------------------------------------------------------------------------
// Arithmetic decoding engine (9.3.4.3).  `val` holds ivlOffset << 22 with up to 22 look-ahead bits of
// the stream below it, so a renormalisation is two shifts.  The stream is consumed 16 bits at a time from
// 2-byte aligned positions (the initial read takes 2 or 3 bytes to get there); the next two halfwords are
// always already loaded (`look0`, `look1`), so no load sits on the per-bin dependency chain and the refill
// path stays a handful of instructions (it is inlined at every bin).  Bits past the end of the substream
// read as zero (as in the CPU oracle).
// ------------------------------------------------------------------------------------------------
struct Engine {
  const uint8_t* data;   // 2-byte aligned on the device
  uint32_t pos, end;     // next halfword to fetch (even byte offset from data), substream end
  uint32_t look0, look1; // prefetched halfwords (look0: big-endian value; look1: see load16_raw)
  uint32_t range, val;
  int nbits;
  uint32_t bins;

  HEIC_HD uint32_t byte_at(uint32_t p) const { return p < end ? data[p] : 0u; }
  HEIC_HD uint32_t load16(uint32_t p) const {  // p even
    if (p >= end) return 0u;
#if defined(__CUDA_ARCH__)
    uint32_t h = *reinterpret_cast<const uint16_t*>(data + p);
    h = __byte_perm(h, 0u, 0x4401);
#else
    uint32_t h = ((uint32_t)data[p] << 8) | (p + 1 < end ? data[p + 1] : 0u);
#endif
    if (p + 1u >= end) h &= 0xff00u;
    return h;
  }
  // The device keeps the second prefetched halfword as it came from memory and turns it into the big-endian value only
  // when it moves up to `look0`, one refill later: the byte swap right behind the load made every refill wait for the
  // load's latency (4 % of the kernel's stall samples).
  HEIC_HD uint32_t load16_raw(uint32_t p) const {  // p even
#if defined(__CUDA_ARCH__)
    return p < end ? (uint32_t)__ldg(reinterpret_cast<const uint16_t*>(data + p)) : 0u;
#else
    return load16(p);
#endif
  }
  HEIC_HD uint32_t finish16(uint32_t h, uint32_t p) const {
#if defined(__CUDA_ARCH__)
    h = __byte_perm(h, 0u, 0x4401);
    if (p + 1u >= end) h &= 0xff00u;
#else
    (void)p;
#endif
    return h;
  }
  // 9.3.2.5 (arithmetic.rs:23-38): ivlCurrRange = 510, ivlOffset = read_bits(9)
  HEIC_HD void init(const uint8_t* d, uint32_t start, uint32_t stop) {
    data = d;
    end = stop;
    range = 510;
    if (start & 1u) {
      val = ((byte_at(start) << 16) | (byte_at(start + 1) << 8) | byte_at(start + 2)) << 7;
      nbits = 15;
      pos = start + 3;
    } else {
      val = ((byte_at(start) << 8) | byte_at(start + 1)) << 15;
      nbits = 7;
      pos = start + 2;
    }
    look0 = load16(pos);
    look1 = load16_raw(pos + 2);
    pos += 4;
  }
  HEIC_HD bool offset_is_illegal() const { return (val >> 22) >= 510u; }
  HEIC_HD void expect_terminate(int) {}  // hook for the test-only encoder engine (tests/synth); nothing to do when decoding
  HEIC_HD void hint_ctx(int) {}          // likewise: tells that engine which context the next decision uses
  HEIC_HD void hint_level_remaining(int, int) {}  // likewise: a coeff_abs_level_remaining (cRiceParam, baseLevel) follows
  HEIC_HD void refill() {
    if (nbits < 7) {
      val |= look0 << (6 - nbits);
      nbits += 16;
      look0 = finish16(look1, pos - 2u);
      look1 = load16_raw(pos);
      pos += 2;
    }
  }
  // 9.3.4.3.2 (arithmetic.rs:97-135) on a context state s = pStateIdx << 1 | valMps; returns the bin and
  // the updated state through s.
  HEIC_HD int decision(const CabacTabs* T, uint32_t& s) {
    const CabacTabs::State st = T->st[s];
    const uint32_t lps4 = st.lps;
    uint32_t nx = st.next;
    const uint32_t q = (range >> 6) & 3u;
    const uint32_t lps = (lps4 >> (q << 3)) & 0xffu;
    range -= lps;
    const uint32_t scaled = range << 22;
    int bin = (int)(s & 1u);
    if (val >= scaled) {
      val -= scaled;
      range = lps;
      bin ^= 1;
      nx >>= 8;
    }
    s = nx & 0xffu;
    const int sh = HEIC_CLZ(range) - 23;  // arithmetic.rs:137-144, all renorm shifts at once
    range <<= sh;
    val <<= sh;
    nbits -= sh;
    bins++;
    refill();
    return bin;
  }
  // 9.3.4.3.4 (arithmetic.rs:146-157)
  HEIC_HD int bypass() {
    val <<= 1;
    nbits--;
    uint32_t scaled = range << 22;
    int bin = 0;
    if (val >= scaled) {
      val -= scaled;
      bin = 1;
    }
    bins++;
    refill();
    return bin;
  }
  // 9.3.4.3.5 (arithmetic.rs:159-169)
  HEIC_HD int terminate() {
    bins++;
    range -= 2;
    if (val >= (range << 22)) return 1;
    int sh = HEIC_CLZ(range) - 23;
    range <<= sh;
    val <<= sh;
    nbits -= sh;
    refill();
    return 0;
  }
  // ---- several bypass bins per step -------------------------------------------------------------------------
  // k bypass bins in a row are the long division of (ivlOffset * 2^k + next k bits) by ivlCurrRange: the quotient holds
  // the bins (first bin = most significant bit), the remainder is the new ivlOffset.  And the first j bins of the k-bin
  // quotient are the j-bin quotient (floor(floor(X / r) / 2^m) == floor(floor(X / 2^m) / r)), so a unary prefix can be
  // decoded speculatively and only the bins it really has are consumed.  k <= 7 <= nbits always holds after a refill;
  // X < 510 * 2^7 fits a float exactly, the estimate of the quotient is off by at most one and is corrected.
  HEIC_HD uint32_t bypass_quot(uint32_t X) const {
#if defined(__CUDA_ARCH__)
    uint32_t q = (uint32_t)__fdividef((float)X, (float)range);
    const int r = (int)X - (int)(q * range);
    if (r < 0) q--;
    else if (r >= (int)range) q++;
    return q;
#else
    return X / range;
#endif
  }
  // consume the first j of the k bins whose numerator / quotient are X / Q; returns those j bins
  HEIC_HD uint32_t bypass_take(uint32_t X, uint32_t Q, int k, int j) {
    const uint32_t Xj = X >> (k - j), Qj = Q >> (k - j);
    val = ((Xj - Qj * range) << 22) | ((val << j) & 0x3fffffu);
    nbits -= j;
    bins += (uint32_t)j;
    refill();
    return Qj;
  }
  HEIC_HD uint32_t bypass_bins(int k) {  // 1 <= k <= 7
    const uint32_t X = val >> (22 - k);
    return bypass_take(X, bypass_quot(X), k, k);
  }
  HEIC_HD uint32_t fl_bypass(int n) {  // decoder.rs:152-164
    uint32_t v = 0;
    HEIC_NO_UNROLL
    while (n > 0) {
      const int k = n < 7 ? n : 7;
      v = (v << k) | bypass_bins(k);
      n -= k;
    }
    return v;
  }
  HEIC_HD uint32_t tr_bypass(uint32_t cmax) {  // decoder.rs:166-190, cRiceParam 0
    uint32_t v = 0;
    HEIC_NO_UNROLL
    while (v < cmax && bypass()) v++;
    return v;
  }
  HEIC_HD uint32_t egk_bypass(int k, int& bad) {  // decoder.rs:206-222 with 32-bit arithmetic (SURVEY Appendix B #11)
    int ones = 0;
    HEIC_NO_UNROLL
    while (bypass()) {
      if (++ones > 31) {
        bad = 1;
        return 0;
      }
    }
    uint32_t suffix = fl_bypass(ones + k);
    return (((1u << ones) - 1u) << k) + suffix;
  }
  HEIC_HD uint32_t coeff_abs_level_remaining(int rice, int& bad) {  // decoder.rs:224-261
    // prefix (up to four ones and the closing zero) and, when it fits, the rice suffix bits from one division
    const int k = 4 + (rice < 3 ? rice : 3);
    const uint32_t X = val >> (22 - k), Q = bypass_quot(X);
    const uint32_t top4 = Q >> (k - 4);
    const int prefix = HEIC_CLZ(~(top4 << 28));  // leading ones of the four prefix bins
    if (prefix >= 4) {
      bypass_take(X, Q, k, 4);
      return (4u << rice) + egk_bypass(rice + 1, bad);
    }
    int j = prefix + 1 + rice;
    if (j <= k) return ((uint32_t)prefix << rice) + (bypass_take(X, Q, k, j) & ((1u << rice) - 1u));
    // rice == 4 and three ones: the last suffix bit does not fit the seven-bin division
    const uint32_t hi = bypass_take(X, Q, k, k) & 7u;
    return ((uint32_t)prefix << rice) + ((hi << 1) | (uint32_t)bypass());
  }
};

// Engine::hint_level_remaining is optional for the engines the parser is instantiated with: one without it compiles and
// behaves as before (overload resolution prefers the first form when the call is well formed).
template <class Eng>
HEIC_HD auto hint_level_remaining(Eng& e, int rice, int base_level, int) -> decltype(e.hint_level_remaining(rice, base_level)) {
  return e.hint_level_remaining(rice, base_level);
}
template <class Eng>
HEIC_HD void hint_level_remaining(Eng&, int, int, long) {}

#if defined(__CUDA_ARCH__) && !defined(HEIC_CABAC_INLINE_ENGINE)
// Out-of-line engine entry points for the device parser.  The engine lives in registers and travels by value (the
// compiler passes and returns the struct in registers), so a call costs a CALL/RET pair; in exchange the decoding
// routines exist once instead of at ~45 call sites.  Inlined everywhere the kernel was 7 K instructions (113 KB) against
// a 32 KB instruction cache and `stall_no_instruction` was its largest stall reason.
#define HEIC_CABAC_OUTLINED 1
struct EngRet {
  Engine e;
  uint32_t v;
  int bad;
};
static __device__ __noinline__ EngRet eng_decision(Engine e, uint32_t ctx_addr, uint32_t sm) {
  uint32_t s = *smem_ptr<uint8_t>(ctx_addr);
  EngRet r;
  r.v = (uint32_t)e.decision(smem_ptr<const CabacTabs>(sm), s);
  *smem_ptr<uint8_t>(ctx_addr) = (uint8_t)s;
  r.e = e;
  r.bad = 0;
  return r;
}
// sig_coeff_flag of scan positions n_start .. 1 of one sub-block (9.3.4.2.5): context of position k = nibble k of `nib`,
// entries `1 << stride_shift` bytes apart from ctx_addr.  One call per sub-block instead of one per bin.
static __device__ __noinline__ EngRet eng_sig_run(Engine e, uint32_t ctx_addr, uint64_t nib, int n_start, int stride_shift, uint32_t sm) {
  const CabacTabs* T = smem_ptr<const CabacTabs>(sm);
  uint32_t sig = 0;
  HEIC_NO_UNROLL
  for (int k = n_start; k > 0; k--) {
    const uint32_t a = ctx_addr + ((uint32_t)((nib >> (4 * k)) & 15u) << stride_shift);
    uint32_t s = *smem_ptr<uint8_t>(a);
    if (e.decision(T, s)) sig |= 1u << k;
    *smem_ptr<uint8_t>(a) = (uint8_t)s;
  }
  EngRet r;
  r.e = e;
  r.v = sig;
  r.bad = 0;
  return r;
}
// coeff_abs_level_greater1_flag of up to eight coefficients of a sub-block (9.3.4.2.6): ctx_addr is context 0 of the
// sub-block's context set; returns the flags as a mask, greater1Ctx and the first position with the flag set in `bad`.
static __device__ __noinline__ EngRet eng_gt1_run(Engine e, uint32_t ctx_addr, uint32_t sig, int stride_shift, uint32_t sm) {
  const CabacTabs* T = smem_ptr<const CabacTabs>(sm);
  uint32_t g1 = 0, m = sig;
  int greater1_ctx = 1, num = 0, last = -1;
  HEIC_NO_UNROLL
  while (m && num < 8) {
    const int k = 31 - __clz(m);
    m &= ~(1u << k);
    const uint32_t a = ctx_addr + ((uint32_t)greater1_ctx << stride_shift);
    uint32_t s = *smem_ptr<uint8_t>(a);
    const int f = e.decision(T, s);
    *smem_ptr<uint8_t>(a) = (uint8_t)s;
    num++;
    if (f) {
      g1 |= 1u << k;
      greater1_ctx = 0;
      if (last < 0) last = k;
    } else if (greater1_ctx > 0 && greater1_ctx < 3) {
      greater1_ctx++;
    }
  }
  EngRet r;
  r.e = e;
  r.v = g1 | (m << 16);  // m: the significant coefficients past the first eight (they carry no greater1 flag)
  r.bad = greater1_ctx | ((last + 1) << 8);
  return r;
}
static __device__ __noinline__ EngRet eng_bypass(Engine e) {
  EngRet r;
  r.v = (uint32_t)e.bypass();
  r.e = e;
  r.bad = 0;
  return r;
}
static __device__ __noinline__ EngRet eng_fl_bypass(Engine e, int n) {
  EngRet r;
  r.v = e.fl_bypass(n);
  r.e = e;
  r.bad = 0;
  return r;
}
static __device__ __noinline__ EngRet eng_tr_bypass(Engine e, uint32_t cmax) {
  EngRet r;
  r.v = e.tr_bypass(cmax);
  r.e = e;
  r.bad = 0;
  return r;
}
static __device__ __noinline__ EngRet eng_egk_bypass(Engine e, int k) {
  EngRet r;
  r.bad = 0;
  r.v = e.egk_bypass(k, r.bad);
  r.e = e;
  return r;
}
static __device__ __noinline__ EngRet eng_calr(Engine e, int rice) {
  EngRet r;
  r.bad = 0;
  r.v = e.coeff_abs_level_remaining(rice, r.bad);
  r.e = e;
  return r;
}
#endif

// 9.3.2.2 (arithmetic.rs:40-78): initValue -> pStateIdx << 1 | valMps
HEIC_HD uint8_t context_init_state(int init_value, int slice_qp) {
  int slope_idx = init_value >> 4, offset_idx = init_value & 15;
  int m = slope_idx * 5 - 45, n = (offset_idx << 3) - 16;
  int pre = clip3i(1, 126, ((m * clip3i(0, 51, slice_qp)) >> 4) + n);
  int mps = pre > 63;
  int p = mps ? pre - 64 : 63 - pre;
  return (uint8_t)((p << 1) | mps);
}

// ------------------------------------------------------------------------------------------------
// Syntax parser.  STRIDE is the distance in bytes between consecutive contexts of this thread's table
// (1 when a warp serves one substream, 32 when the lanes of a warp serve 32 substreams and their
// tables are interleaved so that equal context indices fall into one 32-byte row).
// ------------------------------------------------------------------------------------------------
template <int STRIDE, class Eng = Engine>
struct Parser {
  Eng e;
  // current CU
  int part_nxn, chroma_mode, cu_x, cu_y, cu_log2;
  uint32_t pu_modes;  // IntraPredModeY of the (up to) four prediction blocks, 8 bits each (no indexed arrays: they
                      // would live in local memory)
  int err;
  // What is touched once per transform unit or less -- the tile's arena pointers, its parameter structures and the QP
  // state of 8.6.1 -- is reached through accessors.  On the device it lives in the kernel's shared memory (the tile index
  // and the QP state in per-thread words, the arena bases once per CTA), NOT in registers: held in registers it cost 28 of
  // them for the whole kernel, and the register file is what bounds the CABAC kernel's occupancy (4 CTAs per SM at 64
  // registers against 3 at 80).  On the host (tests/emul, tests/synth, tests/fuzz) they are plain members.
  enum { CW_TP_LO = 0, CW_TP_HI, CW_PP_LO, CW_PP_HI, CW_QP_CODED, CW_QP_DELTA, CW_QP_Y, CW_QP_LAST, CW_QP_PRED, CW_QP_FIRST, CW_QG_X, CW_QG_Y, CW_COUNT };
#if defined(__CUDA_ARCH__)
  static constexpr uint32_t kColdStride = STRIDE == 32 ? 1024u : 64u;  // bytes between a thread's cold words (threads with one x 4)
  uint32_t sm;        // shared-window address of the kernel's dynamic shared memory (tables at 0, arena pointers behind them)
  uint32_t cold_off;  // shared-window address of this thread's first cold word
  HEIC_HD int& cold(int j) const { return *smem_ptr<int>(cold_off + (uint32_t)j * kColdStride); }
  HEIC_HD const Arenas* arenas() const { return smem_ptr<const Arenas>(sm + kSmemArenasOff); }
  // the tile's and its picture's parameter structures: pointers in the thread's cold words (two independent LDS each, instead
  // of the chain arena pointer -> tile index -> tiles[tile].pic -> pics[pic] through global memory)
  HEIC_HD const TileParams* TP() const {
    return reinterpret_cast<const TileParams*>((unsigned long long)(uint32_t)cold(CW_TP_LO) | ((unsigned long long)(uint32_t)cold(CW_TP_HI) << 32));
  }
  HEIC_HD const PicParams* PP() const {
    return reinterpret_cast<const PicParams*>((unsigned long long)(uint32_t)cold(CW_PP_LO) | ((unsigned long long)(uint32_t)cold(CW_PP_HI) << 32));
  }
  HEIC_HD uint32_t* tu_map_p() const { return arenas()->tu_map + TP()->tu_off; }
  HEIC_HD int16_t* coeff_p(int c) const { return arenas()->coeff + TP()->coeff_off[c]; }
  HEIC_HD uint8_t* ipm_p() const { return arenas()->ipm + TP()->map4_off; }
  HEIC_HD uint8_t* ct_depth_p() const { return arenas()->ct_depth + TP()->map8_off; }
  HEIC_HD uint8_t* qp_map_p() const { return arenas()->qp_map + TP()->map8_off; }
  HEIC_HD uint32_t* sao_p() const { return arenas()->sao + TP()->sao_off; }
#else
  const CabacTabs* T;
  uint8_t* ctx;
  const PicParams* pp;
  const TileParams* tp;
  uint32_t* tu_map;
  int16_t *coeff0, *coeff1, *coeff2;
  uint8_t *ipm, *ct_depth, *qp_map;
  uint32_t* sao;
  int cold_words[CW_COUNT];
  HEIC_HD int& cold(int j) { return cold_words[j]; }
  HEIC_HD const TileParams* TP() const { return tp; }
  HEIC_HD const PicParams* PP() const { return pp; }
  HEIC_HD uint32_t* tu_map_p() const { return tu_map; }
  HEIC_HD int16_t* coeff_p(int c) const { return c == 0 ? coeff0 : (c == 1 ? coeff1 : coeff2); }
  HEIC_HD uint8_t* ipm_p() const { return ipm; }
  HEIC_HD uint8_t* ct_depth_p() const { return ct_depth; }
  HEIC_HD uint8_t* qp_map_p() const { return qp_map; }
  HEIC_HD uint32_t* sao_p() const { return sao; }
#endif
  // QP state (8.6.1)
  HEIC_HD int& is_cu_qp_delta_coded() { return cold(CW_QP_CODED); }
  HEIC_HD int& cu_qp_delta_val() { return cold(CW_QP_DELTA); }
  HEIC_HD int& qp_y() { return cold(CW_QP_Y); }
  HEIC_HD int& last_qp_y() { return cold(CW_QP_LAST); }
  HEIC_HD int& qp_y_pred() { return cold(CW_QP_PRED); }
  HEIC_HD int& first_qg_in_row() { return cold(CW_QP_FIRST); }
  HEIC_HD int& qg_x() { return cold(CW_QG_X); }
  HEIC_HD int& qg_y() { return cold(CW_QG_Y); }

#if defined(__CUDA_ARCH__)
  uint32_t ctx_off;  // shared-window address of this thread's context table
  HEIC_HD const CabacTabs* tabs() const { return smem_ptr<const CabacTabs>(sm); }
  HEIC_HD uint32_t ld_ctx(int idx) const { return *smem_ptr<uint8_t>(ctx_off + idx * STRIDE); }
  HEIC_HD void st_ctx(int idx, uint32_t v) { *smem_ptr<uint8_t>(ctx_off + idx * STRIDE) = (uint8_t)v; }
#else
  HEIC_HD const CabacTabs* tabs() const { return T; }
  HEIC_HD uint32_t ld_ctx(int idx) const { return ctx[idx * STRIDE]; }
  HEIC_HD void st_ctx(int idx, uint32_t v) { ctx[idx * STRIDE] = (uint8_t)v; }
#endif
  HEIC_HD int dec(int idx) {
#if defined(HEIC_CABAC_OUTLINED)
    const EngRet r = eng_decision(e, ctx_off + idx * STRIDE, sm);
    e = r.e;
    return (int)r.v;
#else
    uint32_t s = ld_ctx(idx);
    e.hint_ctx(idx);
    const int bin = e.decision(tabs(), s);
    st_ctx(idx, s);
    return bin;
#endif
  }
  HEIC_HD void fail(int code) {
    if (!err) err = code;
  }

  HEIC_HD void init_contexts(int slice_qp) {
    for (int i = 0; i < NUM_CTX; i++) st_ctx(i, context_init_state(tabs()->init_value[i], slice_qp));
  }

  // bypass-coded elements
#if defined(HEIC_CABAC_OUTLINED)
  HEIC_HD uint32_t sig_run(int add, uint64_t nib, int n_start) {
    const EngRet r = eng_sig_run(e, ctx_off + add * STRIDE, nib, n_start, STRIDE == 32 ? 5 : 0, sm);
    e = r.e;
    return r.v;
  }
  HEIC_HD int byp() {
    const EngRet r = eng_bypass(e);
    e = r.e;
    return (int)r.v;
  }
  HEIC_HD uint32_t fl_bypass(int n) {
    const EngRet r = eng_fl_bypass(e, n);
    e = r.e;
    return r.v;
  }
  HEIC_HD uint32_t tr_bypass(uint32_t cmax) {
    const EngRet r = eng_tr_bypass(e, cmax);
    e = r.e;
    return r.v;
  }
  HEIC_HD uint32_t egk_bypass(int k) {
    const EngRet r = eng_egk_bypass(e, k);
    e = r.e;
    if (r.bad) fail(-3);
    return r.v;
  }
  HEIC_HD uint32_t coeff_abs_level_remaining(int rice, int) {
    const EngRet r = eng_calr(e, rice);
    e = r.e;
    if (r.bad) fail(-3);
    return r.v;
  }
#else
  HEIC_HD uint32_t sig_run(int add, uint64_t nib, int n_start) {
    uint32_t sig = 0;
    for (int k = n_start; k > 0; k--)
      if (dec(add + (int)((nib >> (4 * k)) & 15u))) sig |= 1u << k;
    return sig;
  }
  HEIC_HD int byp() { return e.bypass(); }
  HEIC_HD uint32_t fl_bypass(int n) { return e.fl_bypass(n); }
  HEIC_HD uint32_t tr_bypass(uint32_t cmax) { return e.tr_bypass(cmax); }
  HEIC_HD uint32_t egk_bypass(int k) {  // decoder.rs:206-222 with 32-bit arithmetic (SURVEY Appendix B #11)
    int ones = 0;
    while (e.bypass()) {
      if (++ones > 31) {
        fail(-3);
        return 0;
      }
    }
    uint32_t suffix = e.fl_bypass(ones + k);
    return (((1u << ones) - 1u) << k) + suffix;
  }
  HEIC_HD uint32_t coeff_abs_level_remaining(int rice, int base_level) {  // decoder.rs:224-261
    hint_level_remaining(e, rice, base_level, 0);
    uint32_t prefix = 0;
    while (prefix < 4 && e.bypass()) prefix++;
    if (prefix < 4) return (prefix << rice) + e.fl_bypass(rice);
    return (4u << rice) + egk_bypass(rice + 1);
  }
#endif

  // ---- 7.3.8.3 sao() (todo!() at slice.rs:249-251) -------------------------------------------
  HEIC_HD void parse_sao(int rx, int ry) {
    const PicParams* pp = PP();
    const TileParams* tp = TP();
    uint32_t* sao = sao_p();
    uint32_t* p = sao + (size_t)(ry * pp->wctb + rx) * 4;
    int merge_left = 0, merge_up = 0;
    if (rx > 0) merge_left = dec(CTX_SAO_MERGE);
    if (ry > 0 && !merge_left) merge_up = dec(CTX_SAO_MERGE);
    if (merge_left || merge_up) {
      const uint32_t* q = merge_left ? p - 4 : p - (size_t)pp->wctb * 4;
      p[0] = q[0];
      p[1] = q[1];
      p[2] = q[2];
      p[3] = 0;
      return;
    }
    uint32_t w0 = 0, w1 = 0, w2 = 0;
    int type_c = 0, class_c = 0;
    int n_comp = pp->chroma ? 3 : 1;
    for (int c = 0; c < n_comp; c++) {
      if (!((c == 0 && tp->sao_luma) || (c > 0 && tp->sao_chroma))) continue;
      int type;
      if (c == 2) {
        type = type_c;
      } else {  // sao_type_idx: TR cMax 2, bin 0 context coded, bin 1 bypass (decoder.rs:93-100)
        type = 0;
        if (dec(CTX_SAO_TYPE)) type = byp() ? 2 : 1;
        if (c == 1) type_c = type;
      }
      if (!type) continue;
      uint32_t abs4 = 0;  // four sao_offset_abs, 4 bits each
      for (int i = 0; i < 4; i++) abs4 |= tr_bypass(7) << (4 * i);
      uint32_t v = (uint32_t)type;
      if (type == 1) {
        for (int i = 0; i < 4; i++) {
          const int a = (int)((abs4 >> (4 * i)) & 15u);
          const int neg = a ? byp() : 0;
          const int o = neg ? -a : a;
          v |= ((uint32_t)o & 15u) << (8 + 4 * i);
        }
        v |= fl_bypass(5) << 2;  // sao_band_position
      } else {
        int cl;
        if (c == 0) cl = (int)fl_bypass(2);
        else if (c == 1) cl = class_c = (int)fl_bypass(2);
        else cl = class_c;
        v |= (uint32_t)cl << 2;
        v |= (abs4 & 15u) << 8;
        v |= ((abs4 >> 4) & 15u) << 12;
        v |= ((uint32_t)(-(int)((abs4 >> 8) & 15u)) & 15u) << 16;
        v |= ((uint32_t)(-(int)((abs4 >> 12) & 15u)) & 15u) << 20;
      }
      if (c == 0) w0 = v;
      else if (c == 1) w1 = v;
      else w2 = v;
    }
    p[0] = w0;
    p[1] = w1;
    p[2] = w2;
    p[3] = 0;
  }

  // ---- scan helpers (6.5.3-6.5.5) ---------------------------------------------------------------
  // position i of a (1<<lg)x(1<<lg) scan -> x | y << 4
  HEIC_HD uint32_t scan_xy(int scan_idx, int lg, int i) const {
    if (lg == 0) return 0;
    if (scan_idx == 0) {
      uint32_t v;
      if (lg == 2) {
        v = tabs()->diag4[i];
        return (v & 3u) | ((v >> 2) << 4);
      }
      if (lg == 3) {
        v = tabs()->diag8[i];
        return (v & 7u) | ((v >> 3) << 4);
      }
      v = tabs()->diag2[i];
      return (v & 1u) | ((v >> 1) << 4);
    }
    uint32_t a = (uint32_t)i & ((1u << lg) - 1u), b = (uint32_t)i >> lg;
    return scan_idx == 1 ? (a | (b << 4)) : (b | (a << 4));
  }
  HEIC_HD int scan_inv(int scan_idx, int lg, int x, int y) const {
    if (lg == 0) return 0;
    if (scan_idx == 0) {
      if (lg == 2) return tabs()->inv_diag4[(y << 2) | x];
      if (lg == 3) return tabs()->inv_diag8[(y << 3) | x];
      return tabs()->inv_diag2[(y << 1) | x];
    }
    return scan_idx == 1 ? ((y << lg) | x) : ((x << lg) | y);
  }

  HEIC_HD int last_sig_coeff_prefix(int ctx_base, int c_idx, int log2) {  // decoder.rs:109-130
    int ctx_offset, ctx_shift;
    if (c_idx == 0) {
      ctx_offset = 3 * (log2 - 2) + ((log2 - 1) >> 2);
      ctx_shift = (log2 + 1) >> 2;
    } else {
      ctx_offset = 15;
      ctx_shift = log2 - 2;
    }
    int c_max = (log2 << 1) - 1, v = 0;
    while (v < c_max && dec(ctx_base + (v >> ctx_shift) + ctx_offset)) v++;
    return v;
  }

  // ---- 7.3.8.11 residual_coding + 9.3.4.2.4-7; writes TransCoeffLevel (raster n x n) to out -------
  // Split into a prologue (transform_skip_flag, last significant position) and one call per 4x4 sub-block, so that the
  // same code serves the nested walk (host) and the flat per-sub-block loop of the device (coding_tree_unit).
  struct Rc {
    // the block's constants and the greater1 state carried between sub-blocks, packed (the structure is live across every
    // decoding call of the block, and the kernel is bound by its registers):
    //   log2 | c_idx << 3 | scan_idx << 5 | sig_off << 7 | last_sub_block << 13 | last_scan_pos << 19 | tskip << 23 |
    //   sign_hiding << 24 | greater1_ctx << 25 | first_sub_block << 27
    uint32_t k;
    int i;          // next sub-block (scan order, counting down)
    uint64_t csbf;  // coded_sub_block_flag, bit ys*8+xs
    int16_t* out;
    HEIC_HD int tskip() const { return (int)((k >> 23) & 1u); }
  };
  HEIC_HD void rc_begin(Rc& r, int log2, int c_idx, int pred_mode, int16_t* out) {
    const PicParams* pp = PP();
    int tskip = 0;
    if (pp->tskip_enabled && log2 <= 2) tskip = dec(CTX_TSKIP + (c_idx ? 1 : 0));
    int last_x, last_y;
    {
      uint32_t pre = 0;  // both prefixes, 8 bits each, through one call site
HEIC_NO_UNROLL
      for (int d = 0; d < 2; d++) pre |= (uint32_t)last_sig_coeff_prefix(d ? CTX_LAST_Y : CTX_LAST_X, c_idx, log2) << (8 * d);
HEIC_NO_UNROLL
      for (int d = 0; d < 2; d++) {  // suffixes follow both prefixes (7.3.8.11)
        const int pv = (int)((pre >> (8 * d)) & 0xffu);
        if (pv > 3) {
          const int nb = (pv >> 1) - 1;
          const int full = (1 << nb) * (2 + (pv & 1)) + (int)fl_bypass(nb);
          pre = (pre & ~(0xffu << (8 * d))) | ((uint32_t)full << (8 * d));
        }
      }
      last_x = (int)(pre & 0xffu);
      last_y = (int)((pre >> 8) & 0xffu);
    }
    int scan_idx = 0;
    if (log2 == 2 || (log2 == 3 && c_idx == 0)) {
      if (pred_mode >= 6 && pred_mode <= 14) scan_idx = 2;
      else if (pred_mode >= 22 && pred_mode <= 30) scan_idx = 1;
    }
    if (scan_idx == 2) {
      int t = last_x;
      last_x = last_y;
      last_y = t;
    }
    const int lg_sb = log2 - 2;
    const int last_sub_block = scan_inv(scan_idx, lg_sb, last_x >> 2, last_y >> 2);
    const int last_scan_pos = scan_inv(scan_idx, 2, last_x & 3, last_y & 3);
    // sigCtx offset for the non-4x4, non-DC case (9.3.4.2.5)
    const int sig_off = c_idx == 0 ? ((log2 == 3) ? (scan_idx == 0 ? 9 : 15) : 21) : ((log2 == 3) ? 9 : 12);
    r.k = (uint32_t)log2 | ((uint32_t)c_idx << 3) | ((uint32_t)scan_idx << 5) | ((uint32_t)sig_off << 7) |
          ((uint32_t)last_sub_block << 13) | ((uint32_t)last_scan_pos << 19) | ((uint32_t)tskip << 23) |
          ((uint32_t)(pp->sign_hiding ? 1 : 0) << 24) | (1u << 25) | (1u << 27);
    r.i = last_sub_block;
    r.csbf = 0;
    r.out = out;
  }
  HEIC_HD void rc_subblock(Rc& r) {  // sub-block r.i
    const int log2 = (int)(r.k & 7u), c_idx = (int)((r.k >> 3) & 3u), scan_idx = (int)((r.k >> 5) & 3u), n = 1 << log2, lg_sb = log2 - 2,
              sb_w = 1 << lg_sb;
    const int sig_base = CTX_SIG + (c_idx ? 27 : 0), sig_off = (int)((r.k >> 7) & 63u), last_sub_block = (int)((r.k >> 13) & 63u),
              last_scan_pos = (int)((r.k >> 19) & 15u);
    const int i = r.i;
    int16_t* out = r.out;
    uint64_t& csbf = r.csbf;
    int greater1_ctx = (int)((r.k >> 25) & 3u);
    int first_sub_block = (int)((r.k >> 27) & 1u);
    uint32_t sxy = scan_xy(scan_idx, lg_sb, i);
    const int xs = (int)(sxy & 15u), ys = (int)(sxy >> 4);
    int right = (xs < sb_w - 1) ? (int)((csbf >> (ys * 8 + xs + 1)) & 1u) : 0;
    int below = (ys < sb_w - 1) ? (int)((csbf >> ((ys + 1) * 8 + xs)) & 1u) : 0;
    int infer_sb_dc = 0, coded = 1;
    if (i < last_sub_block && i > 0) {
      coded = dec(CTX_CSBF + (c_idx ? 2 : 0) + (right | below));
      infer_sb_dc = 1;
    }
    if (coded) csbf |= (uint64_t)1 << (ys * 8 + xs);
    uint32_t sig = 0;
    int n_start = 15;
    if (i == last_sub_block) {
      n_start = last_scan_pos - 1;
      sig = 1u << last_scan_pos;
    }
    if (coded) {
      const int prev_csbf = right | (below << 1);
      // sigCtx (9.3.4.2.5) of all 16 scan positions of this sub-block as one word of nibbles + one additive term
      const uint64_t nib = tabs()->sig_nib[log2 == 2 ? scan_idx : 3 + scan_idx * 4 + prev_csbf];
      const int add = sig_base + (log2 == 2 ? 0 : ((c_idx == 0 && (xs | ys)) ? 3 : 0) + sig_off);
      if (n_start > 0) sig |= sig_run(add, nib, n_start);
      if (n_start >= 0) {
        if (infer_sb_dc && sig == 0) {
          sig = 1u;  // inferred DC of a coded sub-block with no other significant coefficient
        } else {
          // the DC coefficient of the whole block has its own context (sigCtx 0)
          const int ctx0 = (log2 > 2 && i == 0) ? sig_base : add + (int)(nib & 15u);
          if (dec(ctx0)) sig |= 1u;
        }
      }
    }
    if (!sig) return;
    // 9.3.4.2.6 / 9.3.4.2.7: up to 8 greater1 flags, one greater2 flag
    int ctx_set = (i > 0 && c_idx == 0) ? 2 : 0;
    if (!first_sub_block && greater1_ctx == 0) ctx_set++;
    first_sub_block = 0;
    greater1_ctx = 1;
    uint32_t g1 = 0, beyond8 = 0;
    int last_g1_pos = -1;
    const int last_sig = 31 - HEIC_CLZ(sig);
    const int first_sig = 31 - HEIC_CLZ(sig & (0u - sig));
#if defined(HEIC_CABAC_OUTLINED)
    {
      const EngRet r = eng_gt1_run(e, ctx_off + (CTX_GT1 + (c_idx ? 16 : 0) + (ctx_set << 2)) * STRIDE, sig, STRIDE == 32 ? 5 : 0, sm);
      e = r.e;
      g1 = r.v & 0xffffu;
      beyond8 = r.v >> 16;
      greater1_ctx = r.bad & 0xff;
      last_g1_pos = (r.bad >> 8) - 1;
    }
#else
    {
      uint32_t m = sig;
      int num_g1 = 0;
      while (m && num_g1 < 8) {
        int k = 31 - HEIC_CLZ(m);
        m &= ~(1u << k);
        int f = dec(CTX_GT1 + (c_idx ? 16 : 0) + (ctx_set << 2) + greater1_ctx);
        num_g1++;
        if (f) {
          g1 |= 1u << k;
          greater1_ctx = 0;
          if (last_g1_pos < 0) last_g1_pos = k;
        } else if (greater1_ctx > 0 && greater1_ctx < 3) {
          greater1_ctx++;
        }
      }
      beyond8 = m;
    }
#endif
    r.k = (r.k & ~(7u << 25)) | ((uint32_t)greater1_ctx << 25);  // first_sub_block = 0, greater1Ctx for the next sub-block
    const int sign_hidden = ((r.k >> 24) & 1u) && (last_sig - first_sig > 3);
    int g2 = 0;
    if (last_g1_pos >= 0) g2 = dec(CTX_GT2 + (c_idx ? 4 : 0) + ctx_set);
    // coeff_sign_flag: one bypass bin per coefficient in scan order (none for the hidden one, which comes last):
    // read them in one go, most significant bit = first coefficient
    const int n_sign = HEIC_POPC(sig) - (sign_hidden ? 1 : 0);
    uint32_t sign_bits = n_sign ? fl_bypass(n_sign) << (32 - n_sign) : 0u;
    // baseLevel = 1 + greater1 + greater2, and which coefficients carry a coeff_abs_level_remaining (9.3.3.11 / 7.3.8.11:
    // baseLevel == ((numSigCoeff < 8) ? ((i == firstG1) ? 3 : 2) : 1)) as bit masks, worked out once per sub-block: among the
    // first eight that is "greater1 set" -- for the one coefficient that also has a greater2 flag "greater2 set" -- and
    // every coefficient after the first eight.
    const uint32_t first_g1 = last_g1_pos >= 0 ? 1u << last_g1_pos : 0u;
    const uint32_t g2x = g2 ? first_g1 : 0u;
    const uint32_t need_rem = (g1 & ~first_g1) | g2x | beyond8;
    int sum_abs = 0, rice = 0;
    uint32_t m = sig;
    while (m) {
      int k = 31 - HEIC_CLZ(m);
      m &= ~(1u << k);
      int abs_level = 1 + (int)((g1 >> k) & 1u) + (int)((g2x >> k) & 1u);
      if ((need_rem >> k) & 1u) {
        uint32_t rem = coeff_abs_level_remaining(rice, abs_level);
        if (rem > 32768u) {
          fail(-3);
          return;
        }
        abs_level += (int)rem;
        if (abs_level > 3 * (1 << rice)) rice = rice < 4 ? rice + 1 : 4;  // decoder.rs:230-236
      }
      int v = (sign_bits >> 31) ? -abs_level : abs_level;
      sign_bits <<= 1;
      if (sign_hidden) {
        sum_abs += abs_level;
        if (k == first_sig && (sum_abs & 1)) v = -v;
      }
      uint32_t pxy = scan_xy(scan_idx, 2, k);
      int xc = (xs << 2) + (int)(pxy & 15u), yc = (ys << 2) + (int)(pxy >> 4);
      out[yc * n + xc] = (int16_t)clip3i(-32768, 32767, v);
    }
  }
  HEIC_HD int residual_coding(int log2, int c_idx, int pred_mode, int16_t* out) {
    Rc r;
    rc_begin(r, log2, c_idx, pred_mode, out);
    for (; r.i >= 0 && !err; r.i--) rc_subblock(r);
    return r.tskip();
  }

  // ---- 8.6.1 ------------------------------------------------------------------------------------
  HEIC_HD void set_qp_pred(int x_qg, int y_qg) {
    const PicParams* pp = PP();
    const TileParams* tp = TP();
    const uint8_t* qp_map = qp_map_p();
    int qp_prev = first_qg_in_row() ? tp->slice_qp : last_qp_y();
    first_qg_in_row() = 0;
    int ctb_mask = (1 << pp->log2_ctb) - 1;
    int qa = qp_prev, qb = qp_prev;
    if (x_qg & ctb_mask) qa = qp_map[(y_qg >> 3) * pp->w8 + ((x_qg - 1) >> 3)];
    if (y_qg & ctb_mask) qb = qp_map[((y_qg - 1) >> 3) * pp->w8 + (x_qg >> 3)];
    qp_y_pred() = (qa + qb + 1) >> 1;
    qp_y() = qp_y_pred();
  }

  // ---- 7.3.8.10 transform_unit ------------------------------------------------------------------
  // z4: z-order index of the TU's 4x4 origin inside its CTB; ctb_addr: raster CTB address.  Split into the part before
  // the residuals (tu_begin), the choice of a component's residual block (tu_component) and the tu_map record (tu_end).
  struct Tu {
    int log2, luma_mode, has_chroma, cbf_luma, cbf_cb, cbf_cr;
    uint32_t ti, ts;  // tu_map index; transform_skip_flag of the three components
  };
  HEIC_HD void tu_begin(Tu& t, int x0, int y0, int log2, int blk_idx, int cbf_luma, int cbf_cb, int cbf_cr, uint32_t ctb_addr,
                        uint32_t z4) {
    const PicParams* pp = PP();
    const int pb_shift = part_nxn ? cu_log2 - 1 : cu_log2;
    const int pu_idx = (((x0 - cu_x) >> pb_shift) & 1) | ((((y0 - cu_y) >> pb_shift) & 1) << 1);
    t.luma_mode = (int)((pu_modes >> (8 * pu_idx)) & 0xffu);
    t.has_chroma = pp->chroma && (log2 > 2 || blk_idx == 3);
    t.log2 = log2;
    const int any_cbf = cbf_luma | cbf_cb | cbf_cr;  // 7.3.8.10: parent-inherited chroma cbfs count for blkIdx 0..2 too
    if (!t.has_chroma) cbf_cb = cbf_cr = 0;
    t.cbf_luma = cbf_luma;
    t.cbf_cb = cbf_cb;
    t.cbf_cr = cbf_cr;
    if (any_cbf && pp->cu_qp_delta_enabled && !is_cu_qp_delta_coded()) {
      // cu_qp_delta_abs: prefix TR cMax 5 (bin 0 ctx 0, bins 1-4 ctx 1) + EG0 suffix (decoder.rs:263-284)
      int v = 0;
      while (v < 5 && dec(CTX_CU_QP_DELTA + (v ? 1 : 0))) v++;
      if (v == 5) v += (int)egk_bypass(0);
      int neg = v ? byp() : 0;
      is_cu_qp_delta_coded() = 1;
      cu_qp_delta_val() = neg ? -v : v;
      if (cu_qp_delta_val() < -26 || cu_qp_delta_val() > 25) fail(-3);
      qp_y() = (qp_y_pred() + cu_qp_delta_val() + 52) % 52;
    }
    const int ctb4 = 1 << (pp->log2_ctb - 2);
    t.ti = ctb_addr * (uint32_t)(ctb4 * ctb4) + z4;
    t.ts = 0;
  }
  // residual block of component c: false when its cbf is 0, else the arguments of rc_begin
  HEIC_HD bool tu_component(const Tu& t, int c, int& log2, int& pred_mode, int16_t*& dst) const {
    const int cbf = c == 0 ? t.cbf_luma : (c == 1 ? t.cbf_cb : t.cbf_cr);
    if (!cbf) return false;
    // luma: 16 coefficients per tu_map entry; chroma: 4, at the entry of the 8x8 luma area the block belongs to (the CTB's
    // entry count is a multiple of 4, so ti >> 2 is the chroma block index)
    dst = c == 0 ? coeff_p(0) + (size_t)t.ti * 16 : coeff_p(c) + (size_t)(t.ti >> 2) * 16;
    log2 = c ? (t.log2 > 2 ? t.log2 - 1 : 2) : t.log2;
    pred_mode = c ? chroma_mode : t.luma_mode;
    return true;
  }
  HEIC_HD void tu_end(const Tu& t) {
    const int ts0 = (int)(t.ts & 1u), ts1 = (int)((t.ts >> 1) & 1u), ts2 = (int)((t.ts >> 2) & 1u);
    tu_map_p()[t.ti] = 1u | ((uint32_t)(t.log2 - 2) << 1) | ((uint32_t)t.cbf_luma << 3) | ((uint32_t)t.cbf_cb << 4) |
                   ((uint32_t)t.cbf_cr << 5) | ((uint32_t)t.has_chroma << 6) | ((uint32_t)t.luma_mode << 7) |
                   ((uint32_t)chroma_mode << 13) | ((uint32_t)qp_y() << 19) | ((uint32_t)ts0 << 25) |
                   ((uint32_t)ts1 << 26) | ((uint32_t)ts2 << 27);
  }
  // ---- 7.3.8.8 transform_tree, walked iteratively in z-order over the CU's 4x4 blocks -----------
  struct Tt {
    uint32_t z, n4;             // next 4x4 block of the CU in z-order, their number
    uint32_t cb_mask, cr_mask;  // bit d: cbf_cb / cbf_cr of the current node at trafoDepth d
    uint32_t step;              // 4x4 blocks covered by the leaf found last
  };
  HEIC_HD void tt_begin(Tt& t) const {
    t.z = 0;
    t.n4 = 1u << (2 * (cu_log2 - 2));
    t.cb_mask = t.cr_mask = 0;
    t.step = 0;
  }
  // Descends from the largest block whose origin is t.z to its leaf (split_transform_flag, cbf_cb, cbf_cr, cbf_luma)
  // and starts that transform unit.
  HEIC_HD void tt_leaf(Tt& t, Tu& tu, uint32_t ctb_addr, uint32_t z4_cu) {
    const PicParams* pp = PP();
    const int intra_split = part_nxn;
    const int max_depth = pp->max_trafo_depth_intra + intra_split;
    const uint32_t z = t.z;
    int lvl = cu_log2 - 2;  // largest block whose origin is z
    if (z) {
      int tz = (31 - HEIC_CLZ(z & (0u - z))) >> 1;
      if (tz < lvl) lvl = tz;
    }
    int log2 = lvl + 2;
    for (;;) {
      const int depth = cu_log2 - log2;
      int split;
      if (log2 <= pp->log2_max_tb && log2 > pp->log2_min_tb && depth < max_depth && !(intra_split && depth == 0))
        split = dec(CTX_SPLIT_TRANSFORM + 5 - log2);
      else
        split = (log2 > pp->log2_max_tb) || (intra_split && depth == 0);
      int cbf_cb = 0, cbf_cr = 0;
      if (pp->chroma) {
        int par_cb = depth ? (int)((t.cb_mask >> (depth - 1)) & 1u) : 1;
        int par_cr = depth ? (int)((t.cr_mask >> (depth - 1)) & 1u) : 1;
        if (log2 > 2) {
          if (par_cb) cbf_cb = dec(CTX_CBF_CHROMA + depth);
          if (par_cr) cbf_cr = dec(CTX_CBF_CHROMA + depth);
        } else {  // inferred from the parent when log2TrafoSize == 2
          cbf_cb = depth ? par_cb : 0;
          cbf_cr = depth ? par_cr : 0;
        }
      }
      t.cb_mask = (t.cb_mask & ~(1u << depth)) | ((uint32_t)cbf_cb << depth);
      t.cr_mask = (t.cr_mask & ~(1u << depth)) | ((uint32_t)cbf_cr << depth);
      if (!split) {
        int cbf_luma = dec(CTX_CBF_LUMA + (depth == 0 ? 1 : 0));  // always present for intra CUs
        int x0 = cu_x + (int)(compact1by1(z) << 2), y0 = cu_y + (int)(compact1by1(z >> 1) << 2);
        tu_begin(tu, x0, y0, log2, (int)(z & 3u), cbf_luma, cbf_cb, cbf_cr, ctb_addr, z4_cu + z);
        break;
      }
      log2--;
    }
    t.step = 1u << (2 * (log2 - 2));
  }
  // residuals of the transform unit just started, then its tu_map record (the nested form of the device's flat loop)
  HEIC_HD void tu_residuals(Tu& t) {
    if (err) return;
    // one residual_coding call site for the three components keeps the kernel's instruction footprint small
HEIC_NO_UNROLL
    for (int c = 0; c < 3; c++) {
      int lg, pm;
      int16_t* dst;
      if (!tu_component(t, c, lg, pm, dst)) continue;
      t.ts |= (uint32_t)residual_coding(lg, c, pm, dst) << c;
    }
    tu_end(t);
  }
  HEIC_HD void transform_tree(uint32_t ctb_addr, uint32_t z4_cu) {
    Tt t;
    tt_begin(t);
    while (t.z < t.n4 && !err) {
      Tu tu;
      tt_leaf(t, tu, ctb_addr, z4_cu);
      tu_residuals(tu);
      t.z += t.step;
    }
  }

  // ---- 8.4.2 ------------------------------------------------------------------------------------
  HEIC_HD int derive_luma_mode(int x, int y, int prev_flag, int mpm_idx, int rem) {
    const PicParams* pp = PP();
    const uint8_t* ipm = ipm_p();
    int cand_a = 1, cand_b = 1;
    if (x > 0) cand_a = ipm[(y >> 2) * pp->w4 + ((x - 1) >> 2)];
    if (y > 0 && ((y - 1) >> pp->log2_ctb) == (y >> pp->log2_ctb)) cand_b = ipm[((y - 1) >> 2) * pp->w4 + (x >> 2)];
    int c0, c1, c2;
    if (cand_a == cand_b) {
      if (cand_a < 2) {
        c0 = 0;
        c1 = 1;
        c2 = 26;
      } else {
        c0 = cand_a;
        c1 = 2 + ((cand_a + 29) & 31);
        c2 = 2 + ((cand_a - 2 + 1) & 31);
      }
    } else {
      c0 = cand_a;
      c1 = cand_b;
      if (cand_a != 0 && cand_b != 0) c2 = 0;
      else if (cand_a != 1 && cand_b != 1) c2 = 1;
      else c2 = 26;
    }
    if (prev_flag) return mpm_idx == 0 ? c0 : (mpm_idx == 1 ? c1 : c2);
    int t;
    if (c0 > c1) t = c0, c0 = c1, c1 = t;
    if (c0 > c2) t = c0, c0 = c2, c2 = t;
    if (c1 > c2) t = c1, c1 = c2, c2 = t;
    int mode = rem;
    if (mode >= c0) mode++;
    if (mode >= c1) mode++;
    if (mode >= c2) mode++;
    return mode;
  }

  // ---- 7.3.8.5 coding_unit (I slice) -------------------------------------------------------------
  // prediction part of the CU (everything before its transform tree)
  HEIC_HD void cu_begin(int x0, int y0, int log2) {
    const PicParams* pp = PP();
    uint8_t* ipm = ipm_p();
    const int n = 1 << log2;
    cu_x = x0;
    cu_y = y0;
    cu_log2 = log2;
    part_nxn = 0;
    if (pp->cu_qp_delta_enabled) {
      int mask = (1 << pp->log2_min_cu_qp_delta_size) - 1;
      int x_qg = x0 & ~mask, y_qg = y0 & ~mask;
      if (x_qg != qg_x() || y_qg != qg_y()) {
        qg_x() = x_qg;
        qg_y() = y_qg;
        set_qp_pred(x_qg, y_qg);
      }
      qp_y() = (qp_y_pred() + cu_qp_delta_val() + 52) % 52;
    }
    if (log2 == pp->log2_min_cb) part_nxn = !dec(CTX_PART_MODE);  // decoder.rs:136-149
    if (part_nxn && log2 == 3 && pp->log2_min_tb >= 3) {
      fail(-3);
      return;
    }
    const int n_pu = part_nxn ? 4 : 1, pb = part_nxn ? n >> 1 : n;
    uint32_t prev = 0;  // prev_intra_luma_pred_flag of every prediction block first (7.3.8.5)
    for (int k = 0; k < n_pu; k++) prev |= (uint32_t)dec(CTX_PREV_INTRA) << k;
    pu_modes = 0;
    for (int k = 0; k < n_pu; k++) {
      int mpm_idx = 0, rem = 0;
      const int prev_k = (int)((prev >> k) & 1u);
      if (prev_k) mpm_idx = (int)tr_bypass(2);
      else rem = (int)fl_bypass(5);
      int px = x0 + (k & 1) * pb, py = y0 + (k >> 1) * pb;
      int mode = derive_luma_mode(px, py, prev_k, mpm_idx, rem);
      pu_modes |= (uint32_t)mode << (8 * k);
      // neighbours only ever read the right column and the bottom row of a prediction block
      const int b4 = pb >> 2, x4 = px >> 2, y4 = py >> 2;
      for (int j = 0; j < b4; j++) ipm[(y4 + j) * pp->w4 + x4 + b4 - 1] = (uint8_t)mode;
      for (int j = 0; j < b4 - 1; j++) ipm[(y4 + b4 - 1) * pp->w4 + x4 + j] = (uint8_t)mode;
    }
    if (!part_nxn) pu_modes *= 0x01010101u;
    chroma_mode = 0;
    if (pp->chroma) {  // intra_chroma_pred_mode (decoder.rs:23-35,192-204) + 8.4.3
      int idx = 4;
      if (dec(CTX_CHROMA_PRED)) idx = (int)fl_bypass(2);
      const int luma = (int)(pu_modes & 0xffu);
      if (idx == 4) {
        chroma_mode = luma;
      } else {
        int m = idx == 0 ? 0 : (idx == 1 ? 26 : (idx == 2 ? 10 : 1));
        chroma_mode = (m == luma) ? 34 : m;
      }
    }
  }
  HEIC_HD void cu_end() {
    const PicParams* pp = PP();
    uint8_t* qp_map = qp_map_p();
    // QpY of the CU (8.6.1): CuQpDeltaVal decoded anywhere inside the CU applies to all of it
    const int n = 1 << cu_log2;
    for (int yy = cu_y >> 3; yy < (cu_y + n) >> 3; yy++)
      for (int xx = cu_x >> 3; xx < (cu_x + n) >> 3; xx++) qp_map[yy * pp->w8 + xx] = (uint8_t)qp_y();
    last_qp_y() = qp_y();
  }
  HEIC_HD void coding_unit(int x0, int y0, int log2, uint32_t ctb_addr, uint32_t z4_cu) {
    cu_begin(x0, y0, log2);
    if (err) return;
    transform_tree(ctb_addr, z4_cu);
    cu_end();
  }

  // ---- 7.3.8.4 coding_quadtree (todo!() at slice.rs:253-255), iterative z-order walk of one CTB ---
  // One step of the walk: from the minimum-size block z (z-order inside the CTB) descend through split_cu_flag to the
  // coding unit that starts there.  False: the quadrant lies outside the picture and was skipped (z advanced).
  HEIC_HD bool ctu_next_cu(uint32_t& z, int x_ctb, int y_ctb, int& x0_out, int& y0_out, int& log2_out) {
    const PicParams* pp = PP();
    uint8_t* ct_depth = ct_depth_p();
    const int log2_ctb = pp->log2_ctb, log2_min_cb = pp->log2_min_cb;
    const int max_lvl = log2_ctb - log2_min_cb;
    int lvl = max_lvl;
    if (z) {
      int tz = (31 - HEIC_CLZ(z & (0u - z))) >> 1;
      if (tz < lvl) lvl = tz;
    }
    int log2 = log2_min_cb + lvl;
    const int x0 = x_ctb + (int)(compact1by1(z) << log2_min_cb), y0 = y_ctb + (int)(compact1by1(z >> 1) << log2_min_cb);
    if (x0 >= pp->w || y0 >= pp->h) {  // quadrant entirely outside the picture: not coded
      z += 1u << (2 * lvl);
      return false;
    }
    for (;;) {
      const int depth = log2_ctb - log2, n = 1 << log2;
      int split;
      if (x0 + n <= pp->w && y0 + n <= pp->h && log2 > log2_min_cb) {
        int inc = 0;
        if (x0 > 0 && ct_depth[(y0 >> 3) * pp->w8 + ((x0 - 1) >> 3)] > depth) inc++;
        if (y0 > 0 && ct_depth[((y0 - 1) >> 3) * pp->w8 + (x0 >> 3)] > depth) inc++;
        split = dec(CTX_SPLIT_CU + inc);
      } else {
        split = log2 > log2_min_cb;
      }
      if (pp->cu_qp_delta_enabled && log2 >= pp->log2_min_cu_qp_delta_size) {
        is_cu_qp_delta_coded() = 0;
        cu_qp_delta_val() = 0;
      }
      if (!split) break;
      log2--;
    }
    {
      const int depth = log2_ctb - log2, b8 = 1 << (log2 - 3), x8 = x0 >> 3, y8 = y0 >> 3;
      for (int j = 0; j < b8; j++) ct_depth[(y8 + j) * pp->w8 + x8 + b8 - 1] = (uint8_t)depth;
      for (int j = 0; j < b8 - 1; j++) ct_depth[(y8 + b8 - 1) * pp->w8 + x8 + j] = (uint8_t)depth;
    }
    x0_out = x0;
    y0_out = y0;
    log2_out = log2;
    return true;
  }

  HEIC_HD void coding_tree_unit(int rx, int ry) {
    const PicParams* pp = PP();
    const TileParams* tp = TP();
    const int log2_ctb = pp->log2_ctb, log2_min_cb = pp->log2_min_cb;
    const uint32_t ctb_addr = (uint32_t)(ry * pp->wctb + rx);
    const int x_ctb = rx << log2_ctb, y_ctb = ry << log2_ctb;
    if (!pp->cu_qp_delta_enabled) qp_y() = tp->slice_qp;
    if (tp->sao_luma || tp->sao_chroma) parse_sao(rx, ry);
    const uint32_t n_min = 1u << (2 * (log2_ctb - log2_min_cb));
    uint32_t z = 0;
    while (z < n_min && !err) {
      int x0, y0, log2;
      const uint32_t z_cu = z;
      if (!ctu_next_cu(z, x_ctb, y_ctb, x0, y0, log2)) continue;
      coding_unit(x0, y0, log2, ctb_addr, z_cu << (2 * (log2_min_cb - 2)));
      z += 1u << (2 * (log2 - log2_min_cb));
    }
  }
};

// ------------------------------------------------------------------------------------------------
// 7.3.8.1 slice_segment_data(): the CTU loop of slice.rs:206-231 with the WPP handling the reference
// lacks (SURVEY H16): every CTB row is its own substream located by its entry point, the engine is
// re-initialised there (9.3.2.5) and the contexts are synchronised from the row above after its
// second CTU (9.3.2.2 / 9.3.2.4).  `slot` of `n_slots` threads share the rows of one picture
// round-robin; Sync provides the wavefront:
//   bool wait(int row, int n_ctus)      block until `row` has finished n_ctus CTUs (false: tile aborted)
//   void publish(int row, int n_ctus)   announce progress of `row`
//   uint8_t* save_area(int row)         context snapshot of `row`, entries kSaveStride bytes apart
//   void abort(int code)                record the failure; every later wait() on this tile returns false
// Returns the number of CTUs decoded by this thread.
// ------------------------------------------------------------------------------------------------
template <int STRIDE, class Eng, class Sync>
HEIC_HD uint32_t parse_rows(Parser<STRIDE, Eng>& P, const uint32_t* substreams, int slot, int n_slots, Sync& sync) {
  const PicParams* pp = P.PP();
  const TileParams* tp = P.TP();
  const int wpp = pp->wpp, wctb = pp->wctb, hctb = pp->hctb;
  const int n_ctb = wctb * hctb;
  uint32_t ctus = 0;
  P.qp_y() = P.last_qp_y() = tp->slice_qp;
  P.qp_y_pred() = tp->slice_qp;
  P.qg_x() = P.qg_y() = -1;
  P.is_cu_qp_delta_coded() = 0;
  P.cu_qp_delta_val() = 0;
  P.first_qg_in_row() = 1;
  P.e.bins = 0;
  // Every thread walks all of its (row, CTU) steps even after a failure, so that the wavefront
  // hand-shakes stay matched and no dependent row can hang; a failed thread just stops parsing.
  for (int ry = slot; ry < hctb; ry += n_slots) {
    for (int rx = 0; rx < wctb; rx++) {
      if (wpp && ry > 0) {
        int need = rx == 0 ? (wctb < 2 ? wctb : 2) : rx + 1;
        if (!sync.wait(ry - 1, need)) P.fail(-100);  // another row of this tile failed and recorded its code
      }
      if (!P.err) {
        if (rx == 0 && (ry == 0 || wpp)) {
          uint32_t start = tp->data_off + (wpp ? substreams[ry] : 0u);
          uint32_t stop = (wpp && ry + 1 < (int)tp->n_sub) ? tp->data_off + substreams[ry + 1] : tp->bs_len;
          P.e.init(P.e.data, start, stop);
          if (P.e.offset_is_illegal()) P.fail(-3);  // arithmetic.rs:33-36
          if (ry == 0 || wctb == 1) {
            P.init_contexts(tp->slice_qp);
          } else {
            const uint8_t* src = sync.save_area(ry - 1);
            for (int i = 0; i < NUM_CTX; i++) P.st_ctx(i, src[i * Sync::kSaveStride]);
          }
          P.first_qg_in_row() = 1;
        }
        if (!P.err) P.coding_tree_unit(rx, ry);
        if (!P.err) {
          ctus++;
          if (wpp && rx == 1 && ry + 1 < hctb) {
            uint8_t* dst = sync.save_area(ry);
            for (int i = 0; i < NUM_CTX; i++) dst[i * Sync::kSaveStride] = (uint8_t)P.ld_ctx(i);
          }
          const int addr = ry * wctb + rx;
          P.e.expect_terminate(addr == n_ctb - 1);
          const int end_of_slice = P.e.terminate();  // end_of_slice_segment_flag (slice.rs:214)
          if (end_of_slice != (addr == n_ctb - 1)) {
            P.fail(-3);
          } else if (wpp && rx == wctb - 1 && !end_of_slice) {
            P.e.expect_terminate(1);
            if (!P.e.terminate()) P.fail(-3);  // end_of_subset_one_bit (slice.rs:222-227)
          }
        }
        if (P.err) sync.abort(P.err);
      }
      sync.publish(ry, rx + 1);
    }
  }
  return ctus;
}

}  // namespace dev
}  // namespace heic
