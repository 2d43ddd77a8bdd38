// Stage 3: intra prediction + reconstruction (H.265 8.4.4.2.1-6), absent from the reference
// (slice.rs:253-255 is todo!()).
//
// One CTA per picture (HEIF grid tile); warp r owns CTB rows r, r + R, ... and the rows advance as a
// wavefront (a CTU needs its above-right neighbour, so row r trails row r - 1 by two CTUs; progress
// counters live in shared memory).  With a large batch R = 1: one warp walks a whole picture and never
// waits, the parallelism comes from pictures alone.  Inside a CTU the transform units are inherently
// sequential (each predicts from its neighbours' reconstruction); the 32 lanes split the reference-sample
// gathering, substitution, smoothing and the pixels of the block.
// Per CTU the warp stages, with cp.async, the CTU's residuals (contiguous in the z-ordered coefficient arena)
// and tu_map words in shared memory, keeps the CTU under construction there with a one-sample apron (row above
// incl. the above-right CTU, column to the left), and writes it to HBM once, coalesced, when complete.
#include <cuda_runtime.h>

#include "kernels.h"

namespace heic {
namespace dev {

namespace {

struct Angles {
  int8_t angle[35];
  int16_t inv[15];  // modes 11..25
};
constexpr Angles kAngles = {{0,   0,   32,  26,  21,  17, 13, 9,  5,  2,  0,  -2, -5, -9, -13, -17, -21, -26,
                             -32, -26, -21, -17, -13, -9, -5, -2, 0,  2,  5,  9,  13, 17, 21,  26,  32},
                            {-4096, -1638, -910, -630, -482, -390, -315, -256, -315, -390, -482, -630, -910, -1638, -4096}};
__constant__ Angles kAng = kAngles;

// ---- 4x4 prediction as a table: for mode m and output sample p = (x, y) = (p & 3, p >> 2), word [m * 16 + p] holds
//   bits 0-4 / 8-12   the lanes A and B of the two reference samples the sample is weighed from (lane s holds scan
//                     position s: left(i) = lane 8 - i, top(i) = lane 8 + i), as shuffle source lanes;
//   bits 16-23 / 24-31 their weights wA and wB;
//   bits 5-7          DC: the weight of the DC value in the luma edge filter (8.4.4.2.5);
//   bit 13            modes 10 / 26: the sample lies on the luma edge the filter of 8.4.4.2.6 adjusts.
// Angular (8.4.4.2.6): A, B = ref[iIdx + 1], ref[iIdx + 2] (negative indices projected onto the other edge), wA = 32 - iFact,
// wB = iFact; for modes 10 and 26 (iFact = 0) B is the opposite edge's sample the edge filter needs.  Planar and DC: A =
// left(y + 1), B = top(x + 1); planar weights (3 - x, 3 - y), DC (x == 0, y == 0).  A lane's whole mode-dependent set-up is one
// load instead of a branch per mode class.
struct Pred4Table {
  uint32_t w[35 * 16];
};
constexpr Pred4Table make_pred4_table() {
  Pred4Table t{};
  for (int m = 0; m < 35; m++) {
    for (int p = 0; p < 16; p++) {
      const int x = p & 3, y = p >> 2;
      int la = 7 - y, lb = 9 + x, wa = 0, wb = 0, low = 0;  // planar / DC: left(y + 1), top(x + 1)
      if (m == 0) {
        wa = 3 - x, wb = 3 - y;
      } else if (m == 1) {
        wa = x == 0, wb = y == 0, low = (4 - wa - wb) << 5;
      } else {
        const int angle = kAngles.angle[m];
        const bool vertical = m >= 18;
        const int dir = vertical ? 1 : -1;
        const int tt = ((vertical ? y : x) + 1) * angle, fact = tt & 31;
        const int t1 = (vertical ? x : y) + (tt >> 5) + 1;
        la = 8 + dir * t1;
        lb = la + dir;
        if (angle < 0) {
          const int inv = kAngles.inv[m - 11];
          if (t1 < 0) la = 8 - dir * ((t1 * inv + 128) >> 8);
          if (t1 + 1 < 0) lb = 8 - dir * (((t1 + 1) * inv + 128) >> 8);
        }
        wa = 32 - fact, wb = fact;
        if (m == 26) lb = 7 - y, low = x == 0 ? 1 << 13 : 0;  // v = top(1) + ((left(y + 1) - corner) >> 1) at x = 0
        if (m == 10) lb = 9 + x, low = y == 0 ? 1 << 13 : 0;  // v = left(1) + ((top(x + 1) - corner) >> 1) at y = 0
      }
      t.w[m * 16 + p] = (uint32_t)(la & 31) | ((uint32_t)(lb & 31) << 8) | (uint32_t)low | ((uint32_t)wa << 16) | ((uint32_t)wb << 24);
    }
  }
  return t;
}
__device__ const Pred4Table kPred4 = make_pred4_table();

__device__ __forceinline__ uint32_t compact1(uint32_t v) {
  v &= 0x55u;
  v = (v | (v >> 1)) & 0x33u;
  v = (v | (v >> 2)) & 0x0fu;
  return v;
}
__device__ __forceinline__ int clip8(int v) { return min(255, max(0, v)); }

__device__ __forceinline__ void cp_async16s(uint32_t smem_addr, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_addr), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// A pointer into the kernel's dynamic shared memory kept as its 32-bit shared-window address.  Converting to a C++
// pointer at the point of use keeps the address space visible to the compiler (LDS/STS) while every address derives from
// ONE register-held base: as 64-bit generic pointers the nine of them were re-formed from the symbol's address
// (S2UR SR_CgaCtaId + ULEA, 49 places in the kernel) wherever the register allocator had dropped them.
template <class T>
struct SP {
  uint32_t a;
  __device__ __forceinline__ operator T*() const { return reinterpret_cast<T*>(__cvta_shared_to_generic(a)); }
  __device__ __forceinline__ T& operator[](int i) const { return reinterpret_cast<T*>(__cvta_shared_to_generic(a))[i]; }
  __device__ __forceinline__ SP operator+(int i) const { return SP{a + (uint32_t)(i * (int)sizeof(T))}; }
  __device__ __forceinline__ int operator-(SP o) const { return (int)(a - o.a) / (int)sizeof(T); }
};
struct Ctu {
  int w, h, ctb, ctb4, x_ctb, y_ctb;
  SP<uint8_t> buf[3];   // sample (x, y) relative to the CTU origin at buf[(y + 1) * stride + x + kApron], x, y >= -1
  int stride[3];
  SP<uint8_t> ref;      // reference samples after substitution, s = 0 .. 4n (bottom-left -> corner -> top-right);
                        // the second block of a chroma pair (or the smoothed luma samples) at ref + kRefSpan
  SP<uint8_t> refa;     // angular reference array, refa[-32 .. 64]; second block of a pair at refa + kRefaSpan
  SP<int16_t> res[3];   // residuals of this CTU, z-ordered as in the coefficient arena
  SP<uint32_t> tuw;     // tu_map words of this CTU
  int lane;
  int strong_flag;
};
constexpr int kRefSpan = 144, kRefaSpan = 104;
constexpr int kApron = 4;  // bytes in front of a CTU buffer row: sample x = -1 is its last one

__device__ __forceinline__ uint32_t pack4(int a, int b, int c, int d) {
  return (uint32_t)a | ((uint32_t)b << 8) | ((uint32_t)c << 16) | ((uint32_t)d << 24);
}

// ---- 8.4.4.2.2 reference availability (6.4.1) for a single-slice all-intra picture in z-scan order ---------
// The left column and the top row exist whenever the block is not on the picture border.  The below-left and
// above-right N samples belong to ONE aligned N x N block each, which is either completely reconstructed or not
// started (transform units are atomic in z-order), further cut by the picture limits to a prefix.  So the
// available samples form one interval [lo, hi] of the scan (bottom-left -> corner -> top-right, positions 0 .. 4N), and
// the substitution process ("nearest available sample before, else first one after") is a clamp of s to that interval.
// Reconstructed-yet is a comparison of z-order indices at granularity N inside the CTB: for the below-left
// neighbour (cx - 1, cy + 1) the highest differing coordinate bit is ctz(cx) in x (where it is smaller) and
// ctz(cy + 1) in y (where it is larger), and y wins ties; likewise for the above-right one.  OR-ing the CTB size
// in makes the left / upper CTB (always there) and the lower / right CTB (never there) fall out of the same test.
// Returns lo | hi << 8 (lo > hi: nothing available -> 1 << (bitDepth - 1)).  Pure arithmetic on the block's position, so
// the kernel evaluates it for all transform units of a CTU at once, one lane per unit.
__device__ __forceinline__ uint32_t block_availability(const Ctu& c, int sub, int bx, int by, int log2) {
  const int N = 1 << log2;
  const int units = (c.ctb >> sub) >> log2;  // blocks of this size per CTB side
  const int cx = bx >> log2, cy = by >> log2;
  const int X0 = (c.x_ctb >> sub) + bx, Y0 = (c.y_ctb >> sub) + by;
  const bool left_ok = X0 > 0, top_ok = Y0 > 0;
  int n_bl = 0, n_tr = 0;
  if (left_ok && __ffs(cx | units) > __ffs(cy + 1)) n_bl = min(N, max(0, (c.h >> sub) - (Y0 + N)));
  if (top_ok && __ffs(cy | units) >= __ffs(cx + 1)) n_tr = min(N, max(0, (c.w >> sub) - (X0 + N)));
  const int lo = left_ok ? N - n_bl : 2 * N + 1;
  const int hi = top_ok ? 3 * N + n_tr : 2 * N - 1;
  return (uint32_t)lo | ((uint32_t)hi << 8);
}

// Fields of a transform unit's per-plane word (luma, or the chroma pair), packed for 32 units at a time by the CTU walk:
// mode in bits 14-19, cbf (Cb's for a pair) in bit 29, Cr's cbf in bit 30, and
//   bit 31 set (4x4 block): bits 0-13 the CTU-buffer offset of the block's corner sample (-1, -1), bits 20-23 / 24-28 the
//                           available reference interval (lo, hi) of block_availability();
//   bit 31 clear (larger):  bits 0-3 / 4-7 the block position bx / 4, by / 4, bits 8-10 log2 of its size; (lo, hi) in a
//                           separate word.
constexpr uint32_t kW4 = 1u << 31, kWCbfA = 1u << 29, kWCbfB = 1u << 30;

// Predicts and reconstructs a 4x4 block of one plane, or — `pair` — the Cb and Cr blocks of a chroma pair (same geometry and
// mode; buffers `buf_delta` and residuals `res_delta` apart).  The 17 reference samples sit in lanes 0..16 (lane s holds scan
// position s; a pair's Cr sample in the upper halfword beside the Cb one, so one shuffle and one multiply serve both
// blocks), lane p < 16 predicts sample (p & 3, p >> 2) with what kPred4 says for it; no reference arrays, no smoothing at
// this size, one warp barrier.  The edge filters of DC / horizontal / vertical are luma only.
__device__ __forceinline__ void predict4(int lane, bool pair, uint8_t* buf, int buf_delta, int stride, uint32_t w, int mode,
                                         const int16_t* __restrict__ resid, int res_delta) {
  const uint8_t* corner = buf + (w & 0x3fffu);  // sample (-1, -1)
  const int lo = (w >> 20) & 15, hi = (w >> 24) & 31;
  const uint32_t tw = __ldg(&kPred4.w[mode * 16 + (lane & 15)]);
  uint32_t r;
  {
    const int d = min(max(lane, lo), hi) - 8;  // lanes above 16 fetch position hi again: in bounds, unused
    const int off = d <= 0 ? -d * stride : d;
    r = corner[off];
    if (pair) r |= (uint32_t)corner[off + buf_delta] << 16;
    if (lo > hi) r = pair ? 0x800080u : 0x80u;  // nothing available: 1 << (bitDepth - 1)
  }
  const uint32_t a = __shfl_sync(0xffffffffu, r, (int)tw), b = __shfl_sync(0xffffffffu, r, (int)(tw >> 8));
  uint32_t acc = ((tw >> 16) & 0xffu) * a + (tw >> 24) * b;  // per halfword: below 2^16
  int v0, v1;
  if (mode >= 2) {  // 8.4.4.2.6
    acc += 0x100010u;
    v0 = (int)((acc & 0xffffu) >> 5), v1 = (int)(acc >> 21);
    if (!pair && (mode == 10 || mode == 26)) {
      const int c0 = __shfl_sync(0xffffffffu, (int)r, 8);
      if (tw & (1u << 13)) v0 = clip8((int)a + (((int)b - c0) >> 1));
    }
  } else if (mode == 0) {  // 8.4.4.2.4
    const uint32_t tr = __shfl_sync(0xffffffffu, r, 13), bl = __shfl_sync(0xffffffffu, r, 3);
    acc += (uint32_t)((lane & 3) + 1) * tr + (uint32_t)(((lane >> 2) & 3) + 1) * bl + 0x40004u;
    v0 = (int)((acc & 0xffffu) >> 3), v1 = (int)(acc >> 19);
  } else {  // 8.4.4.2.5: both blocks of a pair summed in one reduction (each sum < 2^11)
    const uint32_t sums = __reduce_add_sync(0xffffffffu, ((0x1ef0u >> lane) & 1u) ? r : 0u);  // lanes 4..7, 9..12
    v0 = (int)(((sums & 0xffffu) + 4) >> 3), v1 = (int)(((sums >> 16) + 4) >> 3);
    if (!pair) v0 = (int)(acc + ((tw >> 5) & 7u) * (uint32_t)v0 + 2) >> 2;
  }
  if (lane < 16) {
    uint8_t* o = buf + (w & 0x3fffu) + 1 + ((lane >> 2) + 1) * stride + (lane & 3);
    if (w & kWCbfA) v0 = clip8(v0 + (int)resid[lane]);
    o[0] = (uint8_t)v0;
    if (pair) {
      if (w & kWCbfB) v1 = clip8(v1 + (int)resid[res_delta + lane]);
      o[buf_delta] = (uint8_t)v1;
    }
  }
  __syncwarp();
}

// Predicts and reconstructs the N x N block at (bx, by) (plane samples, CTU-relative, N >= 8) of one plane, or — `pair` —
// of the two chroma planes together (same geometry and mode; buffers `buf_delta` and residuals `res_delta` apart), which
// shares the availability logic and the loop overheads between Cb and Cr.  A lane produces four horizontally adjacent
// samples per step.  Deliberately one compact, size-generic body with a single call site: the kernel is
// instruction-fetch bound when this code is replicated per size and per component.
// (lo, hi): the interval of available reference positions, from block_availability().
__device__ __forceinline__ void predict_block(const Ctu& c, bool pair, uint8_t* buf, int buf_delta, int stride, int bx, int by,
                                              int log2, int mode, bool cbf_a, bool cbf_b, const int16_t* __restrict__ resid,
                                              int res_delta, int lo, int hi) {
  const int N = 1 << log2, lane = c.lane;
  const int total = 4 * N, cnt = total + 1;  // positions 0 .. 4N: s < 2N left column bottom-up, s = 2N corner, s > 2N top row
  uint8_t* ref = c.ref;
  {
    const uint8_t* corner = buf + by * stride + bx + kApron - 1;  // sample (-1, -1)
    const int n_ref = pair ? 2 * cnt : cnt;
    const int lo_d = lo - 2 * N, hi_d = hi - 2 * N;  // d <= 0: left column (upwards to the corner), d > 0: top row
    if (lo > hi) {
      for (int s = lane; s < 2 * kRefSpan; s += 32) ref[s] = 128;
    } else {
#pragma unroll 1
      for (int s = lane - 2 * N; s < n_ref - 2 * N; s += 32) {
        const bool second = s > 2 * N;
        const int ss = second ? s - cnt : s;                 // position relative to the corner
        const int d = min(max(ss, lo_d), hi_d);
        const uint8_t* src = corner + (d <= 0 ? -d * stride : d);
        if (second) src += buf_delta;
        ref[(second ? ss + kRefSpan : ss) + 2 * N] = *src;
      }
    }
  }
  __syncwarp();
  // ---- 8.4.4.2.3: smoothing (luma only in 4:2:0) ---------------------------------------------------
  const uint8_t* R = ref;
  if (N > 4 && !pair && mode != 1) {
    const int min_dist = min(abs(mode - 26), abs(mode - 10));
    const int thr = N == 8 ? 7 : (N == 16 ? 1 : 0);
    if (min_dist > thr) {
      const bool strong = N == 32 && c.strong_flag && abs((int)ref[64] + ref[128] - 2 * ref[96]) < 8 &&
                          abs((int)ref[64] + ref[0] - 2 * ref[32]) < 8;
      uint8_t* reff = ref + kRefSpan;
#pragma unroll 1
      for (int s = lane; s <= total; s += 32) {
        int v;
        if (s == 0 || s == total) v = ref[s];
        else if (strong) {
          if (s == 64) v = ref[64];
          else if (s < 64) v = (s * ref[64] + (64 - s) * ref[0] + 32) >> 6;
          else v = ((128 - s) * ref[64] + (s - 64) * ref[128] + 32) >> 6;
        } else {
          v = (ref[s - 1] + 2 * ref[s] + ref[s + 1] + 2) >> 2;
        }
        reff[s] = (uint8_t)v;
      }
      __syncwarp();
      R = reff;
    }
  }
  // left(i) = p[-1][i - 1] = R[2N - i], top(i) = p[i - 1][-1] = R[2N + i]; index 0 is the corner
  const int quads = (N * N) >> 2;                // steps of four samples per block
  const int n_items = pair ? 2 * quads : quads;
  const int lq = log2 - 2;                       // log2 of the quads per row
  const bool edge = !pair && N < 32;
  uint8_t* out = buf + (by + 1) * stride + bx + kApron;
  // mode-specific setup
  int dc_pack = 0;
  const int angle = kAng.angle[mode];
  const bool vertical = mode >= 18;
  if (mode == 1) {  // 8.4.4.2.5 DC: both blocks of a pair summed in one packed reduction (each sum < 2^16)
    if (lane < N) {
      dc_pack = (int)R[2 * N - 1 - lane] + R[2 * N + 1 + lane];
      if (pair) dc_pack += ((int)R[kRefSpan + 2 * N - 1 - lane] + R[kRefSpan + 2 * N + 1 + lane]) << 16;
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) dc_pack += __shfl_xor_sync(0xffffffffu, dc_pack, o);
  } else if (mode >= 2) {  // 8.4.4.2.6 angular: ra[i], i = -N .. 2N
    const int top_i = angle < 0 ? N : 2 * N;
    const int dir = vertical ? 1 : -1;
#pragma unroll 1
    for (int second = 0; second < (pair ? 2 : 1); second++) {
      const uint8_t* Rp = R + second * kRefSpan + 2 * N;
      uint8_t* ra = c.refa + second * kRefaSpan;
#pragma unroll 1
      for (int i = lane; i <= top_i; i += 32) ra[i] = Rp[dir * i];
      if (angle < 0) {
        const int last = (N * angle) >> 5;
        const int i = -1 - lane;  // |last| <= N <= 32: one step
        if (last < -1 && i >= last) ra[i] = Rp[-dir * ((i * (int)kAng.inv[mode - 11] + 128) >> 8)];
      }
    }
    __syncwarp();
  }
#pragma unroll 1
  for (int q = lane; q < n_items; q += 32) {
    const int second = q >= quads ? 1 : 0, qq = q - second * quads;
    const int y = qq >> lq, x0 = (qq & ((1 << lq) - 1)) << 2;
    const uint8_t* Rp = R + second * kRefSpan + 2 * N;  // Rp[-i] = left(i), Rp[i] = top(i)
    int v0, v1, v2, v3;
    if (mode == 0) {  // 8.4.4.2.4 planar
      const int L = Rp[-1 - y], tr = Rp[1 + N], bl = Rp[-1 - N];
      const int a = N - 1 - y, base = (N - 1 - x0) * L + (x0 + 1) * tr + (y + 1) * bl + N, step = tr - L, sh = log2 + 1;
      v0 = (base + a * Rp[1 + x0]) >> sh;
      v1 = (base + step + a * Rp[2 + x0]) >> sh;
      v2 = (base + 2 * step + a * Rp[3 + x0]) >> sh;
      v3 = (base + 3 * step + a * Rp[4 + x0]) >> sh;
    } else if (mode == 1) {
      const int dc = (((dc_pack >> (16 * second)) & 0xffff) + N) >> (log2 + 1);
      v0 = v1 = v2 = v3 = dc;
      if (edge) {
        if (y == 0) {
          v0 = (Rp[1 + x0] + 3 * dc + 2) >> 2;
          v1 = (Rp[2 + x0] + 3 * dc + 2) >> 2;
          v2 = (Rp[3 + x0] + 3 * dc + 2) >> 2;
          v3 = (Rp[4 + x0] + 3 * dc + 2) >> 2;
          if (x0 == 0) v0 = (Rp[-1] + 2 * dc + Rp[1] + 2) >> 2;
        } else if (x0 == 0) {
          v0 = (Rp[-1 - y] + 3 * dc + 2) >> 2;
        }
      }
    } else {
      const uint8_t* ra = c.refa + second * kRefaSpan;
      if (vertical) {
        const int t = (y + 1) * angle, fact = t & 31;
        const uint8_t* r5 = ra + x0 + (t >> 5) + 1;
        const int a0 = r5[0], a1 = r5[1], a2 = r5[2], a3 = r5[3], a4 = r5[4];  // a4 unused when fact == 0 (inside refa)
        v0 = ((32 - fact) * a0 + fact * a1 + 16) >> 5;
        v1 = ((32 - fact) * a1 + fact * a2 + 16) >> 5;
        v2 = ((32 - fact) * a2 + fact * a3 + 16) >> 5;
        v3 = ((32 - fact) * a3 + fact * a4 + 16) >> 5;
        if (edge && mode == 26 && x0 == 0) v0 = clip8(Rp[1] + ((Rp[-1 - y] - Rp[0]) >> 1));
      } else {
        const uint8_t* ry = ra + y + 1;
        int t = (x0 + 1) * angle;
        v0 = ((32 - (t & 31)) * ry[t >> 5] + (t & 31) * ry[(t >> 5) + 1] + 16) >> 5;
        t += angle;
        v1 = ((32 - (t & 31)) * ry[t >> 5] + (t & 31) * ry[(t >> 5) + 1] + 16) >> 5;
        t += angle;
        v2 = ((32 - (t & 31)) * ry[t >> 5] + (t & 31) * ry[(t >> 5) + 1] + 16) >> 5;
        t += angle;
        v3 = ((32 - (t & 31)) * ry[t >> 5] + (t & 31) * ry[(t >> 5) + 1] + 16) >> 5;
        if (edge && mode == 10 && y == 0) {
          const int l1 = Rp[-1], c0 = Rp[0];
          v0 = clip8(l1 + ((Rp[1 + x0] - c0) >> 1));
          v1 = clip8(l1 + ((Rp[2 + x0] - c0) >> 1));
          v2 = clip8(l1 + ((Rp[3 + x0] - c0) >> 1));
          v3 = clip8(l1 + ((Rp[4 + x0] - c0) >> 1));
        }
      }
    }
    if (second ? cbf_b : cbf_a) {
      const uint2 r = *reinterpret_cast<const uint2*>(resid + second * res_delta + (qq << 2));
      v0 = clip8(v0 + (int)(int16_t)(r.x & 0xffffu));
      v1 = clip8(v1 + ((int)r.x >> 16));
      v2 = clip8(v2 + (int)(int16_t)(r.y & 0xffffu));
      v3 = clip8(v3 + ((int)r.y >> 16));
    }
    *reinterpret_cast<uint32_t*>(out + second * buf_delta + y * stride + x0) = pack4(v0, v1, v2, v3);
  }
  __syncwarp();
}

// Byte offsets of a warp's scratch areas (sized for the batch's largest CTB), computed on the host: as kernel
// parameters they cost one add from the constant bank wherever a pointer is needed again.
struct IntraLayout {
  int res1, res2, tuw, ref, refa, buf0, buf1, buf2;
  int stride_y, stride_c;  // row strides of the CTU buffers
  int warp_bytes;
};

// 72 registers: 28 one-warp CTAs per SM instead of 24 at 80, no spills (52.7 -> 50.7 ms per 592 images; 64 registers /
// 32 warps measured slower, 53.6 ms, and so did 96 registers / 21 warps, 54.9 ms)
#ifndef HEIC_INTRA_MAXNREG
#define HEIC_INTRA_MAXNREG 72
#endif
__global__ void __maxnreg__(HEIC_INTRA_MAXNREG) intra_kernel(Arenas A, const uint32_t* __restrict__ order, int n_slots, IntraLayout L, int clear_coeff) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const uint32_t tile = order[blockIdx.x];
  const TileParams* tp = A.tiles + tile;
  const PicParams* pp = A.pics + tp->pic;
  if (A.status[tile].code != 0) {
    // a tile that failed to parse is not reconstructed, but its coefficient slots still go back to all-zero (below)
    if (clear_coeff) {
      uint4* z = reinterpret_cast<uint4*>(A.coeff + tp->coeff_off[0]);
      const size_t n16 = (size_t)pp->n_tu * 24 * 2 / 16;
      for (size_t i = threadIdx.x; i < n16; i += blockDim.x) z[i] = make_uint4(0u, 0u, 0u, 0u);
    }
    return;
  }
  const int wctb = pp->wctb, hctb = pp->hctb;
  volatile int* progress = reinterpret_cast<volatile int*>(smem_raw);
  const int progress_bytes = n_slots > 1 ? ((hctb * 4 + 15) & ~15) : 0;
  if (n_slots > 1) {
    for (int i = threadIdx.x; i < hctb; i += blockDim.x) progress[i] = 0;
    __syncthreads();
  }
  const int slot = threadIdx.x >> 5, lane = threadIdx.x & 31;

  Ctu c;
  c.w = pp->w;
  c.h = pp->h;
  c.ctb = 1 << pp->log2_ctb;
  c.ctb4 = c.ctb >> 2;
  c.lane = lane;
  c.strong_flag = pp->strong_intra_smoothing;
  const int n_planes = pp->chroma ? 3 : 1;
  const int n4sq = c.ctb4 * c.ctb4;
  {
    uint32_t wbase = (uint32_t)progress_bytes + (uint32_t)slot * (uint32_t)L.warp_bytes;
    asm volatile("" : "+r"(wbase));  // opaque: keeps the warp's base offset in a register instead of re-deriving it per use
    uint32_t p = (uint32_t)__cvta_generic_to_shared(smem_raw) + wbase;
    asm volatile("" : "+r"(p));  // the one register every shared-memory address of this warp derives from
    c.res[0].a = p;
    c.res[1].a = p + (uint32_t)L.res1;
    c.res[2].a = p + (uint32_t)L.res2;
    c.tuw.a = p + (uint32_t)L.tuw;
    c.ref.a = p + (uint32_t)L.ref;
    c.refa.a = p + (uint32_t)L.refa + 32u;
    c.buf[0].a = p + (uint32_t)L.buf0;
    c.buf[1].a = p + (uint32_t)L.buf1;
    c.buf[2].a = p + (uint32_t)L.buf2;
    c.stride[0] = L.stride_y;
    c.stride[1] = c.stride[2] = L.stride_c;
  }
  const uint32_t* tu_map = A.tu_map + tp->tu_off;
  uint8_t* plane[3] = {A.recon + tp->plane_off[0], A.recon + tp->plane_off[1], A.recon + tp->plane_off[2]};
  const int pitch[3] = {pp->pitch_y, pp->pitch_c, pp->pitch_c};

  for (int ry = slot; ry < hctb; ry += n_slots) {
    for (int rx = 0; rx < wctb; rx++) {
      const uint32_t ctb_addr = (uint32_t)(ry * wctb + rx);
      // ---- stage this CTU's residuals and tu_map words (contiguous in HBM) ------------------------------
      {
        const char* g0 = reinterpret_cast<const char*>(A.coeff + tp->coeff_off[0] + (size_t)ctb_addr * n4sq * 16);
        for (int i = lane * 16; i < n4sq * 32; i += 512) cp_async16s(c.res[0].a + i, g0 + i);
        if (n_planes == 3) {
          const char* g1 = reinterpret_cast<const char*>(A.coeff + tp->coeff_off[1] + (size_t)ctb_addr * n4sq * 4);
          const char* g2 = reinterpret_cast<const char*>(A.coeff + tp->coeff_off[2] + (size_t)ctb_addr * n4sq * 4);
          for (int i = lane * 16; i < n4sq * 8; i += 512) {
            cp_async16s(c.res[1].a + i, g1 + i);
            cp_async16s(c.res[2].a + i, g2 + i);
          }
        }
        const char* gt = reinterpret_cast<const char*>(tu_map + (size_t)ctb_addr * n4sq);
        for (int i = lane * 16; i < n4sq * 4; i += 512) cp_async16s(c.tuw.a + i, gt + i);
      }
      if (n_slots > 1 && ry > 0) {
        const int need = min(rx + 2, wctb);
        if (lane == 0) {
          unsigned ns = 32;
          while (progress[ry - 1] < need) {
            __nanosleep(ns);
            if (ns < 1024) ns *= 2;
          }
        }
        __syncwarp();
        __threadfence_block();
      }
      c.x_ctb = rx * c.ctb;
      c.y_ctb = ry * c.ctb;
      // ---- apron: left column from the CTU just finished (still in shared memory), top row from HBM ----
#pragma unroll
      for (int pl = 0; pl < 3; pl++) {
        if (pl >= n_planes) break;
        const int sub = pl ? 1 : 0, cs = c.ctb >> sub, st = c.stride[pl];
        uint8_t* b = c.buf[pl];
        if (rx > 0)
          for (int y = lane; y < cs; y += 32) b[(y + 1) * st + kApron - 1] = b[(y + 1) * st + kApron + cs - 1];
        if (ry > 0) {
          const int wp = c.w >> sub, x0 = (c.x_ctb >> sub) - 1, y0 = (c.y_ctb >> sub) - 1;
          // aligned 4-byte words from x_ctb - 4 (its last byte is the corner sample) to the end of the above-right CTU;
          // plane widths are multiples of 4, so a word is inside the picture or outside it as a whole
          const uint8_t* src = plane[pl] + (size_t)y0 * pitch[pl];
          for (int j = lane; j <= cs / 2; j += 32) {
            const int x = x0 - 3 + 4 * j;
            if (x >= 0 && x < wp) *reinterpret_cast<uint32_t*>(b + kApron - 4 + 4 * j) = __ldcg(reinterpret_cast<const uint32_t*>(src + x));
          }
        }
      }
      cp_async_wait_all();
      __syncwarp();
      if (clear_coeff) {
        // The residuals now live in shared memory: hand the CTU's coefficient slots back all-zero, which is what the
        // next decode's CABAC stage needs (it only writes significant coefficients).  Coalesced fire-and-forget
        // stores here replace a full-arena memset before every decode.
        const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
        char* g0 = reinterpret_cast<char*>(A.coeff + tp->coeff_off[0] + (size_t)ctb_addr * n4sq * 16);
        for (int i = lane * 16; i < n4sq * 32; i += 512) *reinterpret_cast<uint4*>(g0 + i) = zero;
        if (n_planes == 3) {
          char* g1 = reinterpret_cast<char*>(A.coeff + tp->coeff_off[1] + (size_t)ctb_addr * n4sq * 4);
          char* g2 = reinterpret_cast<char*>(A.coeff + tp->coeff_off[2] + (size_t)ctb_addr * n4sq * 4);
          for (int i = lane * 16; i < n4sq * 8; i += 512) {
            *reinterpret_cast<uint4*>(g1 + i) = zero;
            *reinterpret_cast<uint4*>(g2 + i) = zero;
          }
        }
      }
      // ---- transform units of this CTB in z-order -----------------------------------------------------
      // Everything about a transform unit that is arithmetic on its tu_map word and position (block positions, modes, cbfs,
      // the availability intervals of its luma block and of its chroma pair) is worked out for 32 units at a time, one lane
      // per 4x4 unit, into the per-plane words described at kW4; the sequential walk below then fetches two words per unit
      // with shuffles (a third one for a block larger than 4x4).
      {
        const int buf_delta = (int)(c.buf[2] - c.buf[1]), res_delta = (int)(c.res[2] - c.res[1]);
#pragma unroll 1
        for (int base = 0; base < n4sq; base += 32) {
          const int idx_l = base + lane;
          const uint32_t wl = idx_l < n4sq ? c.tuw[idx_l] : 0u;
          uint32_t pa = 0, pb = 0, pc = 0;  // luma word, availability of the larger blocks (luma | chroma << 16), chroma word
          if (wl & TU_ORIGIN) {
            const int lg = (int)tu_log2(wl);
            const int bxl = (int)compact1((uint32_t)idx_l) << 2, byl = (int)compact1((uint32_t)idx_l >> 1) << 2;
            const uint32_t avl = block_availability(c, 0, bxl, byl, lg);
            pa = (tu_luma_mode(wl) << 14) | ((wl & TU_CBF_Y) ? kWCbfA : 0u);
            if (lg == 2) pa |= kW4 | ((avl & 15u) | (avl >> 4)) << 20 | (uint32_t)(byl * c.stride[0] + bxl + kApron - 1);
            else pa |= (uint32_t)(bxl >> 2) | ((uint32_t)(byl >> 2) << 4) | ((uint32_t)lg << 8), pb = avl;
            if ((wl & TU_HAS_CHROMA) && n_planes == 3) {
              const int lgc = lg > 2 ? lg - 1 : 2;
              const int bxc = (lg > 2 ? bxl : bxl - 4) >> 1, byc = (lg > 2 ? byl : byl - 4) >> 1;
              const uint32_t avc = block_availability(c, 1, bxc, byc, lgc);
              pc = (tu_chroma_mode(wl) << 14) | ((wl & TU_CBF_CB) ? kWCbfA : 0u) | ((wl & TU_CBF_CR) ? kWCbfB : 0u);
              if (lgc == 2) pc |= kW4 | ((avc & 15u) | (avc >> 4)) << 20 | (uint32_t)(byc * c.stride[1] + bxc + kApron - 1);
              else pc |= (uint32_t)(bxc >> 2) | ((uint32_t)(byc >> 2) << 4) | ((uint32_t)lgc << 8), pb |= avc << 16;
            }
          }
          uint32_t todo = __ballot_sync(0xffffffffu, (wl & TU_ORIGIN) != 0);
          while (todo) {  // warp-uniform
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const uint32_t wc = __shfl_sync(0xffffffffu, pc, src);  // non-zero iff the unit carries the chroma pair
            uint32_t w = __shfl_sync(0xffffffffu, pa, src);
            const int idx = base + src;
            // luma, then (when this unit carries them) Cb and Cr as a pair: ONE call site per body keeps the kernel small
#pragma unroll 1
            for (int k = 0;; k++) {
              const bool pr = k != 0;
              uint8_t* buf = pr ? c.buf[1] : c.buf[0];
              const int stride = pr ? c.stride[1] : c.stride[0];
              const int16_t* resid = pr ? c.res[1] + (idx >> 2) * 16 : c.res[0] + idx * 16;
              const int mode = (int)((w >> 14) & 63u);
              if (w & kW4) {
                predict4(lane, pr, buf, buf_delta, stride, w, mode, resid, res_delta);
              } else {
                const uint32_t av = __shfl_sync(0xffffffffu, pb, src) >> (pr ? 16 : 0);  // lo | hi << 8
                predict_block(c, pr, buf, buf_delta, stride, (int)(w & 15u) << 2, (int)((w >> 4) & 15u) << 2, (int)((w >> 8) & 7u),
                              mode, (w & kWCbfA) != 0, (w & kWCbfB) != 0, resid, res_delta, (int)(av & 0xffu), (int)((av >> 8) & 0xffu));
              }
              if (pr || !wc) break;
              w = wc;
            }
          }
        }
      }
      // ---- CTU -> HBM, 4 bytes per lane, rows of the CTU contiguous across lanes -------------------------
#pragma unroll
      for (int pl = 0; pl < 3; pl++) {
        if (pl >= n_planes) break;
        const int sub = pl ? 1 : 0, cs = c.ctb >> sub, st = c.stride[pl];
        const int xo = c.x_ctb >> sub, yo = c.y_ctb >> sub;
        const int wv = min(cs, (c.w >> sub) - xo), hv = min(cs, (c.h >> sub) - yo);
        const int lw = pp->log2_ctb - sub - 2;  // log2 of 4-byte words per CTU row
        const uint8_t* b = c.buf[pl];
        for (int i = lane; i < (hv << lw); i += 32) {
          const int y = i >> lw, xw = (i & ((1 << lw) - 1)) << 2;
          if (xw < wv)
            *reinterpret_cast<uint32_t*>(plane[pl] + (size_t)(yo + y) * pitch[pl] + xo + xw) =
                *reinterpret_cast<const uint32_t*>(b + (y + 1) * st + kApron + xw);
        }
      }
      if (n_slots > 1) {
        __threadfence_block();
        __syncwarp();
        if (lane == 0) progress[ry] = rx + 1;
      } else {
        __syncwarp();
      }
    }
  }
}

IntraLayout intra_layout(int log2_ctb) {
  const int ctb = 1 << log2_ctb, n4 = (ctb >> 2) * (ctb >> 2);
  IntraLayout L;
  int o = n4 * 16 * 2;  // luma residuals first
  L.res1 = o;
  o += n4 * 4 * 2;
  L.res2 = o;
  o += n4 * 4 * 2;
  L.tuw = o;
  o += n4 * 4;
  L.ref = o;
  o += 2 * kRefSpan;
  L.refa = o;
  o += 2 * kRefaSpan;
  // a 4-byte apron on the left (the corner / left-column samples; 4-byte aligned word stores), the CTU and the above-right
  // CTU: 17 and 9 words per row for 32x32 CTBs -- odd, so a column walks all banks -- and 7.3 KB per warp, so that 28 one-warp
  // CTAs fit an SM (24 with the 16-byte apron and 4 bytes of slack this layout had before)
  L.stride_y = 2 * ctb + kApron;
  L.stride_c = ctb + kApron;
  L.buf0 = o;
  o += (ctb + 1) * L.stride_y;
  L.buf1 = o;
  o += (ctb / 2 + 1) * L.stride_c;
  L.buf2 = o;
  o += (ctb / 2 + 1) * L.stride_c;
  L.warp_bytes = (o + 15) & ~15;
  return L;
}

}  // namespace

cudaError_t launch_intra(const Arenas& A, const uint32_t* order, int max_log2_ctb, int max_hctb, int n_slots, bool clear_coeff,
                         cudaStream_t stream) {
  if (!A.n_tiles) return cudaSuccess;
  const IntraLayout L = intra_layout(max_log2_ctb);
  const size_t smem = (n_slots > 1 ? (((size_t)max_hctb * 4 + 15) & ~(size_t)15) : 0) + (size_t)n_slots * L.warp_bytes;
  // the opt-in is per device (and this library serves several devices per process): set it on every launch, it is cheap
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(intra_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  intra_kernel<<<A.n_tiles, 32 * n_slots, smem, stream>>>(A, order, n_slots, L, clear_coeff ? 1 : 0);
  return cudaGetLastError();
}

}  // namespace dev
}  // namespace heic
