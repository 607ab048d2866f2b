// ht_detect.cuh — sm_100a kernels for ccv.grayscale + ccv.detect_objects
// (/root/reference/src/ccv.js:22-32, 109-333).  No tensor cores: byte compares + ordered fp64 adds.
// The whole library is compiled with -fmad=false so that every a*b+c below is two IEEE roundings,
// as in JavaScript.
//
// Everything between the caller's RGBA frames and the raw detection list works on FRAME QUADS: the pyramid arena
// holds one 32-bit word per pixel = that pixel in four consecutive frames (ht_common.cuh).
#pragma once
#include "ht_common.cuh"

namespace ht {

// Which of the 4 frames of a quad take part in a launch: the first n_frames - 4*quad of them (batch calls), or the
// per-quad mask the stream scheduler built (ht_stream_step: only the streams that are in detection mode).
__host__ __device__ __forceinline__ unsigned quad_frames(int quad, int n_frames, const uint8_t *__restrict__ quad_mask) {
  const int left = n_frames - 4 * quad;
  const unsigned prefix = left >= 4 ? 15u : (left > 0 ? (1u << left) - 1u : 0u);
  return quad_mask ? (prefix & quad_mask[quad]) : prefix;
}

__host__ __device__ __forceinline__ uint32_t rgb_bin(uint32_t px) {  // src/camshift.js:63-66, 345-348
  return ((px & 0xf0u) << 4) | ((px >> 8) & 0xf0u) | ((px >> 20) & 0xfu);
}

// ------------------------------------------------------------------------------------------------
// K1  grayscale — src/ccv.js:28-29:  gray = ToUint8Clamp(r*0.3 + g*0.59 + b*0.11)  (fp64, left to right, RN-even)
//
// No integer formula reproduces this: with q = 30r + 59g + 11b the exact value is q/100, and for the 167,836 of the
// 2^24 triples with q % 100 == 50 the fp64 sum lands on either side of k + 0.5 (226 of the 253 tie values of q go
// BOTH ways depending on (r,g,b): tests/test_gray_formula.py), so the three products and two sums are kept in fp64.
// What round 1 paid for were the int<->fp64 CONVERSIONS (I2F.F64 / F2I.F64 run at a quarter of the fp64 rate): here
// a byte becomes a double by planting it in the mantissa of 2^52 and subtracting 2^52 (exact), and the round-half-
// even store is `v + 2^52` read back from the low mantissa bits (exact for 0 <= v < 2^31; proven equal to
// rint() for every triple in the same test).  9 fp64 pipe operations per pixel, no conversions.
__host__ __device__ __forceinline__ uint32_t gray_of(uint32_t px) {
#ifdef __CUDA_ARCH__
  const double M = 4503599627370496.0;   // 2^52
  // one PRMT per channel: the byte, zero-extended, is the low mantissa word of 2^52 + byte
  const double r = __dsub_rn(__hiloint2double(0x43300000, (int)__byte_perm(px, 0u, 0x4440)), M);
  const double g = __dsub_rn(__hiloint2double(0x43300000, (int)__byte_perm(px, 0u, 0x4441)), M);
  const double b = __dsub_rn(__hiloint2double(0x43300000, (int)__byte_perm(px, 0u, 0x4442)), M);
  const double v = __dadd_rn(__dadd_rn(__dmul_rn(r, 0.3), __dmul_rn(g, 0.59)), __dmul_rn(b, 0.11));
  const uint32_t iv = (uint32_t)__double2loint(__dadd_rn(v, M));   // round half to even == Uint8ClampedArray store
  return min(iv, 255u);
#else   // host emulation: the same operations through a union (no FMA contraction: the file is built with -fmad=false
        // and the host compiler is not given an FMA target)
  union { double d; unsigned long long u; } c;
  const double M = 4503599627370496.0;
  volatile double r, g, b, t0, t1, t2, v;
  c.u = 0x4330000000000000ull | (px & 0xffu); r = c.d - M;
  c.u = 0x4330000000000000ull | ((px >> 8) & 0xffu); g = c.d - M;
  c.u = 0x4330000000000000ull | ((px >> 16) & 0xffu); b = c.d - M;
  t0 = r * 0.3; t1 = g * 0.59; t2 = b * 0.11;
  v = t0 + t1; v = v + t2;
  c.d = v + M;
  const uint32_t iv = (uint32_t)(c.u & 0xffffffffull);
  return iv < 255u ? iv : 255u;
#endif
}

// ld.global.nc on the device, a plain load in the host emulation (tests/test_pyramid_host.py)
template <class T>
__host__ __device__ __forceinline__ T ld_ro(const T *p) {
#ifdef __CUDA_ARCH__
  return __ldg(p);
#else
  return *p;
#endif
}

// One thread = 4 horizontally adjacent pixels of the 4 frames of a quad: four 16 B loads (one per frame), sixteen
// gray values, one 16 B store of 4 interleaved words into plane 0.  HIST additionally builds what camshift needs
// from the same read of the frame (src/camshift.js:49-72 via :268): the 4096-bin RGB histogram of each frame
// (shared-memory atomics, flushed per CTA) and the u16 plane of weight-table offsets (8 * bin) that k_track reads.
// grid = (chunks, quads).  HBM-bound: 4 B read + 1 B (+ 2 B) written per pixel.
// gray_item is one loop iteration of a thread (also run on the host by the emulation test, HIST = false).
template <bool VEC, bool HIST>
__host__ __device__ __forceinline__ void gray_item(const uint8_t *__restrict__ rgba, size_t frame_bytes, int quad, unsigned fmask,
                                                   uint32_t *__restrict__ dst_plane, int w, int pitch0, int gpr, int it,
                                                   uint32_t *sh_hist, uint16_t *__restrict__ bins, int n_px) {
  const int row = it / gpr, col = (it - row * gpr) * 4;
  uint32_t px[4][4];
#pragma unroll
  for (int f = 0; f < 4; ++f) {
    px[f][0] = px[f][1] = px[f][2] = px[f][3] = 0;
    if (((fmask >> f) & 1u) && col < w) {
      const uint8_t *src = rgba + (size_t)(4 * quad + f) * frame_bytes + ((size_t)row * w + col) * 4;
      if (VEC) {  // w % 4 == 0 and 16 B aligned frames
        const uint4 v = ld_ro(reinterpret_cast<const uint4 *>(src));
        px[f][0] = v.x; px[f][1] = v.y; px[f][2] = v.z; px[f][3] = v.w;
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (col + i < w) px[f][i] = ld_ro(reinterpret_cast<const uint32_t *>(src) + i);
      }
    }
  }
  // VEC implies w % 4 == 0: a group is entirely inside the frame or entirely in the pad columns - no per-pixel tests
  const bool grp_in = col < w;
  uint32_t out[4];
  if (VEC && grp_in && fmask == 15u) {   // the common case, branch-free: a full quad, a group inside the frame
#pragma unroll
    for (int i = 0; i < 4; ++i)
      out[i] = gray_of(px[0][i]) | (gray_of(px[1][i]) << 8) | (gray_of(px[2][i]) << 16) | (gray_of(px[3][i]) << 24);
  } else
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    out[i] = 0;
    if (VEC ? grp_in : (col + i < w)) {            // pad columns and missing frames are written as 0
#pragma unroll
      for (int f = 0; f < 4; ++f)
        if ((fmask >> f) & 1u) out[i] |= gray_of(px[f][i]) << (8 * f);
    }
  }
  *reinterpret_cast<uint4 *>(dst_plane + (size_t)row * pitch0 + col) = make_uint4(out[0], out[1], out[2], out[3]);
#ifdef __CUDA_ARCH__
  if (HIST) {
#pragma unroll
    for (int f = 0; f < 4; ++f) {
      if (!((fmask >> f) & 1u) || col >= w) continue;
      uint32_t b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        b[i] = rgb_bin(px[f][i]);
        // two frames share a word (16-bit counters: a CTA sees < 65,536 pixels of a frame, enforced by the host)
        if (VEC || col + i < w) atomicAdd(&sh_hist[(f >> 1) * 4096 + b[i]], (f & 1) ? 0x10000u : 1u);   // (col < w was tested above)
      }
      if (bins) {
        uint16_t *bo = bins + (size_t)(4 * quad + f) * n_px + (size_t)row * w + col;
        if (VEC) {
          *reinterpret_cast<uint2 *>(bo) = make_uint2((b[0] << 3) | (b[1] << 19), (b[2] << 3) | (b[3] << 19));
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (col + i < w) bo[i] = (uint16_t)(b[i] << 3);
        }
      }
    }
  }
#endif
}

template <bool VEC, bool HIST>
__global__ void __launch_bounds__(256, 4) k_gray(const uint8_t *__restrict__ rgba, size_t frame_bytes, int n_frames,
                                              uint32_t *__restrict__ arena, size_t quad_stride, int w, int h,
                                              int pitch0, uint32_t *__restrict__ hist, uint16_t *__restrict__ bins,
                                              int chunks, const uint8_t *__restrict__ quad_mask) {
  extern __shared__ uint32_t sh_hist[];   // HIST: [2][4096] words of two 16-bit counters (frames 0|1 and 2|3)
  const int quad = blockIdx.y;
  const unsigned fmask = quad_frames(quad, n_frames, quad_mask);
  if (fmask == 0u) return;
  if (HIST) {
    for (int i = threadIdx.x; i < 2 * 4096; i += 256) sh_hist[i] = 0;
    __syncthreads();
  }
  const int gpr = pitch0 >> 2;                        // groups of 4 pixels per plane row (pad columns included)
  const int n_groups = gpr * h;
  const int per = (n_groups + chunks - 1) / chunks;
  const int beg = blockIdx.x * per, end = min(n_groups, beg + per);
  uint32_t *dst_plane = arena + (size_t)quad * quad_stride;
  for (int it = beg + threadIdx.x; it < end; it += 256)
    gray_item<VEC, HIST>(rgba, frame_bytes, quad, fmask, dst_plane, w, pitch0, gpr, it, sh_hist, bins, w * h);
  if (HIST) {
    __syncthreads();
    for (int f = 0; f < 4; ++f) {
      if (!((fmask >> f) & 1u)) continue;
      uint32_t *out = hist + (size_t)(4 * quad + f) * 4096;
      for (int i = threadIdx.x; i < 4096; i += 256) {
        const uint32_t cnt = (sh_hist[(f >> 1) * 4096 + i] >> (16 * (f & 1))) & 0xffffu;
        if (chunks == 1) out[i] = cnt;
        else if (cnt) atomicAdd(&out[i], cnt);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K0  frame ingest — src/main.js:170: canvasContext.drawImage(videoElement, 0, 0, canvas.width, canvas.height): the
// video frame scaled onto the working canvas, all four channels.  Same DEFINED resampler as the pyramid (exact
// integer bilinear at pixel centres, taps clamped, round half up; oracle/ht_oracle.h), taps computed on the fly.
// One thread per destination pixel: four 4-byte loads, one 4-byte store.  (The 1:1 canvas copy facetrackr makes
// before detection, src/facetrackr.js:140-145, needs no kernel here: nothing on this path modifies its input.)
struct IngestGeom {
  int sw, sh, dw, dh;
  uint32_t magic, shift, half;   // floor(n / (4 dw dh)) == (uint64(n) * magic) >> shift for n <= 255.5 * 4 dw dh
};
// one destination pixel (also run on the host by tests/test_ingest_host.py)
__host__ __device__ __forceinline__ void ingest_pixel(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, const IngestGeom &g,
                                                      int X, int Y, int frame) {
  const uint32_t *s = reinterpret_cast<const uint32_t *>(src) + (size_t)frame * g.sw * g.sh;
  // u = (X + 1/2) sw / dw - 1/2 = ((2X + 1) sw - dw) / (2 dw): floor and numerator of the fraction, exactly
  const int un = (2 * X + 1) * g.sw - g.dw, vn = (2 * Y + 1) * g.sh - g.dh;
  const int Dx = 2 * g.dw, Dy = 2 * g.dh;
  int x0 = un / Dx, y0 = vn / Dy;
  if (un < 0 && x0 * Dx != un) --x0;       // floor for negative numerators (the first column / row when upscaling)
  if (vn < 0 && y0 * Dy != vn) --y0;
  const uint32_t fx = (uint32_t)(un - x0 * Dx), fy = (uint32_t)(vn - y0 * Dy);
  const int xa = x0 < 0 ? 0 : (x0 > g.sw - 1 ? g.sw - 1 : x0), xb = x0 + 1 < 0 ? 0 : (x0 + 1 > g.sw - 1 ? g.sw - 1 : x0 + 1);
  const int ya = y0 < 0 ? 0 : (y0 > g.sh - 1 ? g.sh - 1 : y0), yb = y0 + 1 < 0 ? 0 : (y0 + 1 > g.sh - 1 ? g.sh - 1 : y0 + 1);
  const uint32_t p00 = ld_ro(s + (size_t)ya * g.sw + xa), p01 = ld_ro(s + (size_t)ya * g.sw + xb);
  const uint32_t p10 = ld_ro(s + (size_t)yb * g.sw + xa), p11 = ld_ro(s + (size_t)yb * g.sw + xb);
  const uint32_t w00 = ((uint32_t)Dx - fx) * ((uint32_t)Dy - fy), w01 = fx * ((uint32_t)Dy - fy);
  const uint32_t w10 = ((uint32_t)Dx - fx) * fy, w11 = fx * fy;
  uint32_t out = 0;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const uint32_t num = w00 * ((p00 >> (8 * c)) & 0xffu) + w01 * ((p01 >> (8 * c)) & 0xffu) +
                         w10 * ((p10 >> (8 * c)) & 0xffu) + w11 * ((p11 >> (8 * c)) & 0xffu) + g.half;
    out |= (uint32_t)(((uint64_t)num * g.magic) >> g.shift) << (8 * c);
  }
  reinterpret_cast<uint32_t *>(dst)[((size_t)frame * g.dh + Y) * g.dw + X] = out;
}
__global__ void __launch_bounds__(256) k_ingest(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, IngestGeom g) {
  const int X = blockIdx.x * 64 + (threadIdx.x & 63), Y = blockIdx.y * 4 + (threadIdx.x >> 6);
  if (X >= g.dw || Y >= g.dh) return;
  ingest_pixel(src, dst, g, X, Y, (int)blockIdx.z);
}

// ------------------------------------------------------------------------------------------------
// K2  pyramid level = canvas-shim drawImage (exact integer bilinear, see oracle/ht_oracle.h and
// src/ccv.js:121,128,135,140,145).  One launch per pyramid "generation" (levels whose sources are
// complete).  Block = 32 x 32 pixels of one destination plane of one frame quad; thread = one column x 4 rows.
// Every load and store is a whole word (4 frames): the tap positions, weights and addresses - most of round 1's
// 43 instructions per output pixel - are computed once for four frames.
// byte f (= frame f of the quad) of a pyramid word, zero-extended
__host__ __device__ __forceinline__ uint32_t quad_byte(uint32_t w, int f) {
#ifdef __CUDA_ARCH__
  return __byte_perm(w, 0u, 0x4440u + (unsigned)f);
#else
  return (w >> (8 * f)) & 0xffu;
#endif
}
__host__ __device__ __forceinline__ void resample_thread(const DevPlan &plan, int tile0, uint32_t *__restrict__ arena,
                                                         size_t quad_stride, int bx, int by, int tid) {
  // per-block metadata: one 8 B tile record and one 64 B job record, fetched with vector loads
  const uint2 tl = ld_ro(reinterpret_cast<const uint2 *>(plan.pyr_tiles + tile0 + bx));
  const int job_id = (int)(tl.x & 0xffffu), tx = (int)(tl.x >> 16), ty = (int)(tl.y & 0xffffu);
  const uint4 *jp = reinterpret_cast<const uint4 *>(plan.jobs + job_id);
  const uint4 j0 = ld_ro(jp), j1 = ld_ro(jp + 1), j2 = ld_ro(jp + 2);
  // DevJob: {src_off, dst_off, src_pitch, dst_pitch} {dst_h, dw, dh, col_off} {row_off, magic, shift, half} {..}
  const uint32_t src_off = j0.x, dst_off = j0.y;
  const int src_pitch = (int)j0.z, dst_pitch = (int)j0.w;
  const int dst_h = (int)j1.x, dw = (int)j1.y, dh = (int)j1.z;
  const uint32_t col_off = j1.w, row_off = j2.x, magic = j2.y, shift = j2.z, half = j2.w;
  // lane = column (adjacent lanes read adjacent-ish source words), each thread produces 4 consecutive rows and
  // reuses its column taps for all of them.
  const int lane = tid & 31, warp = tid >> 5;
  const int X = tx * 32 + lane;
  const int Y0 = ty * 32 + warp * 4;
  if (Y0 >= dst_h || X >= dst_pitch) return;
  uint32_t *quad = arena + (size_t)by * quad_stride;
  uint32_t xa = 0, xb = 0, wx0 = 0, wx1 = 0;
  const bool col_ok = X < dw;
  if (col_ok) {
    const uint2 cx = ld_ro(reinterpret_cast<const uint2 *>(plan.taps + col_off + X));   // {a | b<<16, f}
    xa = cx.x & 0xffffu; xb = cx.x >> 16;
    wx1 = cx.y & 0xffffu; wx0 = 2u * (uint32_t)dw - wx1;
  }
  const uint32_t Dy = 2u * (uint32_t)dh;
  const uint32_t *src = quad + src_off;
  // All 16 source words of the thread's 4 rows are requested before any arithmetic; rows below the painted area
  // read row taps {0, 0} and are zeroed afterwards, so the loads need no branches.
  uint32_t oa[4], ob[4], wy1[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int Y = Y0 + r;
    uint2 ry = make_uint2(0u, 0u);
    if (Y < dh) ry = ld_ro(reinterpret_cast<const uint2 *>(plan.taps + row_off + Y));   // warp-uniform
    oa[r] = (ry.x & 0xffffu) * (uint32_t)src_pitch;
    ob[r] = (ry.x >> 16) * (uint32_t)src_pitch;
    wy1[r] = ry.y & 0xffffu;
  }
  uint32_t p[4][4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    p[r][0] = src[oa[r] + xa]; p[r][1] = src[oa[r] + xb];
    p[r][2] = src[ob[r] + xa]; p[r][3] = src[ob[r] + xb];
  }
  uint32_t *dst = quad + dst_off + (uint32_t)Y0 * (uint32_t)dst_pitch + (uint32_t)X;
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const int Y = Y0 + r;
    if (Y >= dst_h) break;
    uint32_t out = 0;
    if (col_ok && Y < dh) {                                  // unpainted columns / rows and the pitch padding are 0
      // the four corner weights are shared by the 4 frames of the word: 4 multiply-adds per frame instead of 6
      const uint32_t wy0 = Dy - wy1[r];
      const uint32_t w00 = wx0 * wy0, w01 = wx1 * wy0, w10 = wx0 * wy1[r], w11 = wx1 * wy1[r];   // sum = 4 dw dh
#pragma unroll
      for (int f = 0; f < 4; ++f) {
        // byte f of the four tap words: one PRMT each (shift + mask compiled to SHF + LOP3: 6 instructions per word)
        const uint32_t a = quad_byte(p[r][0], f), b = quad_byte(p[r][1], f);
        const uint32_t c = quad_byte(p[r][2], f), d = quad_byte(p[r][3], f);
        // == (wx0 a + wx1 b) wy0 + (wx0 c + wx1 d) wy1 + half  <= 255.5 * 4 dw dh < 2^32 (checked by the planner)
        const uint32_t num = w00 * a + w01 * b + w10 * c + w11 * d + half;
        out |= (uint32_t)(((uint64_t)num * magic) >> shift) << (8 * f);
      }
    }
    dst[(uint32_t)r * (uint32_t)dst_pitch] = out;
  }
}

__global__ void __launch_bounds__(256) k_resample(DevPlan plan, int tile0, uint32_t *__restrict__ arena,
                                                  size_t quad_stride, int n_frames, const uint8_t *__restrict__ quad_mask) {
  if (quad_frames(blockIdx.y, n_frames, quad_mask) == 0u) return;
  resample_thread(plan, tile0, arena, quad_stride, (int)blockIdx.x, (int)blockIdx.y, (int)threadIdx.x);
}

// ------------------------------------------------------------------------------------------------
// K3  BBF cascade over all windows of one (frame quad, scale, tile) — src/ccv.js:178-243.
//
// Feature test: min over the p-points > max over the n-points.  The reference's early-outs
// (src/ccv.js:193-218) break exactly when a running min(p) <= running max(n); since min is
// non-increasing and max non-decreasing this is equivalent to the final comparison.
// Stage sum: sequential fp64 adds of alpha in feature order (bit-exact with the JS) wherever a sum is PRODUCED
// (the confidence of a detection) or a decision is a tie; everywhere else the decision `!(sum < threshold)` is
// taken on exact integers or truth tables (tools/gen_cascade_code.py, LateFeat in ht_common.cuh).

__constant__ ConstCascade c_casc;
// The stage evaluators below also compile for the HOST (tests/test_cascade_host.py emulates k_cascade's tile
// evaluation on the CPU with the very same generated code, tile layout, tables and late-stage schedule): device
// code reads the __constant__ image, host code a pointer the self-test sets.
static const ConstCascade *g_host_casc = nullptr;
#ifdef __CUDA_ARCH__
#define HT_CASC c_casc
#else
#define HT_CASC (*g_host_casc)
#endif

// ---- stages specialised at build time (tools/gen_cascade_code.py) ----
__host__ __device__ __forceinline__ unsigned min3_u32(unsigned a, unsigned b, unsigned c) {
#ifdef __CUDA_ARCH__
  return __vimin3_u32(a, b, c);      // VIMNMX3.U32 (plain min() is turned into U16x2 + masks)
#else
  return a < b ? (a < c ? a : c) : (b < c ? b : c);
#endif
}
__host__ __device__ __forceinline__ unsigned max3_u32(unsigned a, unsigned b, unsigned c) {
#ifdef __CUDA_ARCH__
  return __vimax3_u32(a, b, c);
#else
  return a > b ? (a > c ? a : c) : (b > c ? b : c);
#endif
}
__host__ __device__ __forceinline__ uint32_t min3_u16x2(uint32_t a, uint32_t b, uint32_t c) {
#ifdef __CUDA_ARCH__
  return __vimin3_u16x2(a, b, c);    // VIMNMX3.U16x2
#else
  return (min3_u32(a >> 16, b >> 16, c >> 16) << 16) | min3_u32(a & 0xffffu, b & 0xffffu, c & 0xffffu);
#endif
}
__host__ __device__ __forceinline__ uint32_t max3_u16x2(uint32_t a, uint32_t b, uint32_t c) {
#ifdef __CUDA_ARCH__
  return __vimax3_u16x2(a, b, c);
#else
  return (max3_u32(a >> 16, b >> 16, c >> 16) << 16) | max3_u32(a & 0xffffu, b & 0xffffu, c & 0xffffu);
#endif
}
__host__ __device__ __forceinline__ uint32_t frames02(uint32_t w) {   // frames 0 and 2 of a quad word as u16x2
#ifdef __CUDA_ARCH__
  return __byte_perm(w, 0u, 0x4240);
#else
  return w & 0x00ff00ffu;
#endif
}
__host__ __device__ __forceinline__ uint32_t frames13(uint32_t w) {   // frames 1 and 3
#ifdef __CUDA_ARCH__
  return __byte_perm(w, 0u, 0x4341);
#else
  return (w >> 8) & 0x00ff00ffu;
#endif
}
#define HT_GEN_FN __host__ __device__ __forceinline__
#define HT_PW(z, x, y) point_word(z, x, y)
#define HT_MIN2(a, b) min3_u32(a, b, b)
#define HT_MIN3(a, b, c) min3_u32(a, b, c)
#define HT_MAX2(a, b) max3_u32(a, b, b)
#define HT_MAX3(a, b, c) max3_u32(a, b, c)
#define HT_LO(w) frames02(w)
#define HT_HI(w) frames13(w)
#define HT_QMIN2(a, b) min3_u16x2(a, b, b)
#define HT_QMIN3(a, b, c) min3_u16x2(a, b, c)
#define HT_QMAX2(a, b) max3_u16x2(a, b, b)
#define HT_QMAX3(a, b, c) max3_u16x2(a, b, c)
#define HT_QCMP(nm, pm) ((nm) - (pm) + 0x80008000u)   /* bit 15 / 31 clear <=> min(p) > max(n) in that frame */
template <int LUT>
__host__ __device__ __forceinline__ uint32_t lop3(uint32_t a, uint32_t b, uint32_t c) {
#ifdef __CUDA_ARCH__
  uint32_t d;
  asm("lop3.b32 %0, %1, %2, %3, %4;" : "=r"(d) : "r"(a), "r"(b), "r"(c), "n"(LUT));
  return d;
#else
  uint32_t d = 0;   // bit i of LUT is the output for (a,b,c) = bits (2,1,0) of i
  for (int i = 0; i < 8; ++i)
    if ((LUT >> i) & 1) d |= ((i & 4) ? a : ~a) & ((i & 2) ? b : ~b) & ((i & 1) ? c : ~c);
  return d;
#endif
}
// stage decision as a truth table of the four "feature did not fire" bits: x3 ? B(x0,x1,x2) : A(x0,x1,x2)
#define HT_LUT4(x0, x1, x2, x3, A, B) lop3<0xCA>(x3, lop3<B>(x0, x1, x2), lop3<A>(x0, x1, x2))
#include "cascade_face_gen.inc"
#undef HT_GEN_FN
#undef HT_PW
#undef HT_MIN2
#undef HT_MIN3
#undef HT_MAX2
#undef HT_MAX3
#undef HT_LO
#undef HT_HI
#undef HT_QMIN2
#undef HT_QMIN3
#undef HT_QMAX2
#undef HT_QMAX3
#undef HT_QCMP
#undef HT_LUT4

// byte address of a table offset (ConstCascade::off / LateFeat::off): bit 15 selects baseB
__host__ __device__ __forceinline__ unsigned px_at(const uint8_t *__restrict__ tA, const uint8_t *__restrict__ tB, unsigned o) {
  return (o & 0x8000u) ? tB[4u * (o & 0x7fffu)] : tA[4u * o];
}

// The reference's stage sum for one window: ordered fp64 adds, src/ccv.js:186-221.  All table reads are uniform.
__host__ __device__ __noinline__ double stage_sum_ordered(const uint8_t *__restrict__ tA, const uint8_t *__restrict__ tB, int j) {
  const int first = HT_CASC.stage[j].first, last = first + HT_CASC.stage[j].count;
  double sum = 0.0;
  for (int k = first; k < last; ++k) {
    const unsigned kind = HT_CASC.np_nn[k];
    const unsigned np = kind & 15u, nn = kind >> 4;
    unsigned pmin = px_at(tA, tB, HT_CASC.off[k][0]);
    unsigned nmax = px_at(tA, tB, HT_CASC.off[k][5]);
    for (unsigned i = 1; i < np; ++i) pmin = min3_u32(pmin, pmin, px_at(tA, tB, HT_CASC.off[k][i]));
    for (unsigned i = 1; i < nn; ++i) nmax = max3_u32(nmax, nmax, px_at(tA, tB, HT_CASC.off[k][5 + i]));
    const double a = HT_CASC.alpha[k];
    sum += (pmin > nmax) ? a : -a;   // src/ccv.js:194,219 (alpha[2k] == -alpha[2k+1], checked on the host)
  }
  return sum;
}
__host__ __device__ __forceinline__ bool stage_pass_ordered(const uint8_t *tA, const uint8_t *tB, int j) {
  return !(stage_sum_ordered(tA, tB, j) < HT_CASC.stage[j].threshold);   // src/ccv.js:222
}

// predicated ld.shared.u8: lanes with p == false issue no shared-memory access and return dflt
__device__ __forceinline__ unsigned lds_u8_if(unsigned saddr, bool p, unsigned dflt) {
  unsigned v = dflt;
  asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q ld.shared.u8 %0, [%1];\n\t}" : "+r"(v) : "r"(saddr), "r"((unsigned)p));
  return v;
}

// One feature record (LateFeat, three 16-byte loads) for one window, evaluated by one lane: min(p) > max(n).
// sBm = sB - 2^31: an entry with bit 31 set (relative to baseB) then needs no masking.
__device__ __forceinline__ bool feat_fires(unsigned sA, unsigned sBm, const uint4 a, const uint4 b, const uint4 c) {
  const unsigned o[10] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y};
  unsigned vv[10];
#pragma unroll
  for (int s = 0; s < 10; ++s) {
    const unsigned addr = ((int)o[s] < 0 ? sBm : sA) + o[s];
    vv[s] = lds_u8_if(addr, o[s] != LATE_UNUSED, s < 5 ? 255u : 0u);   // unused slots: neutral element, no bank traffic
  }
  const unsigned pm = __vimin3_u32(__vimin3_u32(vv[0], vv[1], vv[2]), vv[3], vv[4]);
  const unsigned nm = __vimax3_u32(__vimax3_u32(vv[5], vv[6], vv[7]), vv[8], vv[9]);
  return pm > nm;
}

// The reference's ordered fp64 stage sum (src/ccv.js:186-221) for ONE window by a whole warp: the 32 lanes evaluate
// 32 features at a time (feature records in ORIGINAL order), the fire bits are collected with a ballot, and every
// lane then performs the same sequential chain of fp64 adds in feature order (uniform alpha reads).  Round 2's
// first version ran stage_sum_ordered on every lane: 14 k instructions of dependent loads per detection, the
// straggler that set the duration of every CTA with a face in it.
__device__ __forceinline__ double stage_sum_ordered_warp(unsigned sA, unsigned sBm, int j, const LateFeat *__restrict__ feat_orig,
                                                         int lane) {
  const int first = c_casc.stage[j].first, count = c_casc.stage[j].count;
  double sum = 0.0;
  for (int base = 0; base < count; base += 32) {
    bool fired = false;
    if (base + lane < count) {
      const uint4 *fp = reinterpret_cast<const uint4 *>(feat_orig + first + base + lane);
      fired = feat_fires(sA, sBm, __ldg(fp), __ldg(fp + 1), __ldg(fp + 2));
    }
    const unsigned mask = __ballot_sync(0xffffffffu, fired);
    const int n = min(32, count - base);
    for (int i = 0; i < n; ++i) {
      const double a = c_casc.alpha[first + base + i];
      sum += ((mask >> i) & 1u) ? a : -a;   // src/ccv.js:194,219 (alpha[2k] == -alpha[2k+1], checked on the host)
    }
  }
  return sum;
}

__device__ __forceinline__ void cp_async4(unsigned saddr, const void *g, bool valid) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(saddr), "l"(g), "r"(valid ? 4u : 0u) : "memory");
}

// Debug switches of the exactness fallbacks (ht_debug_set_exactness): bit 0 = treat every generated byte-stage
// decision as a tie, bit 1 = treat every late-stage integer decision as a tie.  Ties are decided by the reference's
// ordered fp64 adds, so results must not change (tests/test_gpu_quads.py).
// a compile-time int that converts to int in device code (std::integral_constant's conversion is a host function)
template <int V>
struct IntC {
  __host__ __device__ constexpr operator int() const { return V; }
};
// warp-wide reductions in one REDUX instruction each (sm_80+), instead of five shuffle + op rounds
__device__ __forceinline__ int warp_max_i32(int v) { return (int)__reduce_max_sync(0xffffffffu, (unsigned)v); }   // v >= 0
// sum of 32 signed 64-bit values with |v| < 2^46 (late-stage integer sums: <= 66 chunks x |alpha_int| < 2^31 per lane):
// offset to positive, two 24/23-bit halves summed separately (each total < 2^29), recombined
__device__ __forceinline__ long long warp_sum_i64(long long v) {
  const unsigned long long u = (unsigned long long)(v + (1ll << 46));
  const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(u & 0xffffffull));
  const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(u >> 24));
  return (long long)(((unsigned long long)hi << 24) + lo) - (32ll << 46);
}
// position of the r-th (0-based) set bit of w, r < popc(w): five popcount halvings, ~25 instructions (__fns is a
// software loop; round 2, call 8: 7 % of k_cascade's samples sat in it and its caller)
__device__ __forceinline__ int nth_bit32(uint32_t w, int r) {
  int pos = 0, t;
  t = __popc(w & 0xffffu); if (r >= t) { r -= t; pos += 16; w >>= 16; }
  t = __popc(w & 0xffu);   if (r >= t) { r -= t; pos += 8;  w >>= 8; }
  t = __popc(w & 0xfu);    if (r >= t) { r -= t; pos += 4;  w >>= 4; }
  t = __popc(w & 0x3u);    if (r >= t) { r -= t; pos += 2;  w >>= 2; }
  t = (int)(w & 1u);       if (r >= t) pos += 1;
  return pos;
}
// r-th (0-based) set bit of the MASK_WORDS-word mask of class c, or -1.  All reads are shared-memory loads.
__device__ __forceinline__ int nth_set_bit(const uint32_t *__restrict__ masks, int c, int r) {
#pragma unroll
  for (int j = 0; j < MASK_WORDS; ++j) {
    const uint32_t w = masks[j * 32 + c];
    const int pc = __popc(w);
    if (r < pc) return j * 32 + nth_bit32(w, r);
    r -= pc;
  }
  return -1;
}

template <bool FAST>
__global__ void __launch_bounds__(CASCADE_THREADS, CASCADE_MIN_BLOCKS) k_cascade(DevPlan plan, const LateFeat *__restrict__ late,
                                                                const LateFeat *__restrict__ feat_orig,
                                                                const int32_t *__restrict__ late_chunk0,
                                                                const void *__restrict__ tmaps, int tma_quad0,
                                                                const uint32_t *__restrict__ arena, size_t quad_stride,
                                                                int n_frames, uint32_t *__restrict__ raw_keys,
                                                                double *__restrict__ raw_conf,
                                                                uint32_t *__restrict__ raw_count, int raw_cap,
                                                                int force_ties, const uint8_t *__restrict__ quad_mask) {
  if (quad_frames(blockIdx.y, n_frames, quad_mask) == 0u) return;   // uniform over the CTA
  extern __shared__ __align__(128) uint32_t smem[];   // (the TMA destination inside it needs 128-byte alignment)
  uint32_t *tile = smem;                                // TILE_WORDS
  uint32_t *masks = smem + TILE_WORDS;                  // [3][MASK_WORDS][32] survivor bit masks (in / out / being cleared)
  __shared__ __align__(8) unsigned long long tma_bar;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int quad = blockIdx.y;
  const DevCascTile tl = plan.casc_tiles[blockIdx.x];
  const DevScale sc = plan.scales[tl.scale];
  const uint32_t *qa = arena + (size_t)quad * quad_stride;
  const int x0 = tl.tx * TW, y0 = tl.ty * TH;  // quarter-res origin of the tile
  const unsigned fmask = quad_frames(quad, n_frames, quad_mask);

  for (int i = tid; i < 3 * MASK_WORDS * 32; i += CASCADE_THREADS) masks[i] = 0u;

  // ---- stage the three levels in shared memory (layout in ht_common.cuh) ----
  // Level 1 is a plain 2-D box of its plane (L1_ROWS x P1 words): when tensor maps are given it is staged by the
  // TMA engine - one elected thread issues cp.async.bulk.tensor (3-D map: column, row, frame quad; elements outside
  // the plane are zero-filled) completing on an mbarrier - while all threads scatter levels 0 and 2.
  const bool use_tma = tmaps != nullptr;
  if (use_tma) {
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&tma_bar);
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();   // nobody may poll the barrier before it is initialised
    if (tid == 0) {
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"((unsigned)(L1_ROWS * P1 * 4)) : "memory");
      const unsigned dst = (unsigned)__cvta_generic_to_shared(tile + W1);
      const unsigned long long map = (unsigned long long)(reinterpret_cast<const uint8_t *>(tmaps) + 128 * (size_t)tl.scale);
      asm volatile(
          "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
          ::"r"(dst), "l"(map), "r"(2 * x0), "r"(2 * y0), "r"(tma_quad0 + quad), "r"(bar)
          : "memory");
    }
  }
  {
    // 16-byte global loads (4 consecutive pixels x 4 frames), the layout permutation in the shared-memory stores;
    // words outside a plane are zero.  Plane pitches and all tile origins are multiples of 4 words.
    {  // level 0, columns split by parity: X, X+2 -> even half (one 8 B store), X+1, X+3 -> odd half
      const DevPlane pl = plan.planes[sc.p0];
      const uint32_t *src = qa + pl.off;
      const int X0 = 4 * x0, Y0 = 4 * y0;
      constexpr int G0 = (L0_COLS + 3) / 4;             // 38 groups per row (the last one half used)
      for (int i0 = tid; i0 < L0_ROWS * G0; i0 += 4 * CASCADE_THREADS) {
        uint4 v[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int i = i0 + k * CASCADE_THREADS, r = i / G0, X = (i - r * G0) * 4;
          v[k] = make_uint4(0u, 0u, 0u, 0u);
          if (i < L0_ROWS * G0 && Y0 + r < pl.h && X0 + X < pl.pitch)
            v[k] = __ldg(reinterpret_cast<const uint4 *>(src + (size_t)(Y0 + r) * pl.pitch + X0 + X));
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int i = i0 + k * CASCADE_THREADS, r = i / G0, X = (i - r * G0) * 4;
          if (i >= L0_ROWS * G0) break;
          uint32_t *row = tile + tile_l0(r, X);   // (X % 4 == 0: the even half; the odd half is H0 words further)
          if (X + 2 < L0_COLS) *reinterpret_cast<uint2 *>(row) = make_uint2(v[k].x, v[k].z);   // even columns X, X+2
          else row[0] = v[k].x;                            // last group of a row: X+2 is outside the tile
          if (X + 1 < L0_COLS) row[H0] = v[k].y;           // odd columns X+1, X+3
          if (X + 3 < L0_COLS) row[H0 + 1] = v[k].w;
        }
      }
    }
    if (!use_tma) {  // level 1: a plain box, 16-byte cp.async
      const DevPlane pl = plan.planes[sc.p1];
      const uint32_t *src = qa + pl.off;
      const int X0 = 2 * x0, Y0 = 2 * y0;
      constexpr int G1 = P1 / 4;                          // 19 groups per row
      for (int i = tid; i < L1_ROWS * G1; i += CASCADE_THREADS) {
        const int r = i / G1, c = (i - r * G1) * 4;
        const bool ok = (Y0 + r < pl.h) && (X0 + c < pl.pitch);
        const unsigned dst = (unsigned)__cvta_generic_to_shared(tile + tile_l1(r, c));
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(ok ? src + (size_t)(Y0 + r) * pl.pitch + X0 + c : src),
                     "r"(ok ? 16u : 0u) : "memory");
      }
    }
    {  // level 2: the four phase copies interleaved (row 2Y+dy, column 2X+dx): the dx = 0 / 1 copies of one dy are
       // loaded together and written as two 16-byte stores of 8 consecutive words
      constexpr int G2 = (L2_COLS + 3) / 4;               // 10 groups per row
      for (int i = tid; i < 2 * L2_ROWS * G2; i += CASCADE_THREADS) {
        const int dy = i / (L2_ROWS * G2), rem = i - dy * (L2_ROWS * G2), r = rem / G2, c = (rem - r * G2) * 4;
        uint4 v0 = make_uint4(0u, 0u, 0u, 0u), v1 = v0;
        {
          const DevPlane pl = plan.planes[plan.scales[tl.scale].p2[2 * dy]];      // (indexing the register copy `sc` would spill it)
          if (y0 + r < pl.h && x0 + c < pl.pitch) v0 = __ldg(reinterpret_cast<const uint4 *>(qa + pl.off + (size_t)(y0 + r) * pl.pitch + x0 + c));
        }
        {
          const DevPlane pl = plan.planes[plan.scales[tl.scale].p2[2 * dy + 1]];
          if (y0 + r < pl.h && x0 + c < pl.pitch) v1 = __ldg(reinterpret_cast<const uint4 *>(qa + pl.off + (size_t)(y0 + r) * pl.pitch + x0 + c));
        }
        uint32_t *row = tile + tile_l2(2 * r + dy, 2 * c);
        *reinterpret_cast<uint4 *>(row) = make_uint4(v0.x, v1.x, v0.y, v1.y);
        if (2 * c + 8 <= P2) *reinterpret_cast<uint4 *>(row + 4) = make_uint4(v0.z, v1.z, v0.w, v1.w);   // (P2 = 76 = 9 * 8 + 4)
      }
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
  }
  if (use_tma) {   // every thread observes the completion of the bulk copy (phase 0 of the barrier)
    const unsigned bar = (unsigned)__cvta_generic_to_shared(&tma_bar);
    unsigned done = 0;
    for (int spin = 0; !done && spin < (1 << 24); ++spin) {   // bounded: a bad descriptor must not hang the device
      asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                   : "=r"(done) : "r"(bar) : "memory");
    }
    if (!done) __trap();
  }
  __syncthreads();

  // A window of the tile is (class c, bit b): b = 8 v + 4 uh + f, u = class_u(c, v, uh), f = frame in the quad.
  // Lane L evaluates class L in EVERY phase: base words of a warp's 32 windows are consecutive modulo 32 -> every
  // load, quad or byte, is bank-conflict free.
  const uint8_t *tile_b = reinterpret_cast<const uint8_t *>(tile);
  auto emit = [&](int c, int b, double sum) {  // src/ccv.js:227-234: (window id in reference order, last stage sum)
    const int v = b >> 3, uh = (b >> 2) & 1, f = b & 3, u = class_u(c, v, uh);
    const int lx = u >> 1, ly = v >> 1, q = (u & 1) | ((v & 1) << 1);
    const uint32_t key = sc.win_base + (uint32_t)((q * sc.qh + (y0 + ly)) * sc.qw + (x0 + lx));
    const int frame = 4 * quad + f;
    const uint32_t pos = atomicAdd(&raw_count[frame], 1u);
    if (pos < (uint32_t)raw_cap) {
      raw_keys[(size_t)frame * raw_cap + pos] = key;
      raw_conf[(size_t)frame * raw_cap + pos] = sum;
    }
  };
  auto bases = [&](int c, int b, const uint8_t *&tA, const uint8_t *&tB) {
    const int v = b >> 3, uh = (b >> 2) & 1, f = b & 3, u = class_u(c, v, uh);
    tA = tile_b + 4 * (v * VA + u) + f;
    tB = tile_b + 4 * (v * VB + u) + f;
  };
  const int late_first = c_casc.group_first[c_casc.n_groups];
  const bool has_late = late_first < c_casc.n_stages;
  uint32_t *m_in = masks, *m_out = masks + MASK_WORDS * 32, *m_clr = masks + 2 * MASK_WORDS * 32;

  // ---- dense group: every window of the tile.  A warp takes chunks of 4 (v, uh) units = 16 mask bits per lane ----
  {
    static_assert(HT_GEN_QUAD_STAGES == 2, "the dense group is {0,1}");
    uint16_t *m16 = reinterpret_cast<uint16_t *>(m_in);
    for (int chunk = warp; chunk < NV / 2; chunk += CASCADE_WARPS) {
      uint32_t bits = 0;
#pragma unroll 1
      for (int unit = 0; unit < 4; ++unit) {
        const int v = 2 * chunk + (unit >> 1), uh = unit & 1, u = class_u(lane, v, uh);
        const int lx = u >> 1, ly = v >> 1;
        uint32_t m = 0;
        if (FAST) {
          // quad form (cascade_face_gen.inc): 4 frames per lane
          const uint32_t *tA = tile + v * VA + u, *tB = tile + v * VB + u;
          uint32_t a_lo = 0, a_hi = 0;   // alive bits: frame 0 -> lo bit 15, 2 -> lo bit 31, 1 -> hi bit 15, 3 -> hi bit 31
          if (x0 + lx < sc.qw && y0 + ly < sc.qh) {
            a_lo = ((fmask & 1u) ? 0x8000u : 0u) | ((fmask & 4u) ? 0x80000000u : 0u);
            a_hi = ((fmask & 2u) ? 0x8000u : 0u) | ((fmask & 8u) ? 0x80000000u : 0u);
          }
#define HT_QSTAGE(J)                                                                                        \
  if (__any_sync(0xffffffffu, (a_lo | a_hi) != 0u)) {                                                        \
    uint32_t p_lo, p_hi, t_lo, t_hi;                                                                         \
    gen_q_stage##J(tA, tB, p_lo, p_hi, t_lo, t_hi);                                                          \
    t_lo &= a_lo; t_hi &= a_hi;                                                                              \
    if (t_lo | t_hi) { /* exact decimal tie (never seen in practice): the reference's ordered adds decide */ \
      for (int f = 0; f < 4; ++f) {                                                                          \
        const uint32_t bit = (f & 2) ? 0x80000000u : 0x8000u;                                                \
        uint32_t &tt = (f & 1) ? t_hi : t_lo, &pp = (f & 1) ? p_hi : p_lo;                                   \
        if (tt & bit) {                                                                                      \
          const uint8_t *bA = reinterpret_cast<const uint8_t *>(tA) + f, *bB = reinterpret_cast<const uint8_t *>(tB) + f; \
          if (!stage_pass_ordered(bA, bB, J)) pp &= ~bit;                                                    \
        }                                                                                                    \
      }                                                                                                      \
    }                                                                                                        \
    a_lo &= p_lo; a_hi &= p_hi;                                                                              \
  }
          HT_QSTAGE(0)
          HT_QSTAGE(1)
#undef HT_QSTAGE
          m = ((a_lo >> 15) & 1u) | ((a_hi >> 14) & 2u) | ((a_lo >> 29) & 4u) | ((a_hi >> 28) & 8u);
        } else {
          // table-driven: ordered fp64 sums, one frame at a time
          for (int f = 0; f < 4; ++f) {
            bool alive = (x0 + lx < sc.qw) && (y0 + ly < sc.qh) && ((fmask >> f) & 1u);
            const uint8_t *tA = tile_b + 4 * (v * VA + u) + f, *tB = tile_b + 4 * (v * VB + u) + f;
            for (int j = c_casc.group_first[0]; j < c_casc.group_first[1]; ++j) {
              if (!__any_sync(0xffffffffu, alive)) break;
              alive = alive && stage_pass_ordered(tA, tB, j);
            }
            m |= (alive ? 1u : 0u) << f;
          }
        }
        bits |= m << (4 * unit);      // bit (8 v + 4 uh + f) & 15 of this half word
      }
      m16[(((chunk >> 1) * 32 + lane) << 1) | (chunk & 1)] = (uint16_t)bits;
    }
  }
  __syncthreads();

  // ---- survivor masks: lane L walks the set bits of class L; warp w takes the entries of rank w, w + NW, ... ----
  // One group = stages [jb, je).  For the generated cascade the bounds are compile-time constants (integral_constant
  // arguments): the stage loop unrolls and gen_stage's switch folds away (round 2, call 8: 3.4 % of the samples sat in
  // that dispatch).  Returns true when the CTA is finished.
  auto run_group = [&](auto JB, auto JE, const bool emit_here) __attribute__((always_inline)) -> bool {
    const int jb = JB, je = JE;
    int n = 0;
#pragma unroll
    for (int j = 0; j < MASK_WORDS; ++j) n += __popc(m_in[j * 32 + lane]);
    if (warp_max_i32(n) == 0) return true;   // uniform over the CTA
    for (int i = tid; i < MASK_WORDS * 32; i += CASCADE_THREADS) m_clr[i] = 0u;   // the mask of the group after next
    // warp w takes the entries of rank [w n / NW, (w+1) n / NW) of every class: one nth_set_bit per lane and group,
    // then a walk over consecutive set bits (round-2 call 3: rank-strided entries spent 16 % of the kernel's
    // instructions in __fns)
    const int r_beg = (warp * n) / CASCADE_WARPS, r_end = ((warp + 1) * n) / CASCADE_WARPS;
    const int my_iters = r_end - r_beg;
    const int iters = warp_max_i32(my_iters);
    int bpos = my_iters > 0 ? nth_set_bit(m_in, lane, r_beg) : 0;       // bit index of the current entry
    uint32_t cur = my_iters > 0 ? (m_in[(bpos >> 5) * 32 + lane] & (0xffffffffu << (bpos & 31))) : 0u;   // its word, lower bits cleared
    for (int it = 0; it < iters; ++it) {
      bool alive = it < my_iters;
      int b = 0;
      if (alive) {
        while (cur == 0u) { bpos = (bpos | 31) + 1; cur = m_in[(bpos >> 5) * 32 + lane]; }   // next word of the class
        b = (bpos & ~31) | (__ffs(cur) - 1);
        cur &= cur - 1u;
        bpos = b;
      }
      const uint8_t *tA, *tB;
      bases(lane, b, tA, tB);
      double sum = 0.0;
#pragma unroll
      for (int j = jb; j < je; ++j) {
        if (!__any_sync(0xffffffffu, alive)) break;
        if (FAST && j < HT_GEN_STAGES) {
          int rr = gen_stage(j, tA, tB);
          if (force_ties & 1) rr = -1;
          if (rr < 0) rr = stage_pass_ordered(tA, tB, j) ? 1 : 0;
          alive = alive && (rr != 0);
        } else {
          sum = stage_sum_ordered(tA, tB, j);
          alive = alive && !(sum < c_casc.stage[j].threshold);
        }
      }
      if (alive) {
        if (emit_here) {
          if (FAST && je - 1 < HT_GEN_STAGES) sum = stage_sum_ordered(tA, tB, je - 1);
          emit(lane, b, sum);
        } else {
          atomicOr(&m_out[(b >> 5) * 32 + lane], 1u << (b & 31));
        }
      }
    }
    if (emit_here) return true;
    __syncthreads();
    uint32_t *t = m_in; m_in = m_out; m_out = m_clr; m_clr = t;
    return false;
  };
  if (FAST) {
    // the generated groups {2} {3} {4,5} {6,7} (parse_cascade's cuts_fast; the dense group covered {0,1})
    static_assert(HT_GEN_STAGES == 8, "compile-time groups assume 8 generated stages");
    if (run_group(IntC<2>{}, IntC<3>{}, false)) return;
    if (run_group(IntC<3>{}, IntC<4>{}, false)) return;
    if (run_group(IntC<4>{}, IntC<6>{}, false)) return;
    if (run_group(IntC<6>{}, IntC<8>{}, !has_late)) return;
  } else {
    for (int g = 1; g < c_casc.n_groups; ++g)
      if (run_group(c_casc.group_first[g], c_casc.group_first[g + 1], (g == c_casc.n_groups - 1) && !has_late)) return;
  }
  if (!has_late) {
    if (c_casc.n_groups == 1) {   // a cascade that ends with the dense group: emit its survivors
      int n = 0;
#pragma unroll
      for (int j = 0; j < MASK_WORDS; ++j) n += __popc(m_in[j * 32 + lane]);
      for (int r = warp; r < n; r += CASCADE_WARPS) {
        const int b = nth_set_bit(m_in, lane, r);
        const uint8_t *tA, *tB;
        bases(lane, b, tA, tB);
        emit(lane, b, stage_sum_ordered(tA, tB, c_casc.n_stages - 1));
      }
    }
    return;
  }

  // ---- late stages: one warp per surviving window, one feature per lane, exact integer sums.  The features of
  //      a stage are pre-arranged in chunks of 32 (build_late_schedule, ht_api.cu) so that the 32 addresses of
  //      each load slot fall into 32 different banks: the order of an exact integer sum is free ----
  {
    int mylen = 0;
#pragma unroll
    for (int j = 0; j < MASK_WORDS; ++j) mylen += __popc(m_in[j * 32 + lane]);
    int incl = mylen;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31), excl = incl - mylen;
    for (int wdx = warp; wdx < total; wdx += CASCADE_WARPS) {
      const unsigned owner = __ballot_sync(0xffffffffu, wdx >= excl && wdx < incl);
      const int c = __ffs(owner) - 1;
      const int b = nth_set_bit(m_in, c, wdx - __shfl_sync(0xffffffffu, excl, c));
      const uint8_t *tA, *tB;
      bases(c, b, tA, tB);
      const unsigned sA = (unsigned)__cvta_generic_to_shared(tA), sBm = (unsigned)__cvta_generic_to_shared(tB) - 0x80000000u;
      bool pass = true;
      for (int j = late_first; j < c_casc.n_stages && pass; ++j) {
        long long acc = 0;
        const int c0 = late_chunk0[j], c1 = late_chunk0[j + 1];
        for (int ch = c0; ch < c1; ++ch) {
          const uint4 *fp = reinterpret_cast<const uint4 *>(late + (size_t)ch * 32 + lane);
          const uint4 a = __ldg(fp), bb = __ldg(fp + 1), cc = __ldg(fp + 2);
          const int ai = (int)cc.z;                      // alpha_int (0 for padding records)
          acc += feat_fires(sA, sBm, a, bb, cc) ? (long long)ai : -(long long)ai;
        }
        acc = warp_sum_i64(acc);
        const long long thr = c_casc.thr_int[j];
        if (acc == thr || (force_ties & 2))             // exact tie: the reference's ordered adds decide
          pass = !(stage_sum_ordered_warp(sA, sBm, j, feat_orig, lane) < c_casc.stage[j].threshold);
        else pass = acc > thr;
      }
      if (pass) {  // confidence = ordered fp64 sum of the last stage
        const double s = stage_sum_ordered_warp(sA, sBm, c_casc.n_stages - 1, feat_orig, lane);
        if (lane == 0) emit(c, b, s);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// K4  sort raw detections into the reference's (i,q,y,x) order and group them —
// src/ccv.js:34-107 (array_group), 249-332.  One warp per frame.
//
// array_group's union-find yields the connected components of the symmetric closure of the
// predicate, numbered by smallest member index (src/ccv.js:90-105); any components algorithm
// gives the same partition, so min-label propagation is used.  Sums run in list order per class
// (fp64, order-sensitive) exactly as src/ccv.js:274-289.

__device__ __forceinline__ bool group_pred(const Rect &r1, const Rect &r2) {  // src/ccv.js:252-261
  const double distance = floor(r1.width * 0.25 + 0.5);
  return r2.x <= r1.x + distance && r2.x >= r1.x - distance && r2.y <= r1.y + distance &&
         r2.y >= r1.y - distance && r2.width <= floor(r1.width * 1.5 + 0.5) &&
         floor(r2.width * 1.5 + 0.5) >= r1.width;
}

__global__ void __launch_bounds__(128) k_group(DevPlan plan, int n_frames, const uint32_t *__restrict__ raw_keys,
                                               const double *__restrict__ raw_conf,
                                               const uint32_t *__restrict__ raw_count, int raw_cap,
                                               Rect *__restrict__ sorted, int *__restrict__ labels,
                                               Rect *__restrict__ seq2, int min_neighbors,
                                               Rect *__restrict__ out_rects, int32_t *__restrict__ out_counts, int K,
                                               int32_t *__restrict__ overflow_flag) {
  const int lane = threadIdx.x & 31;
  const int frame = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (frame >= n_frames) return;
  const unsigned FULL = 0xffffffffu;
  const uint32_t n_true = raw_count[frame];
  const int n = (int)min(n_true, (uint32_t)raw_cap);
  if (n_true > (uint32_t)raw_cap && lane == 0) atomicOr(overflow_flag, 1);
  const uint32_t *keys = raw_keys + (size_t)frame * raw_cap;
  const double *conf = raw_conf + (size_t)frame * raw_cap;
  Rect *S = sorted + (size_t)frame * raw_cap;
  int *L = labels + (size_t)frame * raw_cap;
  Rect *S2 = seq2 + (size_t)frame * raw_cap;
  Rect *O = out_rects + (size_t)frame * K;

  // 1. rank sort by window id (ids are unique) and decode to rectangles, src/ccv.js:228-233
  for (int i = lane; i < n; i += 32) {
    const uint32_t key = keys[i];
    int rank = 0;
    for (int j = 0; j < n; ++j) rank += (keys[j] < key) ? 1 : 0;
    int s = 0;
    for (int t = 1; t < plan.n_scales; ++t)
      if (plan.scales[t].win_base <= key && plan.scales[t].qw > 0 && plan.scales[t].qh > 0) s = t;
    const DevScale sc = plan.scales[s];
    uint32_t rem = key - sc.win_base;
    const uint32_t per_q = (uint32_t)(sc.qw * sc.qh);
    const uint32_t q = rem / per_q;
    rem -= q * per_q;
    const uint32_t y = rem / (uint32_t)sc.qw, x = rem - y * (uint32_t)sc.qw;
    Rect r;
    r.x = (double)(x * 4 + (q & 1) * 2) * sc.scale_x;
    r.y = (double)(y * 4 + (q >> 1) * 2) * sc.scale_x;  // scale_y == scale_x, src/ccv.js:244-245
    r.width = 24.0 * sc.scale_x;
    r.height = 24.0 * sc.scale_x;
    r.confidence = conf[i];
    r.neighbors = 1;
    r.pad_ = 0;
    S[rank] = r;
  }
  __syncwarp();

  if (!(min_neighbors > 0)) {  // src/ccv.js:249-250: raw list
    for (int i = lane; i < n && i < K; i += 32) O[i] = S[i];
    if (lane == 0) {
      out_counts[frame] = min(n, K);
      if (n > K) atomicOr(overflow_flag, 1);
    }
    return;
  }

  // 2. connected components by min-label propagation + pointer jumping
  for (int i = lane; i < n; i += 32) L[i] = i;
  __syncwarp();
  for (;;) {
    bool changed = false;
    for (int i = lane; i < n; i += 32) {
      const Rect ri = S[i];
      int li = L[i];
      for (int j = 0; j < n; ++j) {
        if (j == i) continue;
        const Rect rj = S[j];
        if (group_pred(ri, rj) || group_pred(rj, ri)) li = min(li, L[j]);
      }
      li = min(li, L[li]);
      if (li < L[i]) { L[i] = li; changed = true; }
    }
    __syncwarp();
    if (!__any_sync(FULL, changed)) break;
  }
  // flatten: every label points at the component's smallest index
  for (int i = lane; i < n; i += 32) {
    int li = L[i];
    while (L[li] != li) li = L[li];
    L[i] = li;
  }
  __syncwarp();

  // 3. per class (in order of smallest member): ordered sums, src/ccv.js:274-303
  int n2 = 0;
  for (int base = 0; base < n; base += 32) {
    const int i = base + lane;
    const bool is_root = (i < n) && (L[i] == i);
    Rect c;
    c.x = c.y = c.width = c.height = c.confidence = 0.0;
    c.neighbors = 0; c.pad_ = 0;
    if (is_root) {
      for (int j = i; j < n; ++j) {
        if (L[j] != i) continue;
        const Rect r1 = S[j];
        if (c.neighbors == 0) c.confidence = r1.confidence;
        ++c.neighbors;
        c.x += r1.x; c.y += r1.y; c.width += r1.width; c.height += r1.height;
        c.confidence = fmax(c.confidence, r1.confidence);
      }
    }
    const bool keep = is_root && c.neighbors >= min_neighbors;
    const unsigned m = __ballot_sync(FULL, keep);
    if (keep) {
      const double nn = (double)c.neighbors;
      Rect r;
      r.x = (c.x * 2 + nn) / (2 * nn);
      r.y = (c.y * 2 + nn) / (2 * nn);
      r.width = (c.width * 2 + nn) / (2 * nn);
      r.height = (c.height * 2 + nn) / (2 * nn);
      r.neighbors = c.neighbors;
      r.confidence = c.confidence;
      r.pad_ = 0;
      S2[n2 + __popc(m & ((1u << lane) - 1u))] = r;
    }
    n2 += __popc(m);
  }
  __syncwarp();

  // 4. drop rectangles contained in a better one, src/ccv.js:307-330
  int n_out = 0;
  for (int base = 0; base < n2; base += 32) {
    const int i = base + lane;
    bool flag = i < n2;
    Rect r1;
    if (flag) {
      r1 = S2[i];
      for (int j = 0; j < n2; ++j) {
        const Rect r2 = S2[j];
        const double distance = floor(r2.width * 0.25 + 0.5);
        if (i != j && r1.x >= r2.x - distance && r1.y >= r2.y - distance &&
            r1.x + r1.width <= r2.x + r2.width + distance && r1.y + r1.height <= r2.y + r2.height + distance &&
            (r2.neighbors > max(3, r1.neighbors) || r1.neighbors < 3)) {
          flag = false;
          break;
        }
      }
    }
    const unsigned m = __ballot_sync(FULL, flag);
    if (flag) {
      const int pos = n_out + __popc(m & ((1u << lane) - 1u));
      if (pos < K) O[pos] = r1;
    }
    n_out += __popc(m);
  }
  if (lane == 0) {
    out_counts[frame] = min(n_out, K);
    if (n_out > K) atomicOr(overflow_flag, 1);
  }
}

}  // namespace ht
