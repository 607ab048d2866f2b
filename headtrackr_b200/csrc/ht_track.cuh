// ht_track.cuh — sm_100a kernels for camshift.Tracker (/root/reference/src/camshift.js) and
// getWhitebalance (/root/reference/src/whitebalance.js).
//
// The reference materialises a whole-frame back-projection (307,200 doubles in nested arrays,
// src/camshift.js:332-353) on every track(); here the weight of a pixel is looked up on the fly
// inside the search window, so a track() costs one streaming histogram pass over the frame plus a
// few window passes that stay in L2.
#pragma once
#include <cooperative_groups.h>

#include <limits>

#include "ht_common.cuh"

namespace ht {

// rgb_bin() (src/camshift.js:63-66, 345-348) is defined in ht_detect.cuh: the fused gray pass uses it too.

// ------------------------------------------------------------------------------------------------
// K1'  4096-bin RGB histogram of whole frames — src/camshift.js:49-72 via :268 — plus the per-pixel
// bin plane (u16) that k_track's window passes read instead of re-decoding RGBA (half the bytes).  The plane
// holds 8 * bin: the byte offset of the pixel's weight in k_track's fp64 table (8 * 4095 < 2^16).
// grid = (chunks, n_frames).  Shared-memory histogram per CTA, flushed to hist[frame][4096].
__global__ void __launch_bounds__(256) k_hist(const uint8_t *__restrict__ rgba, size_t frame_bytes, int n_px,
                                              uint32_t *__restrict__ hist, uint16_t *__restrict__ bins, int chunks,
                                              const uint8_t *__restrict__ enable) {
  __shared__ uint32_t sh[4096];
  if (enable && !enable[blockIdx.y]) return;   // ht_stream_step: only the streams that are tracking
  for (int i = threadIdx.x; i < 4096; i += 256) sh[i] = 0;
  __syncthreads();
  const uint32_t *px = reinterpret_cast<const uint32_t *>(rgba + (size_t)blockIdx.y * frame_bytes);
  uint16_t *bout = bins ? bins + (size_t)blockIdx.y * n_px : nullptr;
  const int n_pair = (n_px + 1) / 2;
  const int per = (n_pair + chunks - 1) / chunks;
  const int beg = blockIdx.x * per, end = min(n_pair, beg + per);
  // the 8 B load / 4 B store of the paired path need this FRAME's pointers aligned: with an odd w*h every odd frame
  // index starts at 4 mod 8 (and its bin plane at 2 mod 4), and the caller's pointer is only 4-byte aligned
  const bool paired = ((reinterpret_cast<uintptr_t>(px) & 7u) == 0) && (!bout || (reinterpret_cast<uintptr_t>(bout) & 3u) == 0);
  for (int i = beg + threadIdx.x; i < end; i += 256) {
    const int p0 = 2 * i;
    if (!paired) {
      for (int p = p0; p < min(p0 + 2, n_px); ++p) {
        const uint32_t b0 = rgb_bin(__ldg(px + p));
        atomicAdd(&sh[b0], 1u);
        if (bout) bout[p] = (uint16_t)(b0 << 3);
      }
    } else if (p0 + 1 < n_px) {
      const uint2 v = __ldg(reinterpret_cast<const uint2 *>(px + p0));
      const uint32_t b0 = rgb_bin(v.x), b1 = rgb_bin(v.y);
      atomicAdd(&sh[b0], 1u);
      atomicAdd(&sh[b1], 1u);
      if (bout) *reinterpret_cast<uint32_t *>(bout + p0) = (b0 << 3) | (b1 << 19);
    } else {
      const uint32_t b0 = rgb_bin(__ldg(px + p0));
      atomicAdd(&sh[b0], 1u);
      if (bout) bout[p0] = (uint16_t)(b0 << 3);
    }
  }
  __syncthreads();
  uint32_t *out = hist + (size_t)blockIdx.y * 4096;
  if (chunks == 1) {
    for (int i = threadIdx.x; i < 4096; i += 256) out[i] = sh[i];
  } else {
    for (int i = threadIdx.x; i < 4096; i += 256)
      if (sh[i]) atomicAdd(&out[i], sh[i]);
  }
}

// ------------------------------------------------------------------------------------------------
// initTracker — src/camshift.js:198-211.  One CTA per slot: model histogram of the rectangle
// (pixels outside the canvas read as 0,0,0,0 -> bin 0, like getImageData), _searchWindow := rect,
// _trackObj := new TrackObj().  rects == NULL -> take the rectangle from det_pick (device pick).
__global__ void __launch_bounds__(256) k_track_init(const uint8_t *__restrict__ rgba, size_t frame_bytes, int W, int H,
                                                    const int32_t *__restrict__ slots,
                                                    const int32_t *__restrict__ rects, int calc_angles,
                                                    uint32_t *__restrict__ model_hist, TrackState *__restrict__ state,
                                                    int32_t *__restrict__ found, const uint8_t *__restrict__ enable) {
  __shared__ uint32_t sh[4096];
  const int k = blockIdx.x;
  if (enable && !enable[k]) return;            // ht_stream_step: only the streams that just found a face
  const int slot = slots ? slots[k] : k;
  const int rx = rects[4 * k + 0], ry = rects[4 * k + 1], rw = rects[4 * k + 2], rh = rects[4 * k + 3];
  if (rw <= 0 || rh <= 0) {  // no candidate (device pick): the slot becomes uninitialised
    if (threadIdx.x == 0) {
      state[slot].initialised = 0;
      if (found) found[k] = 0;
    }
    return;
  }
  for (int i = threadIdx.x; i < 4096; i += 256) sh[i] = 0;
  __syncthreads();
  const uint32_t *px = reinterpret_cast<const uint32_t *>(rgba + (size_t)k * frame_bytes);
  for (int yy = threadIdx.x >> 5; yy < rh; yy += 8) {
    const int cy = ry + yy;
    for (int xx = threadIdx.x & 31; xx < rw; xx += 32) {
      const int cx = rx + xx;
      uint32_t bin = 0;
      if (cx >= 0 && cx < W && cy >= 0 && cy < H) bin = rgb_bin(__ldg(px + (size_t)cy * W + cx));
      atomicAdd(&sh[bin], 1u);
    }
  }
  __syncthreads();
  uint32_t *out = model_hist + (size_t)slot * 4096;
  for (int i = threadIdx.x; i < 4096; i += 256) out[i] = sh[i];
  if (threadIdx.x == 0) {
    TrackState s;
    s.sx = rx; s.sy = ry; s.sw = rw; s.sh = rh;
    s.tx = s.ty = s.tw = s.th = 0;
    s.angle = 0.0;
    s.calc_angles = calc_angles;
    s.initialised = 1;
    state[slot] = s;
    if (found) found[k] = 1;
  }
}

// facetrackr's VJ->CS hand-off on the device — src/facetrackr.js:157-165 (first max-confidence
// candidate), :97 (confidence > -10), :101-106 (Math.floor of x,y,width,height).
__global__ void k_pick_face(const Rect *__restrict__ det, const int32_t *__restrict__ counts, int K, int n,
                            int32_t *__restrict__ rects) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int c = counts[k];
  int32_t r[4] = {0, 0, 0, 0};
  if (c > 0) {
    const Rect *d = det + (size_t)k * K;
    int best = 0;
    for (int i = 1; i < c; ++i)
      if (d[i].confidence > d[best].confidence) best = i;
    if (d[best].confidence > -10.0) {
      r[0] = (int32_t)floor(d[best].x); r[1] = (int32_t)floor(d[best].y);
      r[2] = (int32_t)floor(d[best].width); r[3] = (int32_t)floor(d[best].height);
    }
  }
  rects[4 * k + 0] = r[0]; rects[4 * k + 1] = r[1]; rects[4 * k + 2] = r[2]; rects[4 * k + 3] = r[3];
}

// ------------------------------------------------------------------------------------------------
// Zero-weight marking of the bin plane.  getWeights (src/camshift.js:314-330) gives a pixel the weight
// min(model[bin] / current[bin], 1): it is exactly +0.0 for every colour bin that does not occur in the model
// histogram, i.e. in the face rectangle of initTracker - the vast majority of a frame's pixels (85-99 % on the bench
// frames; a face has a few dozen to a few hundred of the 4096 bins).  Adding +0.0 to a moment sum never changes it,
// so those pixels can be skipped.  This pass rewrites their plane entries to ZERO (0x8000 = 8 * 4096, the table's
// extra +0.0 entry): k_track then skips every 128-pixel row segment whose entries are all ZERO with one warp vote.
// One read + one write of the u16 plane per frame, worth it when several track() calls follow on the same frame.
constexpr uint32_t BIN_ZERO = 8u * 4096u;          // byte offset of wsm[4096]
constexpr uint32_t BIN_ZERO2 = BIN_ZERO | (BIN_ZERO << 16);
__global__ void __launch_bounds__(256) k_bins_mask(uint16_t *__restrict__ bins, int n_px, const uint32_t *__restrict__ model_hist,
                                                   const int32_t *__restrict__ slots, const TrackState *__restrict__ state,
                                                   int chunks, const uint8_t *__restrict__ enable,
                                                   // cost != NULL: only the streams whose previous launch visited more than
                                                   // min_px256 * 256 pixels (k_track's scheduling history) - the pass over
                                                   // the plane is repaid by streams that sweep large windows many times
                                                   const int32_t *__restrict__ cost, int min_px256) {
  __shared__ uint32_t bm[128];                     // bit b set: model histogram bin b is non-zero
  const int k = blockIdx.y;
  if (enable && !enable[k]) return;
  const int slot = slots ? slots[k] : k;
  if (!state[slot].initialised) return;            // k_track refuses such a slot anyway
  if (cost && cost[2 * slot + 1] < min_px256) return;
  const uint32_t *mh = model_hist + (size_t)slot * 4096;
  if (threadIdx.x < 128) {
    uint32_t w = 0;
#pragma unroll 8
    for (int i = 0; i < 32; ++i) w |= (__ldg(mh + 32 * threadIdx.x + i) != 0u ? 1u : 0u) << i;
    bm[threadIdx.x] = w;
  }
  __syncthreads();
  uint16_t *pl = bins + (size_t)k * n_px;
  auto mask2 = [&](uint32_t v) {                   // two u16 entries (8 * bin each)
    const uint32_t b0 = (v & 0xffffu) >> 3, b1 = v >> 19;
    uint32_t o = v;
    if (b0 < 4096u && !((bm[b0 >> 5] >> (b0 & 31u)) & 1u)) o = (o & 0xffff0000u) | BIN_ZERO;
    if (b1 < 4096u && !((bm[b1 >> 5] >> (b1 & 31u)) & 1u)) o = (o & 0x0000ffffu) | (BIN_ZERO << 16);
    return o;
  };
  const bool vec = ((reinterpret_cast<uintptr_t>(pl) & 15u) == 0);
  const int n_grp = vec ? n_px / 8 : 0;            // groups of 8 entries (16 bytes)
  const int per = (n_grp + chunks - 1) / chunks;
  const int beg = blockIdx.x * per, end = min(n_grp, beg + per);
  for (int g = beg + threadIdx.x; g < end; g += 256) {
    uint4 v = *reinterpret_cast<const uint4 *>(pl + 8 * (size_t)g);
    const uint4 o = make_uint4(mask2(v.x), mask2(v.y), mask2(v.z), mask2(v.w));
    if (o.x != v.x || o.y != v.y || o.z != v.z || o.w != v.w) *reinterpret_cast<uint4 *>(pl + 8 * (size_t)g) = o;
  }
  if (blockIdx.x == 0)                             // tail (and unaligned planes): entry by entry
    for (int p = 8 * n_grp + threadIdx.x; p < n_px; p += 256) {
      const uint32_t b = pl[p] >> 3;
      if (b < 4096u && !((bm[b >> 5] >> (b & 31u)) & 1u)) pl[p] = (uint16_t)BIN_ZERO;
    }
}

// ------------------------------------------------------------------------------------------------
// track() — src/camshift.js:213-312.  One CTA per slot runs getWeights, the <=10 mean-shift
// iterations and the camShift epilogue for n_calls successive track() calls on the same frame.

struct Mom {
  double m00, m10, m01, m11, m20, m02;
};

__device__ __forceinline__ int32_t js_to_int32(double v) {  // ES ToInt32 for |v| < 2^31; NaN/Inf -> 0
  if (!isfinite(v)) return 0;
  return (int32_t)v;  // cvt.rzi: truncation toward zero
}

// true when truncating v could flip under the (tiny) summation-order error of a parallel reduction
__device__ __forceinline__ bool trunc_ambiguous(double v) {
  return isfinite(v) && fabs(v - rint(v)) < 1e-7;
}

// Moments in the reference's exact order (x outer, y inner, one accumulator each) —
// src/camshift.js:90-107.  Used by one thread only when a truncation decision is ambiguous.
__device__ __noinline__ Mom moments_serial(const uint16_t *__restrict__ px, int W, int x, int y, int w, int h,
                                           const double *__restrict__ wsm) {
  Mom m = {0, 0, 0, 0, 0, 0};
  for (int i = x; i < w; ++i) {
    const double vx = (double)(i - x);
    for (int j = y; j < h; ++j) {
      const double val = wsm[px[(size_t)j * W + i] >> 3];
      const double vy = (double)(j - y);
      m.m00 += val;
      m.m01 += vy * val;
      m.m10 += vx * val;
      m.m11 += vx * vy * val;
      m.m02 += vy * vy * val;
      m.m20 += vx * vx * val;
    }
  }
  return m;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}

// One thread-block CLUSTER per slot: TRACK_CLUSTER CTAs split the rows of every window pass and
// combine their partial moments through distributed shared memory.  Mean-shift is a serial chain
// of passes per stream (up to 10 per track() call); spreading one pass over several SMs shortens
// the chain of the streams with large windows, which otherwise set the kernel's duration.  The cluster size is a
// launch-time choice: 2, 4 or 8 CTAs per stream.
constexpr int TRACK_THREADS = 256;   // threads per k_track CTA

// Longest-chain-first launch order.  A stream's mean-shift passes form a serial chain whose length grows with its
// search window, and a launch holds only a few hundred streams at a time, so the streams with the largest windows
// are started first (and may be given a larger cluster): otherwise one of them starting in the last wave sets the
// duration of the whole launch.  area[i] = search-window area of stream i; order = indices by descending area
// (ties by index, so the order is deterministic).
__global__ void k_track_area(const TrackState *__restrict__ state, const int32_t *__restrict__ slots, int n,
                             const int32_t *__restrict__ cost, int32_t *__restrict__ area) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int slot = slots ? slots[i] : i;
  const TrackState *s = state + slot;
  long long a = 0;
  if (s->initialised) {
    // History first: what this stream cost in its previous launch (k_track's leader records {passes, window pixels
    // / 256}) predicts the chain it is about to run far better than its current window does - the windows that end
    // up covering the frame start small.  Units: one pass = 120, one pixel per thread of a 256-thread CTA = 1
    // (3 us vs 0.025 us, tools/track_chain_probe.py).  Streams without history: the window area of a typical
    // 70-pass chain.
    const int passes = cost ? cost[2 * slot] : 0;
    if (passes > 0) a = 120ll * passes + cost[2 * slot + 1];
    else a = 120ll * 70 + 70ll * (((long long)max(s->sw, 0) * (long long)max(s->sh, 0)) >> 8);
  }
  area[i] = (int32_t)min(a, (long long)0x7fffffff);
}
__global__ void k_track_rank(const int32_t *__restrict__ area, int n, int32_t *__restrict__ order) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t a = area[i];
  int rank = 0;
  for (int j = 0; j < n; ++j) {
    const int32_t b = __ldg(area + j);
    rank += (b > a || (b == a && j < i)) ? 1 : 0;
  }
  order[rank] = i;
}

// ld.shared.f64 from a 32-bit shared-window address (indexing the __shared__ array through its generic address
// makes the compiler rebuild the cluster-window base, an S2R, for every access)
__device__ __forceinline__ double lds_f64(uint32_t saddr) {
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(saddr));
  return v;
}

__device__ __forceinline__ void row_partial(const uint16_t *__restrict__ row, const double *__restrict__ wsm, int lane,
                                            int wx, int xbeg, int xend, bool vec4, double &r0, double &r1, double &r2) {
  if (vec4) {
    for (int x4 = xbeg + 4 * lane; x4 < xend; x4 += 128) {
      const uint2 v = __ldg(reinterpret_cast<const uint2 *>(row + x4));
      const uint32_t b[4] = {(v.x & 0xffffu) >> 3, v.x >> 19, (v.y & 0xffffu) >> 3, v.y >> 19};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int x = x4 + i;
        const double val = (x >= wx && x < xend) ? wsm[b[i]] : 0.0;   // +0.0 terms leave the sums unchanged
        const double vx = (double)(x - wx);
        r0 += val;
        r1 += vx * val;
        r2 += (vx * vx) * val;
      }
    }
  } else {
    for (int x = wx + lane; x < xend; x += 32) {
      const double val = wsm[row[x] >> 3];
      const double vx = (double)(x - wx);
      r0 += val;
      r1 += vx * val;
      r2 += (vx * vx) * val;
    }
  }
}

// __launch_bounds__: three resident CTAs per SM (80 registers)
template <int TRACK_CLUSTER>
__global__ void __launch_bounds__(TRACK_THREADS, 3)
k_track(const uint16_t *__restrict__ bins, int W, int H, const int32_t *__restrict__ slots,
        const uint32_t *__restrict__ model_hist, const uint32_t *__restrict__ cur_hist, TrackState *__restrict__ state,
        int n_calls, int32_t *__restrict__ out_objs /* 6 x i32 per frame */, int32_t *__restrict__ out_windows,
        int32_t *__restrict__ err_flag, unsigned long long *__restrict__ stats,
        // order != NULL: the k-th cluster runs stream order[list_off + k] (k_track_rank's order); NULL: stream k
        const int32_t *__restrict__ order, int list_off,
        // optional timeline (HT_TRACK_TRACE=1): per stream {globaltimer at start, at end, SM id, passes}
        unsigned long long *__restrict__ trace, size_t trace_stride,
        // memo != 0: moments are a pure function of (frame, weights, window) and all three are fixed for the calls of
        // one launch, so the leader keeps the moments of the last windows it has seen and re-uses them when
        // mean-shift returns to one of them (a converged stream, or one oscillating between two windows)
        int memo,
        // force_serial != 0 (ht_debug_set_exactness bit 2): every pass takes the strict-order fallback
        int force_serial,
        // per slot {passes, window pixels / 256} of this launch: the scheduling key of the next one (k_track_area)
        int32_t *__restrict__ cost,
        // enable != NULL (ht_stream_step): streams with enable[k] == 0 are not in tracking mode and are skipped
        const uint8_t *__restrict__ enable) {
  namespace cg = cooperative_groups;
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ double wsm[4096 + 1];   // [4096] = +0.0: the weight of pixels outside the window
  constexpr int NW = TRACK_THREADS / 32;   // warps per CTA
  __shared__ double red[NW][6];
  // Every CTA of the cluster keeps its OWN copy of the reference's loop state and runs the scalar mean-shift step
  // redundantly (same inputs, same operations -> bit-identical windows), so a pass needs ONE cluster barrier - the
  // exchange of the partial moments - instead of two (round 1: partials to rank 0, barrier, rank 0 publishes the
  // next window, barrier).  cpart is double-buffered by pass parity: a CTA that is already exchanging pass p+1
  // cannot overwrite what a slower CTA still reads for pass p.
  __shared__ double cpart[2][TRACK_CLUSTER][6];  // partial moments of every CTA of the cluster (written remotely)
  __shared__ int win[4];                          // wadx, wady, wadw, wadh of the next pass
  __shared__ int ctrl;                            // 0 = run another pass over win[], 1 = this stream is finished
  constexpr int MEMO_N = 8;
  struct MemoEnt { int w[4]; int exact; int valid; Mom m; };
  __shared__ MemoEnt memo_tab[MEMO_N];            // thread 0 of every CTA
  __shared__ int memo_next;
  __shared__ unsigned long long st_memo_sh;
  const int crank = (int)cluster.block_rank();
  int k = blockIdx.x / TRACK_CLUSTER;
  if (order) k = order[list_off + k];
  if (enable && !enable[k]) return;               // uniform over the cluster, before any cluster barrier
  const int slot = slots ? slots[k] : k;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool leader = (crank == 0 && tid == 0);   // the one thread that writes results, state and statistics
  const bool stepper = (tid == 0);                 // thread 0 of EVERY CTA runs the mean-shift step
  // The reference's loop state lives in shared memory: only the leader thread touches it after this point, and
  // keeping it out of registers leaves them to the pipelined pass loop.
  struct Lead { TrackState s; unsigned long long st_pass, st_serial, st_px; int call, it, prevx, prevy; };
  __shared__ Lead lead_sh;
  if (tid == 0) {
    lead_sh.s = state[slot];
    lead_sh.st_pass = lead_sh.st_serial = lead_sh.st_px = 0;
    lead_sh.call = 0; lead_sh.it = 0; lead_sh.prevx = lead_sh.s.sx; lead_sh.prevy = lead_sh.s.sy;
    memo_next = 0; st_memo_sh = 0;
    for (int i = 0; i < MEMO_N; ++i) memo_tab[i].valid = 0;
  }
  __syncthreads();
  TrackState &s = lead_sh.s;
  if (trace && leader) {
    unsigned long long t; unsigned smid;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    trace[4 * (size_t)k] = t; trace[4 * (size_t)k + 2] = smid;
  }
  if (!s.initialised) {   // uniform over the cluster
    if (leader) {
      atomicOr(err_flag, 1);
      int32_t *o = out_objs + 6 * (size_t)k;
      o[0] = o[1] = o[2] = o[3] = o[4] = o[5] = 0;  // TrackObj() defaults
      if (out_windows) { int32_t *w4 = out_windows + 4 * (size_t)k; w4[0] = w4[1] = w4[2] = w4[3] = 0; }
    }
    return;
  }
  // getWeights — src/camshift.js:314-330 (every CTA keeps its own copy)
  {
    const uint32_t *mh = model_hist + (size_t)slot * 4096, *ch = cur_hist + (size_t)k * 4096;
    for (int i = tid; i < 4096; i += TRACK_THREADS) {
      const uint32_t c = ch[i], m = mh[i];
      double p = 0.0;
      // (a bin absent from the model gives 0 / c = +0.0: no division for it - that is nearly all of the 4096 bins)
      if (c != 0 && m != 0) p = fmin((double)m / (double)c, 1.0);
      wsm[i] = p;
    }
    if (tid == 0) wsm[4096] = 0.0;
  }
  const uint16_t *px = bins + (size_t)k * W * H;   // 12-bit colour bin of every pixel of this slot's frame (k_hist)
  const bool vec4 = (W & 3) == 0;
  int parity = 0;

  // leader-only bookkeeping of the reference's loops (src/camshift.js:213-312)
  unsigned long long &st_pass = lead_sh.st_pass, &st_serial = lead_sh.st_serial, &st_px = lead_sh.st_px;
  int &call = lead_sh.call, &it = lead_sh.it, &prevx = lead_sh.prevx, &prevy = lead_sh.prevy;
  auto publish = [&](int done) {   // stepper: next window (or the finish flag) for this CTA
    const int w0 = max(s.sx, 0), w1 = max(s.sy, 0);                // :286-289
    const int w2 = min(w0 + s.sw, W), w3 = min(w1 + s.sh, H);
    win[0] = w0; win[1] = w1; win[2] = w2; win[3] = w3;
    ctrl = done;
  };
  auto start_call = [&]() {        // leader: returns true when all calls are done
    if (call >= n_calls) return true;
    it = 0; prevx = s.sx; prevy = s.sy;                            // :280-281
    return false;
  };
  if (TRACK_CLUSTER > 1) cluster.sync();  // every CTA is resident before the first remote access
  if (stepper) publish(start_call() ? 1 : 0);
  __syncthreads();

#ifndef HT_TRACK_PASSTRACE
#define HT_TRACK_PASSTRACE 0   // 1 (profiling build): the leader thread accumulates the clock cycles of each phase of a pass
#endif
#if HT_TRACK_PASSTRACE
  long long pt_acc[5] = {0, 0, 0, 0, 0};
  long long pt_t = 0;
#define HT_PT_MARK(i) do { if (trace && leader) { const long long now_ = clock64(); pt_acc[i] += now_ - pt_t; pt_t = now_; } } while (0)
#else
#define HT_PT_MARK(i) do { } while (0)
#endif
  constexpr int ROW_STRIDE = NW * TRACK_CLUSTER;
  while (!ctrl) {
    const int wx = win[0], wy = win[1], ww = win[2] - win[0], wh = win[3] - win[1];
#if HT_TRACK_PASSTRACE
    if (trace && leader) pt_t = clock64();
#endif
    // Each lane reads 4 adjacent pixels (one 8 B load of 4 colour bins) of 4 rows per step.  Rows are assigned by
    // ABSOLUTE frame row (a CTA keeps hitting its own L1 lines when the window shifts between passes).  The steps of
    // a pass (row group x 128-pixel column block) are software-pipelined: the four loads of step t+1 are issued
    // before the arithmetic of step t, so a pass exposes one L2 latency instead of one per step (a pass is a short
    // serial chain: 3-25 steps per thread).  Per step and row: r0 = sum v, r1 = sum vx v; the vy factors are
    // applied once per row and step.
    double a00 = 0, a10 = 0, a01 = 0, a11 = 0, a20 = 0, a02 = 0;
    const int xbeg = wx & ~3, xend = wx + ww;
    const int mine = crank * NW + warp;                          // rows with (wy+yy) % ROW_STRIDE == mine
    const int yy0 = (mine - (wy % ROW_STRIDE) + ROW_STRIDE) % ROW_STRIDE;
    if (vec4) {
      const int n_x = (xend - xbeg + 127) >> 7;
      const int n_rg = (yy0 < wh) ? (wh - yy0 + 4 * ROW_STRIDE - 1) / (4 * ROW_STRIDE) : 0;
      const int total = n_rg * n_x;
      const uint16_t *col = px + (size_t)wy * W + xbeg + 4 * lane;
      const uint32_t wsm_base = (uint32_t)__cvta_generic_to_shared(wsm);
      constexpr uint32_t ZERO_W = 8u * 4096u;   // byte offset of wsm[4096]
      auto issue = [&](int rg, int xi, uint2 (&v)[4]) {
        const int x4 = xbeg + 4 * lane + 128 * xi;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int y = yy0 + (4 * rg + j) * ROW_STRIDE;
          v[j] = (y < wh && x4 < xend) ? __ldg(reinterpret_cast<const uint2 *>(col + (size_t)y * W + 128 * xi))
                                       : make_uint2(ZERO_W | (ZERO_W << 16), ZERO_W | (ZERO_W << 16));
        }
      };
      auto consume = [&](int rg, int xi, const uint2 (&v)[4]) {
        const int x4 = xbeg + 4 * lane + 128 * xi;
        double vx[4], vx2[4];
        bool in[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int x = x4 + i;
          in[i] = (x >= wx && x < xend);
          vx[i] = (double)(x - wx);
          vx2[i] = vx[i] * vx[i];
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          // a 128-pixel row segment whose entries are all ZERO (k_bins_mask: colours absent from the model; rows below
          // the window) adds +0.0 to every sum: skip it with one vote (uniform over the warp)
          if (!__any_sync(0xffffffffu, v[j].x != BIN_ZERO2 || v[j].y != BIN_ZERO2)) continue;
          const int y = yy0 + (4 * rg + j) * ROW_STRIDE;
          // table offsets (the plane holds 8 * bin); rows below the window were "loaded" as ZERO_W by issue()
          const uint32_t b[4] = {v[j].x & 0xffffu, v[j].x >> 16, v[j].y & 0xffffu, v[j].y >> 16};
          double r0 = 0.0, r1 = 0.0, r2 = 0.0;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            // pixels outside the window read the extra table entry wsm[4096] == +0.0, which leaves the sums unchanged
            const double val = lds_f64(wsm_base + (in[i] ? b[i] : ZERO_W));
            r0 += val;
            r1 = fma(vx[i], val, r1);     // fused: this fast path is validated by trunc_ambiguous, the strict
            r2 = fma(vx2[i], val, r2);    // reference order (separate multiply and add) is moments_serial
          }
          const double vy = (double)y;
          a00 += r0; a10 += r1; a20 += r2;
          a01 = fma(vy, r0, a01); a11 = fma(vy, r1, a11); a02 = fma(vy * vy, r0, a02);
        }
      };
      uint2 va[4], vb[4];
      int rg = 0, xi = 0;
      if (total > 0) issue(0, 0, va);
      for (int t = 0; t < total; t += 2) {
        int rg1 = rg, xi1 = xi + 1;
        if (xi1 == n_x) { xi1 = 0; ++rg1; }
        if (t + 1 < total) issue(rg1, xi1, vb);
        consume(rg, xi, va);
        int rg2 = rg1, xi2 = xi1 + 1;
        if (xi2 == n_x) { xi2 = 0; ++rg2; }
        if (t + 2 < total) issue(rg2, xi2, va);
        if (t + 1 < total) consume(rg1, xi1, vb);
        rg = rg2; xi = xi2;
      }
    } else {
      for (int yy = yy0; yy < wh; yy += 4 * ROW_STRIDE) {
        double r[4][3];
#pragma unroll
        for (int j = 0; j < 4; ++j) r[j][0] = r[j][1] = r[j][2] = 0.0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int y = yy + j * ROW_STRIDE;
          if (y < wh) row_partial(px + (size_t)(wy + y) * W, wsm, lane, wx, xbeg, xend, false, r[j][0], r[j][1], r[j][2]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const double vy = (double)(yy + j * ROW_STRIDE);
          a00 += r[j][0]; a10 += r[j][1]; a20 += r[j][2];
          a01 += vy * r[j][0]; a11 += vy * r[j][1]; a02 += (vy * vy) * r[j][0];
        }
      }
    }
    HT_PT_MARK(0);                     // pixel loop of this thread (loads, lookups, FMAs)
    a00 = warp_sum(a00); a10 = warp_sum(a10); a01 = warp_sum(a01);
    a11 = warp_sum(a11); a20 = warp_sum(a20); a02 = warp_sum(a02);
    if (lane == 0) {
      red[warp][0] = a00; red[warp][1] = a10; red[warp][2] = a01;
      red[warp][3] = a11; red[warp][4] = a20; red[warp][5] = a02;
    }
    __syncthreads();
    HT_PT_MARK(1);                     // warp sums + wait for the CTA's slowest warp
    if (tid < 6 * TRACK_CLUSTER) {   // fixed-order sums (run-to-run deterministic), one copy into every CTA
      const int q = tid % 6, r = tid / 6;
      double t = 0;
      for (int w8 = 0; w8 < NW; ++w8) t += red[w8][q];
      cluster.map_shared_rank(&cpart[0][0][0], r)[(parity * TRACK_CLUSTER + crank) * 6 + q] = t;
    }
    if (TRACK_CLUSTER > 1) cluster.sync(); else __syncthreads();
    HT_PT_MARK(2);                     // cross-warp sum, remote stores, cluster barrier (wait for the slowest CTA)
    if (stepper) {
      Mom m = {0, 0, 0, 0, 0, 0};
      for (int r = 0; r < TRACK_CLUSTER; ++r) {
        m.m00 += cpart[parity][r][0]; m.m10 += cpart[parity][r][1]; m.m01 += cpart[parity][r][2];
        m.m11 += cpart[parity][r][3]; m.m20 += cpart[parity][r][4]; m.m02 += cpart[parity][r][5];
      }
      bool exact = false;          // m is in the reference's strict summation order (moments_serial)
      bool fresh = true;           // m was computed by this pass (false: taken from the memo)
      int cw0 = win[0], cw1 = win[1], cw2 = win[2], cw3 = win[3];   // the window m belongs to
      ++st_pass;
      st_px += (unsigned long long)(max(ww, 0)) * (unsigned long long)(max(wh, 0));
      for (;;) {
        double inv = 1.0 / m.m00;                                    // :109-111
        double vxf = m.m10 * inv - s.sw / 2.0, vyf = m.m01 * inv - s.sh / 2.0;
        if (!exact && (force_serial || trunc_ambiguous(vxf) || trunc_ambiguous(vyf))) {
          m = moments_serial(px, W, cw0, cw1, cw2, cw3, wsm);
          exact = true;
          ++st_serial;
          inv = 1.0 / m.m00;
          vxf = m.m10 * inv - s.sw / 2.0;
          vyf = m.m01 * inv - s.sh / 2.0;
        }
        s.sx += js_to_int32(vxf);                                    // :295-296
        s.sy += js_to_int32(vyf);
        const bool conv = (s.sx == prevx && s.sy == prevy);         // :299
        bool done = false;
        if (conv || it == 9) {
          // final moments (second == true) are those of this window.  camShift epilogue - src/camshift.js:230-258 -
          // computed once; when the moments are in the parallel order and a `<< 2` truncation (or, with angles, the sign
          // of b) is not safe, the strict moments replace them and the epilogue is recomputed from those.
          s.sx = max(0, min(s.sx, W));                                   // :308-309
          s.sy = max(0, min(s.sy, H));
          for (;;) {
            const double invM00 = 1.0 / m.m00;
            const double xc = m.m10 * invM00, yc = m.m01 * invM00;
            const double mu20 = m.m20 - m.m10 * xc, mu02 = m.m02 - m.m01 * yc, mu11 = m.m11 - m.m01 * xc;
            const double a = mu20 * invM00, c = mu02 * invM00;
            double l1, l2, ang = 3.141592653589793 / 2;
            bool amb = false;
            if (s.calc_angles) {
              const double b = mu11 * invM00;
              const double d = a + c;
              const double e = sqrt((4 * b * b) + ((a - c) * (a - c)));
              l1 = sqrt((d - e) * 0.5); l2 = sqrt((d + e) * 0.5);
              // `if (ang < 0) ang += PI` (src/camshift.js:244) follows the SIGN of b = mu11 / m00: for a symmetric blob
              // b is rounding residue and the parallel summation order may flip it (angle off by PI, far outside
              // the 1e-4 tolerance) - take the strict order whenever b is not clearly away from 0
              amb = fabs(b) <= 1e-9 * (fabs(a) + fabs(c) + 1.0);
              if (exact || !(amb || trunc_ambiguous(l1) || trunc_ambiguous(l2))) {
                ang = atan2(2 * b, a - c + e);
                if (ang < 0) ang = ang + 3.141592653589793;
              }
            } else {
              l1 = sqrt(a); l2 = sqrt(c);
            }
            if (!exact && (amb || trunc_ambiguous(l1) || trunc_ambiguous(l2))) {
              m = moments_serial(px, W, cw0, cw1, cw2, cw3, wsm); exact = true; ++st_serial;
              continue;
            }
            s.tw = (int32_t)((uint32_t)js_to_int32(l1) << 2);
            s.th = (int32_t)((uint32_t)js_to_int32(l2) << 2);
            s.angle = ang;
            break;
          }
          s.tx = (int32_t)floor(fmax(0.0, fmin(s.sx + s.sw / 2.0, (double)W)));   // :253-254
          s.ty = (int32_t)floor(fmax(0.0, fmin(s.sy + s.sh / 2.0, (double)H)));
          s.sw = (int32_t)floor(1.1 * s.tw);                             // :257-258
          s.sh = (int32_t)floor(1.1 * s.th);
          ++call;
          done = start_call();
        } else {
          prevx = s.sx;
          prevy = s.sy;
          ++it;
        }
        if (memo && fresh) {        // remember this window's moments (the strict ones if they had to be computed)
          MemoEnt &e = memo_tab[memo_next];
          memo_next = (memo_next + 1) % MEMO_N;
          e.w[0] = cw0; e.w[1] = cw1; e.w[2] = cw2; e.w[3] = cw3;
          e.exact = exact ? 1 : 0; e.m = m; e.valid = 1;
        }
        if (done) { publish(1); break; }
        if (memo) {                 // the next window (src/camshift.js:286-289) may be one whose moments are known
          const int n0 = max(s.sx, 0), n1 = max(s.sy, 0);
          const int n2 = min(n0 + s.sw, W), n3 = min(n1 + s.sh, H);
          int hit = -1;
          for (int i = 0; i < MEMO_N; ++i) {
            const MemoEnt &e = memo_tab[i];
            if (e.valid && e.w[0] == n0 && e.w[1] == n1 && e.w[2] == n2 && e.w[3] == n3) hit = i;
          }
          if (hit >= 0) {
            m = memo_tab[hit].m; exact = memo_tab[hit].exact != 0; fresh = false;
            cw0 = n0; cw1 = n1; cw2 = n2; cw3 = n3;
            ++st_memo_sh;
            continue;
          }
        }
        publish(0);
        break;
      }
    }
    HT_PT_MARK(3);                     // scalar mean-shift step
    parity ^= 1;
    __syncthreads();
    HT_PT_MARK(4);                     // CTA barrier that publishes the next window
  }
  if (leader) {
    if (cost) {
      cost[2 * slot] = (int32_t)min(st_pass, 0x7fffffffull);
      cost[2 * slot + 1] = (int32_t)min(st_px >> 8, 0x7fffffffull);
    }
    if (stats) {
      atomicAdd(&stats[0], st_pass); atomicAdd(&stats[1], st_serial);
      atomicAdd(&stats[2], st_px); atomicAdd(&stats[3], (unsigned long long)call);
      atomicAdd(&stats[4], st_memo_sh);
    }
    state[slot] = s;
    if (trace) {
      unsigned long long t;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
      trace[4 * (size_t)k + 1] = t; trace[4 * (size_t)k + 3] = st_pass;
#if HT_TRACK_PASSTRACE
      // phase totals (SM clock cycles) behind the per-stream records: [max_frames x 4][max_frames x 8]
      for (int i = 0; i < 5; ++i) trace[trace_stride + 8 * (size_t)k + i] = (unsigned long long)pt_acc[i];
#endif
    }
    int32_t *o = out_objs + 6 * (size_t)k;
    o[0] = s.tx; o[1] = s.ty; o[2] = s.tw; o[3] = s.th;
    *reinterpret_cast<double *>(o + 4) = s.angle;
    if (out_windows) {
      int32_t *w4 = out_windows + 4 * (size_t)k;
      w4[0] = s.sx; w4[1] = s.sy; w4[2] = s.sw; w4[3] = s.sh;
    }
  }
  if (TRACK_CLUSTER > 1) cluster.sync();  // no CTA may exit while another one can still address its shared memory
}

// ------------------------------------------------------------------------------------------------
// facetrackr's per-frame state machine on the device (src/facetrackr.js:67-126 with whitebalancing off, plus the
// lost-face rule of src/main.js:230-244) for n independent streams: ht_stream_step.
//   mode[k] : 0 = "VJ" (detect on this frame), 1 = "CS" (camshift on this frame)
// k_stream_plan runs before the frame's kernels and turns the modes into the masks they take; k_stream_update runs
// after them, writes the frame's event record and applies the transitions.
struct StreamEvent {       // == ht_stream_event (include/headtrackr_b200.h)
  int32_t detection;       // 1 = "VJ", 2 = "CS"  (facetrackr TrackObj.detection, src/facetrackr.js:233-241)
  int32_t status;          // bit 0: VJ found a face, the stream switches to CS (src/facetrackr.js:97-108)
                           // bit 1: CS lost the face (width or height 0), the stream re-detects (src/main.js:230-244)
  double x, y, width, height, angle, confidence;
};

// ------------------------------------------------------------------------------------------------
// What src/main.js does with a "CS" result after facetrackr: "found" status, Smoother (src/smoother.js:25-87),
// the wait for a stable head diagonal (src/main.js:262-281) and headposition.Tracker (src/headposition.js:35-191),
// as a per-stream epilogue of the state machine - one `headtrackingEvent {x, y, z}` record per stream and frame
// (SURVEY.md 8f-3).  Scalar fp64 code, operation for operation as the JavaScript (the library is built with
// -fmad=false); only atan / tan come from CUDA's libm instead of V8's (<= 2 ulp).
struct HeadParams {            // == ht_head_params (include/headtrackr_b200.h)
  int32_t smoothing;           // src/main.js:39   (default 1)
  int32_t head_position;       // src/main.js:55   (default 1)
  int32_t edgecorrection;      // src/headposition.js:44-48 (default 1)
  int32_t pad_;
  double alpha;                // Smoother(0.35, ...)            src/main.js:163
  double fov_deg;              // params.fov; <= 0: estimate it  src/main.js:283-288
  double camera_offset;        // params.cameraOffset (11.5)     src/main.js:53
  double distance_to_screen;   // 60                             src/headposition.js:75-79
  // constants of the 16 x 19 cm head model, filled by the library with the host's libm (src/headposition.js:53-63)
  double sin_hsa, cos_hsa, tan_hsa, head_diag_cm;
};
struct HeadState {
  int32_t face_found, sm_init, n_diag, hp_init, first_run, pad_;
  double sp[5];                // Smoother state: x, y, z, width, height (sp2 IS sp: src/smoother.js:28)
  double diag[6];              // headDiagonal
  double fov_saved_deg;        // `fov` of src/main.js:59,288
  double tan_fov_width, head_diag_cam;   // headposition.Tracker
};
struct HeadEvent {             // == ht_head_event
  int32_t valid;               // 1: a headtrackingEvent was dispatched on this frame
  int32_t status;              // bit 0: headtrackrStatus "found" on this frame (src/main.js:246-249)
  double x, y, z;              // src/headposition.js:183-188
  double fx, fy, fwidth, fheight;   // the (smoothed) face object the position was computed from
};

__host__ __device__ inline double js_nan() {
#ifdef __CUDA_ARCH__
  return __longlong_as_double(0x7ff8000000000000ll);
#else
  return std::numeric_limits<double>::quiet_NaN();
#endif
}

__host__ __device__ inline void head_new_state(HeadState &s) {
  s.face_found = s.sm_init = s.n_diag = s.hp_init = 0;
  s.first_run = 1; s.pad_ = 0;
  for (int i = 0; i < 5; ++i) s.sp[i] = 0.0;
  for (int i = 0; i < 6; ++i) s.diag[i] = 0.0;
  s.fov_saved_deg = 0.0; s.tan_fov_width = 0.0; s.head_diag_cam = 0.0;
}

// one frame of one stream: (x, y, w, h) = the CS TrackObj, lost = width or height 0
__host__ __device__ inline void head_step(HeadState &s, const HeadParams &p, bool is_cs, double x, double y, double w, double h,
                                          bool lost, double camw, double camh, HeadEvent &out) {
  const double PI = 3.141592653589793;
  out.valid = 0; out.status = 0; out.x = out.y = out.z = 0.0; out.fx = out.fy = out.fwidth = out.fheight = 0.0;
  if (!is_cs) return;
  if (lost) {                                  // src/main.js:230-244: new facetrackr, faceFound = false, headposition = undefined
    s.face_found = 0; s.hp_init = 0;
    return;
  }
  if (!s.face_found) { out.status |= 1; s.face_found = 1; }          // :246-249
  if (p.smoothing) {                                                  // :255-261
    const double nan = js_nan();                 // faceObj.z is undefined (src/main.js:259) -> NaN
    if (!s.sm_init) { s.sm_init = 1; s.sp[0] = x; s.sp[1] = y; s.sp[2] = nan; s.sp[3] = w; s.sp[4] = h; }
    const double pos[5] = {x, y, nan, w, h};
    const double a = p.alpha;
    for (int i = 0; i < 5; ++i) {                                     // src/smoother.js:39-42 with sp2 === sp
      s.sp[i] = a * pos[i] + (1 - a) * s.sp[i];
      s.sp[i] = a * s.sp[i] + (1 - a) * s.sp[i];
    }
    // predict(0): step = 0, ratio = (alpha * 0) / (1 - alpha), a = 2 + ratio, b = 1 + ratio (src/smoother.js:77-84)
    const double ratio = (a * 0.0) / (1 - a), A = 2 + ratio, B = 1 + ratio;
    x = A * s.sp[0] - B * s.sp[0]; y = A * s.sp[1] - B * s.sp[1];
    w = A * s.sp[3] - B * s.sp[3]; h = A * s.sp[4] - B * s.sp[4];
  }
  out.fx = x; out.fy = y; out.fwidth = w; out.fheight = h;
  if (!p.head_position) return;
  bool track_now = s.hp_init != 0;
  if (!s.hp_init) {                                                   // src/main.js:264-294
    bool stable = false;
    const double headdiag = sqrt(w * w + h * h);
    if (s.n_diag < 6) s.diag[s.n_diag++] = headdiag;
    else {
      for (int i = 0; i < 5; ++i) s.diag[i] = s.diag[i + 1];
      s.diag[5] = headdiag;
      double mx = s.diag[0], mn = s.diag[0];
      bool any_nan = false;
      for (int i = 0; i < 6; ++i) { any_nan = any_nan || (s.diag[i] != s.diag[i]); mx = s.diag[i] > mx ? s.diag[i] : mx; mn = s.diag[i] < mn ? s.diag[i] : mn; }
      if (!any_nan && (mx - mn) < 5) stable = true;                   // Math.max/min are NaN if any element is
    }
    if (stable) {                                                     // new headposition.Tracker(faceObj, W, H, {...})
      s.head_diag_cam = sqrt((w * w) + (h * h));                      // src/headposition.js:66-68
      double fov_width;
      if (s.first_run) {
        if (!(p.fov_deg > 0.0)) {                                     // :69-84
          const double head_width_cam = p.sin_hsa * s.head_diag_cam;
          const double camwidth_at_default_face_cm = (camw / head_width_cam) * 16;
          fov_width = atan((camwidth_at_default_face_cm / 2) / p.distance_to_screen) * 2;
        } else {
          fov_width = p.fov_deg * PI / 180;
        }
        s.fov_saved_deg = fov_width * 180 / PI;                       // getFOV(), src/main.js:288
        s.first_run = 0;
      } else {
        fov_width = s.fov_saved_deg * PI / 180;                       // {fov : fov}, src/main.js:291
      }
      s.tan_fov_width = 2 * tan(fov_width / 2);                       // src/headposition.js:87
      s.hp_init = 1;
      track_now = true;
    }
  }
  if (!track_now) return;
  // headposition.Tracker.track — src/headposition.js:91-191
  double fx = x, fy = y, hdc = s.head_diag_cam;
  const double sin_hsa = p.sin_hsa, cos_hsa = p.cos_hsa, tan_hsa = p.tan_hsa;
  if (p.edgecorrection) {
    const double margin = 11;
    const double leftDistance = fx - (w / 2), rightDistance = camw - (fx + (w / 2));
    const double topDistance = fy - (h / 2), bottomDistance = camh - (fy + (h / 2));
    const bool onVerticalEdge = (leftDistance < margin || rightDistance < margin);
    const bool onHorizontalEdge = (topDistance < margin || bottomDistance < margin);
    if (onHorizontalEdge) {
      if (onVerticalEdge) {                                           // corner: keep the previous diagonal
        if (leftDistance < margin) fx = w - (hdc * sin_hsa / 2); else fx = fx - (w / 2) + (hdc * sin_hsa / 2);
        if (topDistance < margin) fy = h - (hdc * cos_hsa / 2); else fy = fy - (h / 2) + (hdc * cos_hsa / 2);
      } else if (topDistance < margin) {
        const double ow = topDistance / margin, ew = (margin - topDistance) / margin;
        fy = h - (ow * (h / 2) + ew * ((w / tan_hsa) / 2));
        hdc = ew * (w / sin_hsa) + ow * (sqrt((w * w) + (h * h)));
      } else {
        const double ow = bottomDistance / margin, ew = (margin - bottomDistance) / margin;
        fy = fy - (h / 2) + (ow * (h / 2) + ew * ((w / tan_hsa) / 2));
        hdc = ew * (w / sin_hsa) + ow * (sqrt((w * w) + (h * h)));
      }
    } else if (onVerticalEdge) {
      if (leftDistance < margin) {
        const double ow = leftDistance / margin, ew = (margin - leftDistance) / margin;
        hdc = ew * (h / cos_hsa) + ow * (sqrt((w * w) + (h * h)));
        fx = w - (ow * (w / 2) + (ew) * (h * tan_hsa / 2));
      } else {
        const double ow = rightDistance / margin, ew = (margin - rightDistance) / margin;
        hdc = ew * (h / cos_hsa) + ow * (sqrt((w * w) + (h * h)));
        fx = fx - (w / 2) + (ow * (w / 2) + ew * (h * tan_hsa / 2));
      }
    } else {
      hdc = sqrt((w * w) + (h * h));
    }
  } else {
    hdc = sqrt((w * w) + (h * h));
  }
  s.head_diag_cam = hdc;
  const double z = (p.head_diag_cm * camw) / (s.tan_fov_width * hdc);              // :165
  const double hx = -((fx / camw) - 0.5) * z * s.tan_fov_width;                    // :170
  double hy = -((fy / camh) - 0.5) * z * s.tan_fov_width * (camh / camw);
  hy = hy + p.camera_offset;                                                      // :175-180
  out.valid = 1; out.x = hx; out.y = hy; out.z = z;
}

__global__ void k_stream_plan(const int32_t *__restrict__ mode, int n, uint8_t *__restrict__ vj_quad_mask,
                              uint8_t *__restrict__ cs_enable, uint8_t *__restrict__ init_enable) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  cs_enable[k] = mode[k] == 1 ? 1 : 0;
  init_enable[k] = 0;
  if ((k & 3) == 0) {
    unsigned m = 0;
    for (int f = 0; f < 4 && k + f < n; ++f) m |= (mode[k + f] == 0 ? 1u : 0u) << f;
    vj_quad_mask[k >> 2] = (uint8_t)m;
  }
}

__global__ void k_stream_update(int32_t *__restrict__ mode, int n, const Rect *__restrict__ det,
                                const int32_t *__restrict__ counts, int K, const int32_t *__restrict__ objs,
                                int32_t *__restrict__ rects, uint8_t *__restrict__ init_enable,
                                StreamEvent *__restrict__ events,
                                // optional head-position epilogue (ht_stream_head_config): per-stream state, parameters,
                                // one HeadEvent per stream; camw / camh = the canvas size
                                HeadState *__restrict__ head_state, const HeadParams *__restrict__ head_params,
                                HeadEvent *__restrict__ head_events, int camw, int camh) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  StreamEvent e;
  e.status = 0;
  e.x = e.y = e.width = e.height = e.angle = 0.0;     // new TrackObj(), src/facetrackr.js:233-241
  e.confidence = -10000.0;
  if (mode[k] == 0) {                                  // doVJDetection, src/facetrackr.js:137-175
    e.detection = 1;
    const int c = counts[k];
    if (c > 0) {
      const Rect *d = det + (size_t)k * K;
      int best = 0;
      for (int i = 1; i < c; ++i)
        if (d[i].confidence > d[best].confidence) best = i;   // first maximum, :161-165
      e.x = d[best].x; e.y = d[best].y; e.width = d[best].width; e.height = d[best].height;
      e.confidence = d[best].confidence;
    }
    if (e.confidence > -10.0) {                        // :97: switch to camshift, initTracker on THIS frame
      rects[4 * k + 0] = (int32_t)floor(e.x); rects[4 * k + 1] = (int32_t)floor(e.y);
      rects[4 * k + 2] = (int32_t)floor(e.width); rects[4 * k + 3] = (int32_t)floor(e.height);
      init_enable[k] = 1;
      mode[k] = 1;
      e.status |= 1;
    }
  } else {                                             // doCSDetection, src/facetrackr.js:178-209
    e.detection = 2;
    const int32_t *o = objs + 6 * (size_t)k;
    e.x = o[0]; e.y = o[1]; e.width = o[2]; e.height = o[3];
    e.angle = *reinterpret_cast<const double *>(o + 4);
    e.confidence = 1.0;
    if (o[2] == 0 || o[3] == 0) {                      // src/main.js:230: lost -> a fresh facetrackr without whitebalancing
      mode[k] = 0;
      e.status |= 2;
    }
  }
  events[k] = e;
  if (head_state) {
    HeadState hs = head_state[k];
    HeadEvent he;
    head_step(hs, *head_params, e.detection == 2, e.x, e.y, e.width, e.height, (e.status & 2) != 0, (double)camw, (double)camh, he);
    head_state[k] = hs;
    if (head_events) head_events[k] = he;
  }
}

// getBackProjectionImg — src/camshift.js:177-196 (debug path)
__global__ void k_backproj(const uint8_t *__restrict__ rgba, int n_px, const uint32_t *__restrict__ mh,
                           const uint32_t *__restrict__ ch, uint8_t *__restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_px) return;
  const uint32_t bin = rgb_bin(reinterpret_cast<const uint32_t *>(rgba)[i]);
  const uint32_t c = ch[bin];
  double p = 0.0;
  if (c != 0) p = fmin((double)mh[bin] / (double)c, 1.0);
  const uint32_t v = (uint32_t)floor(255 * p);
  reinterpret_cast<uint32_t *>(out)[i] = v | (v << 8) | (v << 16) | 0xff000000u;
}

// ------------------------------------------------------------------------------------------------
// getWhitebalance — src/whitebalance.js:17-26.  The reference sums bytes in fp64; the sums are
// exact integers, so integer accumulation in any order is bit-identical.
__global__ void __launch_bounds__(256) k_wb_sums(const uint8_t *__restrict__ rgba, size_t frame_bytes, int n_px,
                                                 unsigned long long *__restrict__ sums, int chunks) {
  const uint32_t *px = reinterpret_cast<const uint32_t *>(rgba + (size_t)blockIdx.y * frame_bytes);
  const int per = (n_px + chunks - 1) / chunks;
  const int beg = blockIdx.x * per, end = min(n_px, beg + per);
  unsigned long long r = 0, g = 0, b = 0;
  for (int i = beg + threadIdx.x; i < end; i += 256) {
    const uint32_t p = __ldg(px + i);
    r += p & 0xffu; g += (p >> 8) & 0xffu; b += (p >> 16) & 0xffu;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    r += __shfl_down_sync(0xffffffffu, r, o);
    g += __shfl_down_sync(0xffffffffu, g, o);
    b += __shfl_down_sync(0xffffffffu, b, o);
  }
  if ((threadIdx.x & 31) == 0) {
    unsigned long long *s = sums + 3 * (size_t)blockIdx.y;
    atomicAdd(&s[0], r); atomicAdd(&s[1], g); atomicAdd(&s[2], b);
  }
}

__global__ void k_wb_final(const unsigned long long *__restrict__ sums, int n, int n_px, double *__restrict__ out) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const double sz = (double)n_px;
  const double avgr = (double)sums[3 * k] / sz, avgg = (double)sums[3 * k + 1] / sz, avgb = (double)sums[3 * k + 2] / sz;
  out[k] = (avgr + avgg + avgb) / 3;  // src/whitebalance.js:23-26
}

}  // namespace ht
