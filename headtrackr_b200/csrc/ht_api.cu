// ht_api.cu — host side of libheadtrackr_b200.so: the C ABI declared in include/headtrackr_b200.h,
// the pyramid/tile planner, and the kernel launches.  sm_100a only; there is no CPU fallback.
#include "../../include/headtrackr_b200.h"

#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <tuple>
#include <vector>

#include "ht_common.cuh"
#include "ht_detect.cuh"
#include "ht_track.cuh"

using namespace ht;

static_assert(sizeof(ht_rect) == sizeof(Rect), "ht_rect layout");
static_assert(sizeof(ht_rect) == 48, "ht_rect is 48 bytes");
static_assert(sizeof(ht_trackobj) == 24, "ht_trackobj is 24 bytes");

namespace {

thread_local std::string g_create_error;

template <class T>
inline T align_up(T v, T a) { return (v + a - 1) / a * a; }

// ------------------------------------------------------------------------------------------------
// device buffer that only ever grows (no allocation on the steady-state per-frame path)
struct DevBuf {
  void *p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};

// ------------------------------------------------------------------------------------------------
// Plan: everything that depends only on (w, h, interval) — src/ccv.js:110-160
struct Plan {
  int w = 0, h = 0, interval = 0;
  int next = 0, scale_upto = 0, n_slots = 0;
  std::vector<int> slot_w, slot_h;
  std::vector<int> plane_id;            // [slot*4+q] -> dense plane id or -1
  std::vector<DevPlane> planes;
  std::vector<DevJob> jobs;             // sorted by generation
  std::vector<TapEnt> taps;
  std::vector<DevPyrTile> pyr_tiles;    // grouped by generation
  std::vector<int> gen_tile_begin;      // size n_gens+1
  std::vector<DevScale> scales;
  std::vector<DevCascTile> casc_tiles;
  size_t arena_stride = 0;              // WORDS per frame quad (4 frames interleaved)
  uint32_t windows_per_frame = 0;
  DevBuf dev;
  DevPlan dplan{};
};

// floor(n / d) == (uint64(n) * M) >> k for all n <= 255 d + d / 2  (d = 4 dw dh): the exact-division constants of a
// canvas-shim drawImage.  false when the numerators do not fit 32 bits.
bool bilinear_division_constants(unsigned long long d, uint32_t &magic, uint32_t &shift) {
  const unsigned __int128 nmax = (unsigned __int128)d * 255 + d / 2 + 1;
  if (d == 0 || nmax >= ((unsigned __int128)1 << 32)) return false;
  int k = 32;
  while ((((unsigned __int128)1) << k) <= nmax * d) ++k;
  const unsigned __int128 M = ((((unsigned __int128)1) << k) / d) + 1;
  if (k > 63 || M >= ((unsigned __int128)1 << 32) || nmax * M >= ((unsigned __int128)1 << 64)) return false;
  magic = (uint32_t)M; shift = (uint32_t)k;
  return true;
}

int build_plan(Plan &P, int W, int H, int interval, int casc_w, int casc_h, std::string &err, bool upload = true) {
  P.w = W; P.h = H; P.interval = interval;
  const double scale = std::pow(2.0, 1.0 / (interval + 1.0));                      // ccv.js:110
  P.next = interval + 1;                                                            // ccv.js:111
  P.scale_upto = (int)std::floor(std::log((double)std::min(casc_w, casc_h)) / std::log(scale));  // :112
  P.n_slots = P.scale_upto + P.next * 2;                                            // :113
  if (P.n_slots > 120 || P.scale_upto < 1) { err = "unsupported interval"; return HT_ERR_ARG; }
  P.slot_w.assign(P.n_slots, 0); P.slot_h.assign(P.n_slots, 0);
  P.slot_w[0] = W; P.slot_h[0] = H;
  for (int i = 1; i <= interval; ++i) {                                             // :117-120
    P.slot_w[i] = (int)std::floor((double)W / std::pow(scale, (double)i));
    P.slot_h[i] = (int)std::floor((double)H / std::pow(scale, (double)i));
  }
  for (int i = P.next; i < P.n_slots; ++i) {                                        // :124-127
    P.slot_w[i] = P.slot_w[i - P.next] / 2;
    P.slot_h[i] = P.slot_h[i - P.next] / 2;
  }
  for (int i = 0; i < P.n_slots; ++i)
    if (P.slot_w[i] <= 0 || P.slot_h[i] <= 0) {
      err = "frame too small: pyramid level " + std::to_string(i) + " would be 0-sized (a browser throws here)";
      return HT_ERR_SIZE;
    }
  // ---- planes ----
  P.plane_id.assign((size_t)P.n_slots * 4, -1);
  size_t off = 0;
  auto add_plane = [&](int slot, int q) {
    DevPlane pl;
    pl.w = P.slot_w[slot]; pl.h = P.slot_h[slot];
    pl.pitch = align_up(pl.w, 4);             // words (one word = the pixel in the 4 frames of a quad)
    off = align_up(off, (size_t)64);          // 256 B
    pl.off = (uint32_t)off;
    off += (size_t)pl.pitch * pl.h;
    P.plane_id[(size_t)slot * 4 + q] = (int)P.planes.size();
    P.planes.push_back(pl);
  };
  for (int s = 0; s < P.n_slots; ++s) {
    add_plane(s, 0);
    if (s >= 2 * P.next) for (int q = 1; q < 4; ++q) add_plane(s, q);
  }
  if (off > 0x3C000000ull) { err = "frame too large"; return HT_ERR_SIZE; }
  P.arena_stride = align_up(off, (size_t)64);   // words per frame quad
  // ---- resample jobs, by generation ----
  std::vector<int> gen(P.n_slots, 0);
  int n_gens = 1;
  for (int s = 1; s < P.n_slots; ++s) {
    gen[s] = (s <= interval) ? 1 : gen[s - P.next] + 1;
    n_gens = std::max(n_gens, gen[s] + 1);
  }
  struct JobSpec { int gen, src_slot, dst_slot, q, sx, sy, sw, sh, dw, dh; };
  std::vector<JobSpec> specs;
  for (int s = 1; s < P.n_slots; ++s) {
    const int src = (s <= interval) ? 0 : s - P.next;
    const int sw = P.slot_w[src], sh = P.slot_h[src], w = P.slot_w[s], h = P.slot_h[s];
    specs.push_back({gen[s], src, s, 0, 0, 0, sw, sh, w, h});                       // :121, :128
    if (s >= 2 * P.next) {
      specs.push_back({gen[s], src, s, 1, 1, 0, sw - 1, sh, w - 2, h});            // :135
      specs.push_back({gen[s], src, s, 2, 0, 1, sw, sh - 1, w, h - 2});            // :140
      specs.push_back({gen[s], src, s, 3, 1, 1, sw - 1, sh - 1, w - 2, h - 2});    // :145
    }
  }
  std::stable_sort(specs.begin(), specs.end(), [](const JobSpec &a, const JobSpec &b) { return a.gen < b.gen; });
  P.gen_tile_begin.assign(n_gens + 1, 0);
  int cur_gen = 1;
  P.gen_tile_begin[0] = 0; P.gen_tile_begin[1] = 0;
  for (const JobSpec &js : specs) {
    while (cur_gen < js.gen) { ++cur_gen; P.gen_tile_begin[cur_gen] = (int)P.pyr_tiles.size(); }
    DevJob j{};
    j.src = P.plane_id[(size_t)js.src_slot * 4];
    j.dst = P.plane_id[(size_t)js.dst_slot * 4 + js.q];
    int dw = js.dw, dh = js.dh;
    if (dw <= 0 || dh <= 0 || js.sw <= 0 || js.sh <= 0) dw = dh = 0;  // paints nothing
    j.dw = dw; j.dh = dh;
    if (dw > 0) {
      if (dw > 32767 || dh > 32767 || js.sx + js.sw > 65535 || js.sy + js.sh > 65535) { err = "frame too large"; return HT_ERR_SIZE; }
      auto make_taps = [&](int d, int s, int s0) {
        const uint32_t first = (uint32_t)P.taps.size();
        for (int X = 0; X < d; ++X) {
          const long long un = (2LL * X + 1) * s - d;
          long long x0 = un / (2LL * d);
          if (un < 0 && (un % (2LL * d)) != 0) --x0;
          const long long f = un - x0 * 2LL * d;
          const long long a = std::min<long long>(std::max<long long>(x0, 0), s - 1);
          const long long b = std::min<long long>(std::max<long long>(x0 + 1, 0), s - 1);
          TapEnt t; t.a = (uint16_t)(a + s0); t.b = (uint16_t)(b + s0); t.f = (uint16_t)f; t.pad_ = 0;
          P.taps.push_back(t);
        }
        return first;
      };
      while (P.taps.size() & 3) P.taps.push_back(TapEnt{0, 0, 0, 0}); // column tables start 32 B aligned
      j.col_off = make_taps(dw, js.sw, js.sx);
      while (P.taps.size() & 3) P.taps.push_back(TapEnt{0, 0, 0, 0}); // k_resample reads column taps four at a time
      j.row_off = make_taps(dh, js.sh, js.sy);
      const unsigned long long d = 4ull * dw * dh;
      if (!bilinear_division_constants(d, j.magic, j.shift)) { err = "frame too large for 32-bit bilinear numerators"; return HT_ERR_SIZE; }
      j.half = (uint32_t)(d / 2);
    }
    const int job_id = (int)P.jobs.size();
    P.jobs.push_back(j);
    const DevPlane &dp = P.planes[j.dst];
    const DevPlane &spl = P.planes[j.src];
    j.src_off = spl.off; j.dst_off = dp.off; j.src_pitch = spl.pitch; j.dst_pitch = dp.pitch; j.dst_h = dp.h;
    P.jobs.back() = j;
    for (int ty = 0; ty < (dp.h + 31) / 32; ++ty)
      for (int tx = 0; tx < (dp.pitch + 31) / 32; ++tx) {
        DevPyrTile t; t.job = (uint16_t)job_id; t.tx = (uint16_t)tx; t.ty = (uint16_t)ty; t.pad_ = 0;
        P.pyr_tiles.push_back(t);
      }
  }
  while (cur_gen < n_gens) { ++cur_gen; P.gen_tile_begin[cur_gen] = (int)P.pyr_tiles.size(); }
  P.gen_tile_begin[n_gens] = (int)P.pyr_tiles.size();
  // ---- scales and cascade tiles ----
  double scale_x = 1.0;
  uint32_t win_base = 0;
  for (int i = 0; i < P.scale_upto; ++i) {                                          // ccv.js:154
    DevScale sc{};
    sc.p0 = P.plane_id[(size_t)i * 4];
    sc.p1 = P.plane_id[(size_t)(i + P.next) * 4];
    for (int q = 0; q < 4; ++q) sc.p2[q] = P.plane_id[(size_t)(i + 2 * P.next) * 4 + q];
    sc.qw = P.slot_w[i + 2 * P.next] - casc_w / 4;                                  // :155
    sc.qh = P.slot_h[i + 2 * P.next] - casc_h / 4;                                  // :156
    sc.win_base = win_base;
    sc.scale_x = scale_x;
    if (sc.qw > 0 && sc.qh > 0) {
      win_base += 4u * (uint32_t)sc.qw * (uint32_t)sc.qh;
      for (int ty = 0; ty < (sc.qh + TH - 1) / TH; ++ty)
        for (int tx = 0; tx < (sc.qw + TW - 1) / TW; ++tx) {
          DevCascTile t; t.scale = (uint16_t)i; t.tx = (uint16_t)tx; t.ty = (uint16_t)ty; t.pad_ = 0;
          P.casc_tiles.push_back(t);
        }
    }
    P.scales.push_back(sc);
    scale_x *= scale;                                                               // :244
  }
  P.windows_per_frame = win_base;
  if (!upload) return HT_OK;   // host-only self-test
  // ---- upload ----
  size_t o_planes = 0, o_jobs = align_up(o_planes + P.planes.size() * sizeof(DevPlane), (size_t)256);
  size_t o_taps = align_up(o_jobs + P.jobs.size() * sizeof(DevJob), (size_t)256);
  size_t o_pt = align_up(o_taps + P.taps.size() * sizeof(TapEnt), (size_t)256);
  size_t o_sc = align_up(o_pt + P.pyr_tiles.size() * sizeof(DevPyrTile), (size_t)256);
  size_t o_ct = align_up(o_sc + P.scales.size() * sizeof(DevScale), (size_t)256);
  size_t total = align_up(o_ct + P.casc_tiles.size() * sizeof(DevCascTile), (size_t)256);
  std::vector<uint8_t> host(total, 0);
  memcpy(host.data() + o_planes, P.planes.data(), P.planes.size() * sizeof(DevPlane));
  memcpy(host.data() + o_jobs, P.jobs.data(), P.jobs.size() * sizeof(DevJob));
  memcpy(host.data() + o_taps, P.taps.data(), P.taps.size() * sizeof(TapEnt));
  memcpy(host.data() + o_pt, P.pyr_tiles.data(), P.pyr_tiles.size() * sizeof(DevPyrTile));
  memcpy(host.data() + o_sc, P.scales.data(), P.scales.size() * sizeof(DevScale));
  memcpy(host.data() + o_ct, P.casc_tiles.data(), P.casc_tiles.size() * sizeof(DevCascTile));
  if (P.dev.reserve(total) != cudaSuccess) { err = "cudaMalloc(plan) failed"; return HT_ERR_CUDA; }
  if (cudaMemcpy(P.dev.p, host.data(), total, cudaMemcpyHostToDevice) != cudaSuccess) { err = "plan upload failed"; return HT_ERR_CUDA; }
  uint8_t *b = P.dev.as<uint8_t>();
  P.dplan.planes = reinterpret_cast<const DevPlane *>(b + o_planes);
  P.dplan.jobs = reinterpret_cast<const DevJob *>(b + o_jobs);
  P.dplan.taps = reinterpret_cast<const TapEnt *>(b + o_taps);
  P.dplan.pyr_tiles = reinterpret_cast<const DevPyrTile *>(b + o_pt);
  P.dplan.scales = reinterpret_cast<const DevScale *>(b + o_sc);
  P.dplan.casc_tiles = reinterpret_cast<const DevCascTile *>(b + o_ct);
  P.dplan.n_planes = (int)P.planes.size(); P.dplan.n_jobs = (int)P.jobs.size();
  P.dplan.n_scales = (int)P.scales.size(); P.dplan.n_casc_tiles = (int)P.casc_tiles.size();
  return HT_OK;
}

// ------------------------------------------------------------------------------------------------
// "HTC1" cascade blob (tools/pack_cascade.py) -> device tables
struct HostCascade {
  int n_stages = 0, n_features = 0, width = 0, height = 0;
  ConstCascade cc;      // image of the __constant__ table
  uint64_t id = 0;      // FNV-1a of cc: identical cascades share the loaded constants
  bool fast = false;    // blob == the cascade the generated stages were specialised for
  std::vector<LateFeat> late;          // late-stage records in scheduled order, 32 per chunk
  size_t n_sched = 0;                  // records of the schedule; late[n_sched + k] = feature k in original order
  std::vector<int32_t> late_chunk0;    // [n_stages + 1] first chunk of every stage
  int late_conflicts = 0;              // bank conflicts the schedule could not avoid (diagnostic)
};

// which cascade image is currently in c_casc, per device
uint64_t g_loaded_cascade[64] = {0};

int parse_cascade(const void *blob, size_t len, HostCascade &hc, std::string &err) {
  const uint8_t *b = static_cast<const uint8_t *>(blob);
  if (!b || len < 24 || memcmp(b, "HTC1", 4) != 0) { err = "cascade blob: bad magic"; return HT_ERR_CASCADE; }
  uint32_t hdr[5];
  memcpy(hdr, b + 4, 20);
  hc.n_stages = (int)hdr[0]; hc.n_features = (int)hdr[1]; hc.width = (int)hdr[2]; hc.height = (int)hdr[3];
  if (hc.n_stages < 1 || hc.n_stages > MAX_STAGES) { err = "cascade blob: stage count"; return HT_ERR_CASCADE; }
  if (hc.width != 24 || hc.height != 24) { err = "cascade blob: only 24x24 BBF windows are supported"; return HT_ERR_CASCADE; }
  const size_t need = 24 + (size_t)hc.n_stages * 16 + (size_t)hc.n_features * 48;
  if (len < need) { err = "cascade blob: truncated"; return HT_ERR_CASCADE; }
  if (hc.n_features > MAX_FEATS) { err = "cascade blob: more features than the constant table holds"; return HT_ERR_CASCADE; }
  const uint8_t *ps = b + 24, *pf = ps + (size_t)hc.n_stages * 16, *pa = pf + (size_t)hc.n_features * 32;
  ConstCascade &cc = hc.cc;
  memset(&cc, 0, sizeof(cc));
  int total = 0;
  for (int j = 0; j < hc.n_stages; ++j) {
    uint32_t cnt, first; double thr;
    memcpy(&cnt, ps + 16 * j, 4); memcpy(&first, ps + 16 * j + 4, 4); memcpy(&thr, ps + 16 * j + 8, 8);
    if ((int)first != total || (int)(first + cnt) > hc.n_features) { err = "cascade blob: stage table"; return HT_ERR_CASCADE; }
    total += (int)cnt;
    cc.stage[j].first = (int)first; cc.stage[j].count = (int)cnt; cc.stage[j].threshold = thr;
  }
  cc.n_stages = hc.n_stages;
  if (total != hc.n_features) { err = "cascade blob: feature count"; return HT_ERR_CASCADE; }
  auto point_off = [&](int z, int x, int y, bool &ok) -> uint16_t {
    const int lim = (24 >> z) - 1;
    if (z < 0 || z > 2 || x < 0 || y < 0 || x > lim || y > lim) { ok = false; return 0; }
    return (uint16_t)(point_word(z, x, y) | (z > 0 ? 0x8000 : 0));   // bit 15: relative to baseB
  };
  for (int k = 0; k < hc.n_features; ++k) {
    const uint8_t *r = pf + (size_t)k * 32;
    const int size = r[0];
    if (size < 1 || size > 5) { err = "cascade blob: feature size"; return HT_ERR_CASCADE; }
    bool ok = true;
    int cnt[2] = {0, 0};
    for (int side = 0; side < 2; ++side) {
      const uint8_t *z = r + (side ? 17 : 2), *x = z + 5, *y = z + 10;
      uint16_t *dst = &cc.off[k][side ? 5 : 0];
      if ((int8_t)z[0] < 0) { err = "cascade blob: slot 0 must be a valid point (src/ccv.js:191-192)"; return HT_ERR_CASCADE; }
      const uint16_t first = point_off((int8_t)z[0], x[0], y[0], ok);
      int m = 0;  // min/max are order independent: valid points are compacted to the front
      for (int q = 0; q < size; ++q)
        if ((int8_t)z[q] >= 0) dst[m++] = point_off((int8_t)z[q], x[q], y[q], ok);
      cnt[side] = m;
      for (; m < 5; ++m) dst[m] = first;
    }
    if (!ok) { err = "cascade blob: point out of the 24x24 window"; return HT_ERR_CASCADE; }
    cc.np_nn[k] = (uint8_t)(cnt[0] | (cnt[1] << 4));
    double a[2];
    memcpy(a, pa + (size_t)k * 16, 16);
    if (!(a[0] == -a[1])) { err = "cascade blob: alpha[2k] != -alpha[2k+1] (unsupported)"; return HT_ERR_CASCADE; }
    cc.alpha[k] = a[1];
  }
  // exact integer images of alpha / threshold (see LateFeat in ht_common.cuh)
  bool ints_ok = true;
  std::vector<long long> a_int((size_t)hc.n_features, 0);
  auto to_int = [&](double v, long long &out) {
    const double scaled = v * 1e8;
    const long long r = llround(scaled);
    out = r;
    return std::fabs(scaled - (double)r) < 1e-3 && ((double)r / 1e8) == v && std::llabs(r) < (1ll << 40);
  };
  for (int k = 0; k < hc.n_features; ++k)
    if (!to_int(cc.alpha[k], a_int[k]) || std::llabs(a_int[k]) > 0x7fffffffll) ints_ok = false;
  for (int j = 0; j < hc.n_stages; ++j) {
    long long ti = 0;
    if (!to_int(cc.stage[j].threshold, ti)) ints_ok = false;
    cc.thr_int[j] = ti;
  }
  uint64_t bh = 1469598103934665603ull;
  for (size_t i = 0; i < len; ++i) { bh ^= b[i]; bh *= 1099511628211ull; }
  hc.fast = (bh == HT_GEN_BLOB_ID) && (len == need) && ints_ok && hc.n_stages >= HT_GEN_STAGES && !getenv("HT_NO_LATE");
  if (getenv("HT_NO_FAST")) hc.fast = false;  // A/B switch for profiling: table-driven stages only
  // lane-per-window groups, then either warp-per-window late stages (exact integers) or, when the cascade's
  // numbers are not 8-digit decimals, lane-per-window groups to the end.
  {
    int g = 0;
    const int cuts_fast[] = {0, 2, 3, 4, 6};         // {0,1} {2} {3} {4,5} {6,7}: the generated stages
    const int cuts_int[] = {0, 2, 4, 6};
    const int cuts_fp[] = {0, 2, 4, 6, 9};
    static_assert(HT_GEN_STAGES == 8, "cuts_fast assumes 8 generated stages");
    if (hc.fast) {
      for (int cpos : cuts_fast) cc.group_first[g++] = cpos;
      cc.group_first[g] = HT_GEN_STAGES;
      cc.late_int = 1;
    } else if (ints_ok && !getenv("HT_NO_LATE")) {
      for (int cpos : cuts_int) if (cpos < hc.n_stages) cc.group_first[g++] = cpos;
      cc.group_first[g] = std::min(8, hc.n_stages);
      cc.late_int = 1;
    } else {
      for (int cpos : cuts_fp) if (cpos < hc.n_stages) cc.group_first[g++] = cpos;
      cc.group_first[g] = hc.n_stages;
      cc.late_int = 0;
    }
    cc.n_groups = g;
  }
  // ---- late-stage schedule: chunks of 32 records with bank-conflict-free load slots (LateFeat) ----
  hc.late.clear();
  hc.late_chunk0.assign((size_t)hc.n_stages + 1, 0);
  hc.late_conflicts = 0;
  for (int j = 0; j < hc.n_stages; ++j) {
    hc.late_chunk0[j] = (int32_t)(hc.late.size() / 32);
    if (j < cc.group_first[cc.n_groups]) continue;
    std::vector<int> rem;
    for (int k = cc.stage[j].first; k < cc.stage[j].first + cc.stage[j].count; ++k) rem.push_back(k);
    std::stable_sort(rem.begin(), rem.end(), [&](int x, int y) {   // features with many points first
      const int sx = (cc.np_nn[x] & 15) + (cc.np_nn[x] >> 4), sy = (cc.np_nn[y] & 15) + (cc.np_nn[y] >> 4);
      return sx > sy;
    });
    while (!rem.empty()) {
      int bank_word[10][32];                       // word offset that occupies (slot, bank), or -1
      for (auto &row : bank_word) for (int &v : row) v = -1;
      // place one side (p: slots 0-4, n: slots 5-9) of feature k; returns the conflicts it adds (dry = do not commit)
      auto place_side = [&](int k, int side, uint16_t *out, bool allow_conflicts, bool dry) -> int {
        const int cnt = side ? (cc.np_nn[k] >> 4) : (cc.np_nn[k] & 15);
        const uint16_t *pt = &cc.off[k][side ? 5 : 0];
        int order[5] = {0, 1, 2, 3, 4}, best_cost = 1 << 30, best[5] = {0, 1, 2, 3, 4};
        do {   // slot of point i = order[i]; <= 120 permutations
          int cost = 0;
          for (int i = 0; i < cnt; ++i) {
            const int slot = side * 5 + order[i], word = pt[i] & 0x7fff, bw = bank_word[slot][word & 31];
            if (bw >= 0 && bw != word) cost += 1 << 10;   // a bank conflict
            cost += order[i];                              // prefer the low slots: a slot nobody uses costs no wavefront
          }
          if (cost < best_cost) { best_cost = cost; for (int i = 0; i < 5; ++i) best[i] = order[i]; }
        } while (std::next_permutation(order, order + 5));
        const int conflicts = best_cost >> 10;
        if (conflicts && !allow_conflicts) return -1;
        if (!dry) {
          for (int i = 0; i < cnt; ++i) {
            const int slot = side * 5 + best[i], word = pt[i] & 0x7fff;
            if (bank_word[slot][word & 31] < 0) bank_word[slot][word & 31] = word;
            out[slot] = pt[i];
          }
        }
        return conflicts;
      };
      for (int lane = 0; lane < 32; ++lane) {
        struct { uint16_t off[10]; int32_t a_int; } lf;   // scheduled in ConstCascade's 16-bit offsets, encoded at the end
        for (int q = 0; q < 10; ++q) lf.off[q] = 0xFFFF;
        lf.a_int = 0;
        if (!rem.empty()) {
          size_t pick = rem.size();
          for (size_t i = 0; i < rem.size() && pick == rem.size(); ++i)
            if (place_side(rem[i], 0, lf.off, false, true) == 0 && place_side(rem[i], 1, lf.off, false, true) == 0) pick = i;
          if (pick == rem.size()) {   // nothing fits conflict-free: take the feature that adds the fewest conflicts
            int best_c = 1 << 30;
            for (size_t i = 0; i < rem.size(); ++i) {
              const int cfl = place_side(rem[i], 0, lf.off, true, true) + place_side(rem[i], 1, lf.off, true, true);
              if (cfl < best_c) { best_c = cfl; pick = i; }
            }
          }
          const int k = rem[pick];
          hc.late_conflicts += place_side(k, 0, lf.off, true, false) + place_side(k, 1, lf.off, true, false);
          lf.a_int = (int32_t)a_int[k];
          rem.erase(rem.begin() + (long)pick);
        }
        LateFeat rec{};
        for (int q = 0; q < 10; ++q) rec.off[q] = late_encode(lf.off[q]);
        rec.a_int = lf.a_int;
        hc.late.push_back(rec);
      }
    }
  }
  hc.late_chunk0[hc.n_stages] = (int32_t)(hc.late.size() / 32);
  if (hc.late.empty()) hc.late.resize(32);
  // every feature once more in ORIGINAL order: the warp-parallel ordered fp64 sum (stage_sum_ordered_warp)
  hc.n_sched = hc.late.size();
  for (int k = 0; k < hc.n_features; ++k) {
    LateFeat lf{};
    for (int q = 0; q < 10; ++q) lf.off[q] = LATE_UNUSED;
    for (int q = 0; q < (cc.np_nn[k] & 15); ++q) lf.off[q] = late_encode(cc.off[k][q]);
    for (int q = 0; q < (cc.np_nn[k] >> 4); ++q) lf.off[5 + q] = late_encode(cc.off[k][5 + q]);
    lf.a_int = (int32_t)a_int[k];
    hc.late.push_back(lf);
  }
  uint64_t hsh = 1469598103934665603ull;
  const uint8_t *cb = reinterpret_cast<const uint8_t *>(&cc);
  for (size_t i = 0; i < sizeof(cc); ++i) { hsh ^= cb[i]; hsh *= 1099511628211ull; }
  hc.id = hsh ? hsh : 1;
  return HT_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
struct ht_ctx {
  ht_config cfg{};
  int K = 64, raw_cap = 1024;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  std::string err;
  uint64_t launches = 0;

  HostCascade hc;
  DevBuf d_casc;  // LateFeat table

  std::map<std::tuple<int, int, int>, std::unique_ptr<Plan>> plans;
  Plan *last_plan = nullptr;
  int last_n = 0;

  DevBuf arena, d_frames, raw_keys, raw_conf, raw_count, sorted, labels, seq2, d_out_rects, d_out_counts, d_flags;
  DevBuf bins;  // [frames][h][w] u16 colour-bin planes written by k_hist, read by k_track
  DevBuf model_hist, cur_hist, track_state, d_slots, d_rects, d_found, d_objs, d_windows, d_wb_sums, d_wb_out, d_scratch;

  // optional per-kernel-class device timing (CUDA events on the launching stream) for bench.py's roofline
  bool prof_on = false;
  struct ProfSpan { int cls; cudaEvent_t a, b; };
  std::vector<ProfSpan> prof_spans;
  std::vector<cudaEvent_t> prof_free;
  double prof_ms[HT_PROF_N] = {0};
  uint64_t prof_launches[HT_PROF_N] = {0};

  cudaEvent_t prof_event() {
    cudaEvent_t e = nullptr;
    if (!prof_free.empty()) { e = prof_free.back(); prof_free.pop_back(); }
    else cudaEventCreate(&e);
    return e;
  }
  void prof_begin(int cls) {
    if (!prof_on) return;
    ProfSpan s{cls, prof_event(), prof_event()};
    cudaEventRecord(s.a, stream);
    prof_spans.push_back(s);
  }
  void prof_end() {
    if (!prof_on) return;
    cudaEventRecord(prof_spans.back().b, stream);
  }

  cudaStream_t aux_stream = nullptr;        // tracking of part p overlaps the detection of part p+1 (ht_detect_track)
  cudaEvent_t aux_done = nullptr, part_events[4] = {nullptr, nullptr, nullptr, nullptr};
  unsigned part_seq = 0;
  // ht_set_pipeline: ht_detect_track on device-resident frames with device outputs leaves the tracking of call s on
  // the aux stream and returns; it runs under the detection of call s+1 (k_track is a latency chain that leaves
  // most issue slots idle, the detection kernels are throughput-bound).  What the two touch in common is double
  // buffered by call parity (bin planes, current-frame histograms) or ordered by an event (the caller's rectangle
  // arrays: k_group of call s+1 waits for the tracking of call s).  Every other entry point joins first.
  int pipeline = 0;
  bool aux_pending = false;                 // work on aux_stream that the context's stream has not waited for yet
  cudaEvent_t pipe_detect_done = nullptr;
  int pipe_parity = 0;
  size_t bins_off = 0, hist_off = 0;        // element offsets of the active bin-plane / histogram buffer (parity)
  // Tracking of part p on a second stream while part p+1 is uploaded / detected (ht_detect_track).  Default (-1):
  // only for HOST frames, where the batch arrives at PCIe speed and the GPU has idle time to fill - measured e2e
  // 37.6k vs 33.0k frames/s with 4 parts (8 parts 36.8k, 16 parts 28.6k).  For device-resident frames it was
  // measured slower (24.4-26.7 vs 22.3 ms per step) and stays off.  HT_OVERLAP=0 disables, HT_OVERLAP=<parts> forces.
  int detect_pipe = 0;                      // HT_DETECT_PIPE=1: gray + pyramid of wave w+1 on a second stream under the cascade of wave w
  int wave_frames = 0;                      // frames per wave of run_detect (HT_WAVE); 0: from wave_mb
  int wave_mb = 2048;                       // pyramid-arena budget of one wave in MB (HT_WAVE_MB).  64 (half of the L2) keeps
                                            // the pyramid out of HBM but costs 28 % throughput in launch tails: lab notes
  int force_ties = 0;                       // ht_debug_set_exactness: force the exactness fallbacks (tests)
  cudaStream_t pipe_stream = nullptr;
  cudaEvent_t pipe_start = nullptr, pipe_events[4] = {};
  bool use_tma = true;                      // stage level-1 cascade tiles with cp.async.bulk.tensor (HT_TMA=0: 16-byte cp.async)
  DevBuf d_tmaps;                           // [arenas][scales] 128 B CUtensorMaps over the level-1 planes
  const void *tmap_arena = nullptr;
  const void *tmap_plan = nullptr;
  size_t tmap_wave_words = 0;
  int tmap_arenas = 0;
  int last_wave_f0 = 0, last_wave_n = 0;    // frames whose pyramid is still in the arena (ht_debug_plane)
  const uint32_t *last_wave_arena = nullptr;
  DevBuf d_late_chunk0;
  int overlap_track = -1;
  int overlap_parts = 0;
  cudaStream_t copy_stream = nullptr;       // H2D staging stream of ht_detect_track
  cudaEvent_t compute_done = nullptr;
  std::vector<cudaEvent_t> chunk_events;
  int h2d_chunk = 64;                       // frames per pipelined upload chunk
  int track_cluster = 0;                    // >0: force that k_track cluster size, 2, 4 or 8 (HT_TRACK_CLUSTER, A/B profiling)
  bool track_memo = true;                   // k_track re-uses the moments of windows it has already summed in this
                                            // launch (ht_set_track_memo / HT_TRACK_MEMO=0 for the strict A/B)
  bool track_trace = false;                 // HT_TRACK_TRACE=1: k_track writes a per-stream timeline (ht_debug_track_trace)
  DevBuf d_trace;
  bool track_lpt = true;                    // longest-chain-first launch order (HT_TRACK_LPT=0 disables)
  DevBuf d_stream_mode, d_stream_mask, d_stream_cs, d_stream_init, d_stream_events;   // ht_stream_step
  DevBuf d_head_state, d_head_params, d_head_events;                                  // ht_stream_head_config
  bool head_on = false;
  DevBuf d_track_cost;                      // [max_frames][2] {passes, window pixels / 256} per slot
  int track_heavy_div = 128;                // >0: the n/div costliest streams run on clusters of
  int track_heavy_cluster = 8;              //     track_heavy_cluster CTAs (HT_TRACK_HEAVY=div[,cluster])
  int track_mid_div = 32, track_mid_cluster = 4;  // HT_TRACK_MID=div[,cluster]: the next n/32 costliest streams on clusters of 4
                                                  // (call 4: 4.12 -> 3.40 ms per 1024 x 30 calls with n/16; call 17, with
                                                  // prioritised tier streams: n/64 + n/16 3.17, n/128 + n/32 2.97, n/64 + n/48 3.00)
  cudaStream_t tier_stream[3] = {nullptr, nullptr, nullptr};   // heavy, mid, rest
  cudaEvent_t tier_done[3] = {nullptr, nullptr, nullptr};
  int track_mask_frames = 4;                // >0: mask only streams whose last launch swept more than this many frames' worth of pixels
  int track_mask_min = 4;                   // HT_TRACK_MASK=<min n_calls> (0: off): zero-weight marking of the bin plane before k_track
  cudaEvent_t sched_ready = nullptr;
  DevBuf d_sched;                           // k_track launch-order scratch: [area | order][max_frames]

  int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof(buf), fmt, ap); va_end(ap);
    err = buf;
    return code;
  }
};

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return ctx->fail(HT_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

namespace {

bool is_device_ptr(const void *p) {
  if (!p) return false;
  cudaPointerAttributes a{};
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// (ht_set_pipeline) order everything still running on the aux stream before later work on the context's stream, and go
// back to the first bin-plane / histogram buffer.  Called by every entry point except the pipelined ht_detect_track.
int join_aux(ht_ctx *ctx) {
  if (ctx->aux_pending) {
    CK(cudaStreamWaitEvent(ctx->stream, ctx->aux_done, 0));
    ctx->aux_pending = false;
  }
  ctx->bins_off = 0; ctx->hist_off = 0; ctx->pipe_parity = 0;
  return HT_OK;
}

int get_plan(ht_ctx *ctx, int w, int h, int interval, Plan **out) {
  if (w <= 0 || h <= 0 || interval < 0 || interval > 15) return ctx->fail(HT_ERR_ARG, "bad w/h/interval");
  if (w > ctx->cfg.max_width || h > ctx->cfg.max_height)
    return ctx->fail(HT_ERR_SIZE, "frame %dx%d exceeds the context maximum %dx%d", w, h, ctx->cfg.max_width, ctx->cfg.max_height);
  auto key = std::make_tuple(w, h, interval);
  auto it = ctx->plans.find(key);
  if (it == ctx->plans.end()) {
    std::unique_ptr<Plan> p(new Plan());
    std::string err;
    int rc = build_plan(*p, w, h, interval, ctx->hc.width, ctx->hc.height, err);
    if (rc != HT_OK) return ctx->fail(rc, "%s", err.c_str());
    it = ctx->plans.emplace(key, std::move(p)).first;
  }
  *out = it->second.get();
  return HT_OK;
}

// stage n frames on the device if the caller passed host memory
int device_frames(ht_ctx *ctx, const uint8_t *rgba, int n, int w, int h, const uint8_t **out) {
  if (!rgba) return ctx->fail(HT_ERR_ARG, "rgba is NULL");
  if ((reinterpret_cast<uintptr_t>(rgba) & 3u) != 0) return ctx->fail(HT_ERR_ARG, "rgba must be 4-byte aligned");
  if (is_device_ptr(rgba)) { *out = rgba; return HT_OK; }
  const size_t bytes = (size_t)n * w * h * 4;
  CK(ctx->d_frames.reserve(bytes));
  CK(cudaMemcpyAsync(ctx->d_frames.p, rgba, bytes, cudaMemcpyHostToDevice, ctx->stream));
  *out = ctx->d_frames.as<uint8_t>();
  return HT_OK;
}

// argument check of every batched entry point; it also joins a pipelined call's tracking (ht_set_pipeline) unless the
// caller is the pipelined path itself
int check_batch(ht_ctx *ctx, int n, bool join = true) {
  if (n <= 0 || n > ctx->cfg.max_frames) return ctx->fail(HT_ERR_ARG, "n=%d outside [1,%d]", n, ctx->cfg.max_frames);
  if (join) return join_aux(ctx);
  return HT_OK;
}

int upload_slots(ht_ctx *ctx, const int32_t *slots, int n, const int32_t **d_slots) {
  *d_slots = nullptr;
  if (!slots) return HT_OK;
  if (is_device_ptr(slots)) { *d_slots = slots; return HT_OK; }
  // two entries with the same slot would make two clusters of k_track (or two CTAs of k_track_init) race on
  // state[slot] / model_hist[slot].  (Device-resident slot arrays are the caller's responsibility: see the header.)
  std::vector<uint8_t> seen((size_t)ctx->cfg.max_frames, 0);
  for (int i = 0; i < n; ++i) {
    if (slots[i] < 0 || slots[i] >= ctx->cfg.max_frames) return ctx->fail(HT_ERR_ARG, "slot %d out of range", slots[i]);
    if (seen[(size_t)slots[i]]++) return ctx->fail(HT_ERR_ARG, "slot %d appears twice in one batch", slots[i]);
  }
  CK(ctx->d_slots.reserve(sizeof(int32_t) * ctx->cfg.max_frames));
  CK(cudaMemcpyAsync(ctx->d_slots.p, slots, sizeof(int32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
  *d_slots = ctx->d_slots.as<int32_t>();
  return HT_OK;
}

int ensure_tracker_buffers(ht_ctx *ctx) {
  const size_t mf = (size_t)ctx->cfg.max_frames;
  if (!ctx->model_hist.p) {
    CK(ctx->model_hist.reserve(mf * 4096 * sizeof(uint32_t)));
    CK(ctx->cur_hist.reserve(2 * mf * 4096 * sizeof(uint32_t)));   // two parities (ht_set_pipeline)
    CK(ctx->track_state.reserve(mf * sizeof(TrackState)));
    CK(cudaMemsetAsync(ctx->track_state.p, 0, mf * sizeof(TrackState), ctx->stream));
    CK(ctx->d_rects.reserve(mf * 4 * sizeof(int32_t)));
    CK(ctx->d_found.reserve(mf * sizeof(int32_t)));
    CK(ctx->d_objs.reserve(mf * 6 * sizeof(int32_t)));
    CK(ctx->d_windows.reserve(mf * 4 * sizeof(int32_t)));
    CK(ctx->d_sched.reserve(2 * mf * sizeof(int32_t)));
    CK(ctx->d_track_cost.reserve(2 * mf * sizeof(int32_t)));
    CK(cudaMemsetAsync(ctx->d_track_cost.p, 0, 2 * mf * sizeof(int32_t), ctx->stream));
    if (ctx->track_trace) {   // [mf x 4] per-stream records, then [mf x 8] phase totals (HT_TRACK_PASSTRACE builds)
      CK(ctx->d_trace.reserve(12 * mf * sizeof(unsigned long long)));
      CK(cudaMemsetAsync(ctx->d_trace.p, 0, 12 * mf * sizeof(unsigned long long), ctx->stream));
    }
  }
  return HT_OK;
}

int launch_hist(ht_ctx *ctx, const uint8_t *d_rgba, int n, int w, int h, uint32_t *hist, uint16_t *bins,
                const uint8_t *enable = nullptr) {
  const int n_px = w * h;
  int chunks = 1;
  if (n < 592) chunks = std::min(64, std::max(1, 1184 / n));  // keep ~8 CTAs per SM busy for small batches
  if (chunks > 1) CK(cudaMemsetAsync(hist, 0, (size_t)n * 4096 * sizeof(uint32_t), ctx->stream));   // (also for disabled frames: harmless)
  ctx->prof_begin(HT_PROF_HIST);
  k_hist<<<dim3(chunks, n), 256, 0, ctx->stream>>>(d_rgba, (size_t)n_px * 4, n_px, hist, bins, chunks, enable);
  ctx->prof_end();
  ++ctx->launches;
  CK(cudaGetLastError());
  return HT_OK;
}

// per-launch options of k_track that do not depend on the batch
struct TrackOpts {
  unsigned long long *trace;   // HT_TRACK_TRACE=1: per-stream timeline buffer (else NULL)
  size_t trace_stride;         // u64 entries between a stream's record and its phase totals
  int memo;                    // ht_ctx::track_memo
  int force_serial;            // ht_ctx::force_ties & 4
  int32_t *cost;               // per slot {passes, window pixels / 256} of the last launch (scheduling history)
  const uint8_t *enable;       // ht_stream_step: per stream, 0 = not tracking this frame (else NULL)
};

template <int C>
cudaError_t launch_track_c(cudaStream_t st, int n, const uint16_t *bins, int w, int h, const int32_t *d_slots,
                           const uint32_t *mh, const uint32_t *ch, TrackState *state, int n_calls, int32_t *d_objs,
                           int32_t *d_win, int32_t *flag, unsigned long long *stats, const int32_t *order, int list_off,
                           TrackOpts opt) {
  // Same shared-memory carve-out as k_cascade (the maximum): an SM only changes its L1 / shared split when it is idle,
  // so CTAs of kernels that ask for different splits do not mix on one SM - and k_track is meant to run beside the
  // detection kernels of the next call (ht_set_pipeline).
  static bool carveout_set = false;
  if (!carveout_set) {
    cudaError_t ce = cudaFuncSetAttribute(k_track<C>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (ce != cudaSuccess) return ce;
    carveout_set = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)n * C);
  cfg.blockDim = dim3(TRACK_THREADS);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k_track<C>, bins, w, h, d_slots, mh, ch, state, n_calls, d_objs, d_win, flag, stats,
                            order, list_off, opt.trace, opt.trace_stride, opt.memo, opt.force_serial, opt.cost, opt.enable);
}

// cluster size chosen at run time: 2, 4 or 8 CTAs per stream (any other value: 8)
cudaError_t launch_track_cluster(int c, cudaStream_t st, int n, const uint16_t *bins, int w, int h, const int32_t *d_slots,
                                 const uint32_t *mh, const uint32_t *ch, TrackState *state, int n_calls, int32_t *d_objs,
                                 int32_t *d_win, int32_t *flag, unsigned long long *stats, const int32_t *order,
                                 int list_off, TrackOpts opt) {
  switch (c) {
    case 2: return launch_track_c<2>(st, n, bins, w, h, d_slots, mh, ch, state, n_calls, d_objs, d_win, flag, stats, order, list_off, opt);
    case 4: return launch_track_c<4>(st, n, bins, w, h, d_slots, mh, ch, state, n_calls, d_objs, d_win, flag, stats, order, list_off, opt);
    default: return launch_track_c<8>(st, n, bins, w, h, d_slots, mh, ch, state, n_calls, d_objs, d_win, flag, stats, order, list_off, opt);
  }
}

int launch_track(ht_ctx *ctx, int n, int f0, const uint16_t *bins, int w, int h, const int32_t *d_slots, const uint32_t *mh,
                 const uint32_t *ch, TrackState *state, int n_calls, int32_t *d_objs, int32_t *d_win, int32_t *flag,
                 const uint8_t *enable = nullptr) {
  unsigned long long *stats = ctx->d_flags.as<unsigned long long>() + 8;
  cudaStream_t st = ctx->stream;
  // several track() calls on this frame: mark the plane entries whose weight is +0.0 first (k_bins_mask), k_track then
  // skips whole row segments of them.  (One call per frame - ht_stream_step - does not repay the extra pass.)
  if (ctx->track_mask_min > 0 && n_calls >= ctx->track_mask_min) {
    const int chunks = std::max(1, std::min(64, 1184 / std::max(1, n)));
    // selective (default): only streams whose previous launch visited more than track_mask_frames whole frames' worth
    // of pixels (history of the slot; first launch: nobody) - 1/10 of the bench mix, and nearly all of its pixel visits
    const int min_px256 = (int)std::min<long long>(((long long)ctx->track_mask_frames * w * h) >> 8, 0x7fffffff);
    k_bins_mask<<<dim3((unsigned)chunks, (unsigned)n), 256, 0, st>>>(const_cast<uint16_t *>(bins), w * h, mh, d_slots, state, chunks, enable,
                                                                     ctx->track_mask_frames > 0 ? ctx->d_track_cost.as<int32_t>() : nullptr, min_px256);
    ++ctx->launches;
  }
  const TrackOpts opt{ctx->track_trace ? ctx->d_trace.as<unsigned long long>() + 4 * (size_t)f0 : nullptr,
                      // (the kernel indexes both areas with the stream number relative to f0)
                      4 * (size_t)ctx->cfg.max_frames - 4 * (size_t)f0 + 8 * (size_t)f0,
                      ctx->track_memo ? 1 : 0, (ctx->force_ties & 4) ? 1 : 0, ctx->d_track_cost.as<int32_t>(), enable};
  // per-chunk launch-order scratch: [area n][order n]
  int32_t *area = ctx->d_sched.as<int32_t>() + (size_t)f0;
  int32_t *order = ctx->d_sched.as<int32_t>() + (size_t)ctx->cfg.max_frames + f0;
  cudaError_t e = cudaSuccess;
  // few streams -> 8 CTAs per stream (latency of one stream); many streams -> 2 (more streams resident).
  // measured on 1024 streams x 30 calls in index order: 1 CTA 9.7 ms, 2 CTAs 6.1 ms, 4 CTAs 6.2 ms, 8 CTAs 10.1 ms
  int c = ctx->track_cluster;
  if (c <= 0) c = (n >= 256) ? 2 : (n >= 32 ? 4 : 8);
  const bool lpt = ctx->track_lpt && n >= 128;     // below that every stream is resident from the start
  if (!lpt) {
    e = launch_track_cluster(c, st, n, bins, w, h, d_slots, mh, ch, state, n_calls, d_objs, d_win, flag, stats, nullptr, 0, opt);
    ++ctx->launches;
  } else {
    // longest chain first: order the streams by their expected cost (k_track_area / k_track_rank)
    k_track_area<<<(n + 255) / 256, 256, 0, st>>>(state, d_slots, n, ctx->d_track_cost.as<int32_t>(), area);
    k_track_rank<<<(n + 255) / 256, 256, 0, st>>>(area, n, order);
    ctx->launches += 2;
    // Tiers by cost rank, each on its own stream so that they run concurrently, costliest first:
    //   the costliest n / heavy_div streams on clusters of 8 (long chains over large windows: shorten every pass),
    //   the next n / mid_div on clusters of 4, the rest on clusters of `c` (2).
    struct Tier { int count, cluster, side; };   // side >= 0: ctx->tier_stream[side]; -1: the context's stream
    Tier tiers[3];
    int n_tiers = 0, left = n;
    auto take = [&](int div, int cl, int side) {
      const int k = (div > 0) ? std::min(left, n / div) : 0;
      if (k > 0) { tiers[n_tiers++] = Tier{k, cl, side}; left -= k; }
    };
    take(ctx->track_heavy_div, ctx->track_heavy_cluster, 0);
    take(ctx->track_mid_div, ctx->track_mid_cluster, 1);
    // Round 2, call 8 timeline: with the default tier on the context's own stream (no event wait) its 1,888 CTAs
    // reached the GPU first and filled every slot with ITS costliest streams; the heavy and middle tiers - the
    // longest chains of the launch - started 1.4 ms late and the launch ended at 1.4 + 2.3 ms.  Now every tier sits
    // on a side stream behind the same event, submitted costliest tier first, and the side streams carry
    // descending priorities (heavy > mid > rest), so a free slot always goes to the longest pending chain.
    const bool rest_side = ctx->track_heavy_div > 0 || ctx->track_mid_div > 0;
    if (left > 0) tiers[n_tiers++] = Tier{left, c, rest_side ? 2 : -1};
    if (n_tiers > 1) {
      int prio_least = 0, prio_greatest = 0;
      CK(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));   // numerically lower = more urgent
      for (int t = 0; t < 3; ++t)
        if (!ctx->tier_stream[t]) {
          CK(cudaStreamCreateWithPriority(&ctx->tier_stream[t], cudaStreamNonBlocking, std::min(prio_least, prio_greatest + t)));
          CK(cudaEventCreateWithFlags(&ctx->tier_done[t], cudaEventDisableTiming));
        }
      if (!ctx->sched_ready) CK(cudaEventCreateWithFlags(&ctx->sched_ready, cudaEventDisableTiming));
      CK(cudaEventRecord(ctx->sched_ready, st));
    }
    int off = 0;
    for (int t = 0; t < n_tiers && e == cudaSuccess; ++t) {
      cudaStream_t ts = tiers[t].side >= 0 ? ctx->tier_stream[tiers[t].side] : st;
      if (tiers[t].side >= 0) CK(cudaStreamWaitEvent(ts, ctx->sched_ready, 0));
      e = launch_track_cluster(tiers[t].cluster, ts, tiers[t].count, bins, w, h, d_slots, mh, ch, state, n_calls, d_objs, d_win,
                               flag, stats, order, off, opt);
      ++ctx->launches;
      if (tiers[t].side >= 0) CK(cudaEventRecord(ctx->tier_done[tiers[t].side], ts));
      off += tiers[t].count;
    }
    for (int t = 0; t < n_tiers; ++t)
      if (tiers[t].side >= 0) CK(cudaStreamWaitEvent(st, ctx->tier_done[tiers[t].side], 0));
  }
  if (e != cudaSuccess) return ctx->fail(HT_ERR_CUDA, "k_track launch: %s", cudaGetErrorString(e));
  return HT_OK;
}

int track_init_common(ht_ctx *ctx, const int32_t *slots, int n, const uint8_t *d_rgba, int w, int h,
                      const int32_t *d_rects, int calc_angles, int32_t *out_found) {
  const int32_t *d_slots = nullptr;
  int rc = upload_slots(ctx, slots, n, &d_slots);
  if (rc != HT_OK) return rc;
  const bool found_dev = out_found && is_device_ptr(out_found);
  int32_t *d_found = out_found ? (found_dev ? out_found : ctx->d_found.as<int32_t>()) : nullptr;
  ctx->prof_begin(HT_PROF_TRACK_INIT);
  k_track_init<<<n, 256, 0, ctx->stream>>>(d_rgba, (size_t)w * h * 4, w, h, d_slots, d_rects, calc_angles ? 1 : 0,
                                           ctx->model_hist.as<uint32_t>(), ctx->track_state.as<TrackState>(), d_found, nullptr);
  ctx->prof_end();
  ++ctx->launches;
  CK(cudaGetLastError());
  if (out_found && !found_dev) {
    CK(cudaMemcpyAsync(out_found, d_found, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return HT_OK;
}

// Shared memory of one k_cascade CTA: the staged tile and three sets of per-class survivor bit masks.
constexpr size_t CASC_SMEM = (size_t)TILE_WORDS * 4 + 3 * (size_t)MASK_WORDS * 32 * sizeof(uint32_t);
constexpr size_t GRAY_HIST_SMEM = 2 * 4096 * sizeof(uint32_t);   // two frames per word, 16-bit counters

int set_kernel_attributes(ht_ctx *ctx) {
  CK(cudaFuncSetAttribute(k_cascade<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CASC_SMEM));
  CK(cudaFuncSetAttribute(k_cascade<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CASC_SMEM));
  CK(cudaFuncSetAttribute(k_cascade<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  CK(cudaFuncSetAttribute(k_cascade<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
  CK(cudaFuncSetAttribute(k_gray<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GRAY_HIST_SMEM));
  CK(cudaFuncSetAttribute(k_gray<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GRAY_HIST_SMEM));
  return HT_OK;
}

// Tensor maps for the TMA staging of level-1 cascade tiles: one 3-D map (column, row, frame quad) per scale and
// arena over the pyramid arena (32-bit elements: one word = the pixel in 4 frames).  Re-encoded whenever the arena
// allocation, its partition into waves or the plan changes.
int ensure_tensor_maps(ht_ctx *ctx, Plan *P, int n_arenas, size_t wave_words, int quads_per_arena) {
  if (ctx->tmap_arena == ctx->arena.p && ctx->tmap_plan == P && ctx->tmap_wave_words == wave_words && ctx->tmap_arenas == n_arenas)
    return HT_OK;
  typedef CUresult (*encode_fn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static encode_fn encode = nullptr;
  if (!encode) {
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn) {
      cudaGetLastError();
      ctx->use_tma = false;   // old driver: level 1 is staged with 16-byte cp.async like the other levels
      return HT_OK;
    }
    encode = reinterpret_cast<encode_fn>(fn);
  }
  static_assert(sizeof(CUtensorMap) == 128, "CUtensorMap is 128 bytes");
  const size_t ns = P->scales.size();
  std::vector<CUtensorMap> maps(ns * (size_t)n_arenas);
  memset(maps.data(), 0, maps.size() * sizeof(CUtensorMap));
  for (int a = 0; a < n_arenas; ++a)
    for (size_t i = 0; i < ns; ++i) {
      const DevScale &sc = P->scales[i];
      if (sc.qw <= 0 || sc.qh <= 0) continue;
      const DevPlane &pl = P->planes[sc.p1];
      cuuint64_t dims[3] = {(cuuint64_t)pl.pitch, (cuuint64_t)pl.h, (cuuint64_t)quads_per_arena};
      cuuint64_t strides[2] = {(cuuint64_t)pl.pitch * 4, (cuuint64_t)P->arena_stride * 4};
      cuuint32_t box[3] = {(cuuint32_t)P1, (cuuint32_t)L1_ROWS, 1};
      cuuint32_t estr[3] = {1, 1, 1};
      void *base = ctx->arena.as<uint32_t>() + (size_t)a * wave_words + pl.off;
      CUresult r = encode(&maps[(size_t)a * ns + i], CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, base, dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return ctx->fail(HT_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d) for scale %d", (int)r, (int)i);
    }
  CK(ctx->d_tmaps.reserve(maps.size() * sizeof(CUtensorMap)));
  CK(cudaMemcpyAsync(ctx->d_tmaps.p, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));   // `maps` is a local; re-encoding only happens when buffers change
  ctx->tmap_arena = ctx->arena.p;
  ctx->tmap_plan = P;
  ctx->tmap_wave_words = wave_words;
  ctx->tmap_arenas = n_arenas;
  return HT_OK;
}

// what camshift needs from the frame, produced by the gray pass of the same read (src/camshift.js:268)
struct HistOut {
  uint32_t *hist;   // [n][4096] current-frame histograms (frame f0 first), or NULL
  uint16_t *bins;   // [n][h*w]  weight-table offsets, or NULL
};

// gray -> pyramid -> cascade -> sort+group for frames [f0, f0+n) of a device-resident batch.
// Every per-frame buffer is indexed by absolute frame number so that chunks can be pipelined.
//
// The frames are processed in WAVES of ctx->wave_frames (whole frame quads): the pyramid arena holds one wave
// (8 MB per 640x480 quad) and is re-used by the next one, so that it lives in the 126 MB L2 instead of making a
// round trip through HBM for the whole batch (round 1: 1.86 GB read by k_cascade per 1024 frames).  With
// ctx->detect_pipe the gray + pyramid kernels of wave w+1 run on a second stream (and a second arena) under the
// cascade of wave w.
int run_detect(ht_ctx *ctx, Plan *P, const uint8_t *d_rgba_batch, int f0, int n, int min_neighbors, Rect *d_rects_batch,
               int32_t *d_counts_batch, HistOut ho = HistOut{nullptr, nullptr}, const uint8_t *quad_mask = nullptr,
               cudaEvent_t before_group = nullptr) {
  cudaStream_t st = ctx->stream;
  const int w = P->w, h = P->h;
  const size_t frame_bytes = (size_t)w * h * 4;
  // frames per wave: HT_WAVE, or as many as fit the arena budget (one frame of a quad costs arena_stride bytes)
  const int wave = ctx->wave_frames > 0 ? std::max(4, ctx->wave_frames & ~3)
                                        : std::max(4, (int)std::min<size_t>(((size_t)ctx->wave_mb << 20) / P->arena_stride, 1u << 20) & ~3);
  const size_t wave_words = P->arena_stride * (size_t)(wave / 4);
  const bool piped = ctx->detect_pipe > 0 && n > wave;
  CK(ctx->arena.reserve(wave_words * 4 * (piped ? 2 : 1)));
  if (ctx->use_tma) {
    const int trc = ensure_tensor_maps(ctx, P, piped ? 2 : 1, wave_words, wave / 4);
    if (trc != HT_OK) return trc;
  }
  CK(cudaMemsetAsync(ctx->raw_count.as<uint32_t>() + f0, 0, sizeof(uint32_t) * n, st));
  if (ho.hist) CK(cudaMemsetAsync(ho.hist, 0, (size_t)n * 4096 * sizeof(uint32_t), st));
  // make this context's cascade the active __constant__ table (contexts with the same blob share it;
  // contexts with DIFFERENT cascades must not run concurrently on one device)
  if (g_loaded_cascade[ctx->cfg.device & 63] != ctx->hc.id) {
    CK(cudaDeviceSynchronize());   // kernels of other contexts may still be reading the previous table
    CK(cudaMemcpyToSymbolAsync(c_casc, &ctx->hc.cc, sizeof(ConstCascade), 0, cudaMemcpyHostToDevice, st));
    CK(cudaStreamSynchronize(st)); // ... and contexts sharing this cascade skip the upload, so it must have landed
    g_loaded_cascade[ctx->cfg.device & 63] = ctx->hc.id;
  }
  if (piped && !ctx->pipe_stream) {
    CK(cudaStreamCreateWithFlags(&ctx->pipe_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ctx->pipe_start, cudaEventDisableTiming));
    for (int i = 0; i < 4; ++i) CK(cudaEventCreateWithFlags(&ctx->pipe_events[i], cudaEventDisableTiming));
  }
  if (piped) {   // earlier work on the arena / frames is ordered before the first pyramid
    CK(cudaEventRecord(ctx->pipe_start, st));
    CK(cudaStreamWaitEvent(ctx->pipe_stream, ctx->pipe_start, 0));
  }
  const bool vec = (w % 4 == 0) && ((reinterpret_cast<uintptr_t>(d_rgba_batch) & 15u) == 0);
  int wi = 0;
  for (int w0 = 0; w0 < n; w0 += wave, ++wi) {
    const int nw = std::min(wave, n - w0), fa = f0 + w0, quads = (nw + 3) / 4;
    uint32_t *arena = ctx->arena.as<uint32_t>() + (piped ? (size_t)(wi & 1) * wave_words : 0);
    const uint8_t *d_rgba = d_rgba_batch + (size_t)fa * frame_bytes;
    const uint8_t *qm = quad_mask ? quad_mask + w0 / 4 : nullptr;   // (ht_stream_step) quads of this wave that have work
    cudaStream_t ps = piped ? ctx->pipe_stream : st;
    if (piped && wi >= 2) CK(cudaStreamWaitEvent(ps, ctx->pipe_events[2 + (wi & 1)], 0));   // cascade of wave wi-2 is done with this arena
    ctx->stream = ps;
    // K1 grayscale (+ histogram + bin plane) -> plane 0
    {
      const bool hist = ho.hist != nullptr;
      const int target = hist ? 592 : 1184;      // CTAs: 4 (32 KB of histograms each, register-limited) or 8 per SM
      int chunks = std::max(1, std::min(h, (target + quads - 1) / quads));
      if (hist) chunks = std::max(chunks, (w * h + 59999) / 60000);   // 16-bit histogram counters per CTA
      uint32_t *hp = hist ? ho.hist + (size_t)w0 * 4096 : nullptr;
      uint16_t *bp = ho.bins ? ho.bins + (size_t)w0 * w * h : nullptr;
      ctx->prof_begin(HT_PROF_GRAY);
      const dim3 grid((unsigned)chunks, (unsigned)quads);
      if (hist) {
        if (vec) k_gray<true, true><<<grid, 256, GRAY_HIST_SMEM, ps>>>(d_rgba, frame_bytes, nw, arena, P->arena_stride, w, h, P->planes[0].pitch, hp, bp, chunks, qm);
        else k_gray<false, true><<<grid, 256, GRAY_HIST_SMEM, ps>>>(d_rgba, frame_bytes, nw, arena, P->arena_stride, w, h, P->planes[0].pitch, hp, bp, chunks, qm);
      } else {
        if (vec) k_gray<true, false><<<grid, 256, 0, ps>>>(d_rgba, frame_bytes, nw, arena, P->arena_stride, w, h, P->planes[0].pitch, nullptr, nullptr, chunks, qm);
        else k_gray<false, false><<<grid, 256, 0, ps>>>(d_rgba, frame_bytes, nw, arena, P->arena_stride, w, h, P->planes[0].pitch, nullptr, nullptr, chunks, qm);
      }
      ctx->prof_end();
      ++ctx->launches;
    }
    // K2 pyramid generations
    for (size_t g = 1; g + 1 < P->gen_tile_begin.size(); ++g) {
      const int t0 = P->gen_tile_begin[g], t1 = P->gen_tile_begin[g + 1];
      if (t1 > t0) {
        ctx->prof_begin(HT_PROF_PYRAMID);
        k_resample<<<dim3(t1 - t0, quads), 256, 0, ps>>>(P->dplan, t0, arena, P->arena_stride, nw, qm);
        ctx->prof_end();
        ++ctx->launches;
      }
    }
    ctx->stream = st;
    if (piped) {
      CK(cudaEventRecord(ctx->pipe_events[wi & 1], ps));
      CK(cudaStreamWaitEvent(st, ctx->pipe_events[wi & 1], 0));
    }
    // K3 cascade
    if (!P->casc_tiles.empty()) {
      ctx->prof_begin(HT_PROF_CASCADE);
      auto kern = ctx->hc.fast ? k_cascade<true> : k_cascade<false>;
      kern<<<dim3((unsigned)P->casc_tiles.size(), quads), CASCADE_THREADS, CASC_SMEM, st>>>(
          P->dplan, ctx->d_casc.as<LateFeat>(), ctx->d_casc.as<LateFeat>() + ctx->hc.n_sched, ctx->d_late_chunk0.as<int32_t>(),
          (ctx->use_tma && ctx->d_tmaps.p) ? ctx->d_tmaps.as<uint8_t>() + (piped ? (size_t)(wi & 1) : 0) * P->scales.size() * 128 : nullptr, 0,
          arena, P->arena_stride, nw,
          ctx->raw_keys.as<uint32_t>() + (size_t)fa * ctx->raw_cap, ctx->raw_conf.as<double>() + (size_t)fa * ctx->raw_cap,
          ctx->raw_count.as<uint32_t>() + fa, ctx->raw_cap, ctx->force_ties, qm);
      ctx->prof_end();
      ++ctx->launches;
    }
    if (piped) CK(cudaEventRecord(ctx->pipe_events[2 + (wi & 1)], st));
    ctx->last_wave_f0 = fa;
    ctx->last_wave_n = nw;
    ctx->last_wave_arena = arena;
  }
  // K4 sort + group
  if (before_group) CK(cudaStreamWaitEvent(st, before_group, 0));   // (pipelined calls) the previous call's tracking still reads the rectangle arrays
  ctx->prof_begin(HT_PROF_GROUP);
  k_group<<<(n + 3) / 4, 128, 0, st>>>(P->dplan, n, ctx->raw_keys.as<uint32_t>() + (size_t)f0 * ctx->raw_cap,
                                       ctx->raw_conf.as<double>() + (size_t)f0 * ctx->raw_cap,
                                       ctx->raw_count.as<uint32_t>() + f0, ctx->raw_cap,
                                       ctx->sorted.as<Rect>() + (size_t)f0 * ctx->raw_cap,
                                       ctx->labels.as<int>() + (size_t)f0 * ctx->raw_cap,
                                       ctx->seq2.as<Rect>() + (size_t)f0 * ctx->raw_cap, min_neighbors,
                                       d_rects_batch + (size_t)f0 * ctx->K, d_counts_batch + f0, ctx->K,
                                       ctx->d_flags.as<int32_t>());
  ctx->prof_end();
  ++ctx->launches;
  CK(cudaGetLastError());
  return HT_OK;
}

// pick (optional) + initTracker + n_calls x track() for frames [f0, f0+n); slot of frame k is k (slots == NULL)
int run_track_from_detect(ht_ctx *ctx, const uint8_t *d_rgba_batch, int w, int h, int f0, int n, const Rect *d_det,
                          const int32_t *d_cnt, int calc_angles, int n_calls, int32_t *d_found, int32_t *d_objs,
                          int32_t *d_win) {
  cudaStream_t st = ctx->stream;
  const uint8_t *d_rgba = d_rgba_batch + (size_t)f0 * w * h * 4;
  int32_t *d_rects4 = ctx->d_rects.as<int32_t>() + 4 * (size_t)f0;
  ctx->prof_begin(HT_PROF_TRACK_INIT);
  k_pick_face<<<(n + 127) / 128, 128, 0, st>>>(d_det + (size_t)f0 * ctx->K, d_cnt + f0, ctx->K, n, d_rects4);
  k_track_init<<<n, 256, 0, st>>>(d_rgba, (size_t)w * h * 4, w, h, nullptr, d_rects4, calc_angles ? 1 : 0,
                                  ctx->model_hist.as<uint32_t>() + (size_t)f0 * 4096,
                                  ctx->track_state.as<TrackState>() + f0, d_found ? d_found + f0 : nullptr, nullptr);
  ctx->prof_end();
  ctx->launches += 2;
  if (n_calls > 0) {
    // the current-frame histograms and the bin plane were produced by the gray pass of run_detect (one frame read)
    uint16_t *bins = ctx->bins.as<uint16_t>() + ctx->bins_off + (size_t)f0 * w * h;
    ctx->prof_begin(HT_PROF_TRACK);
    int rc = launch_track(ctx, n, f0, bins, w, h, nullptr, ctx->model_hist.as<uint32_t>() + (size_t)f0 * 4096,
                      ctx->cur_hist.as<uint32_t>() + ctx->hist_off + (size_t)f0 * 4096, ctx->track_state.as<TrackState>() + f0, n_calls,
                      d_objs + 6 * (size_t)f0, d_win ? d_win + 4 * (size_t)f0 : nullptr, ctx->d_flags.as<int32_t>() + 2);
    if (rc != HT_OK) return rc;
    ctx->prof_end();
  }
  CK(cudaGetLastError());
  return HT_OK;
}

// Host frames -> ctx->d_frames in chunks on the copy stream; chunk c is complete when ctx->chunk_events[c] fires.
int upload_chunks(ht_ctx *ctx, const uint8_t *rgba, int n, size_t frame_bytes, int *chunk_out, int *n_chunks_out) {
  CK(ctx->d_frames.reserve(frame_bytes * (size_t)n));
  if (!ctx->copy_stream) {
    CK(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  }
  const int chunk = std::max(1, std::min(n, ctx->h2d_chunk));
  const int n_chunks = (n + chunk - 1) / chunk;
  while ((int)ctx->chunk_events.size() < n_chunks) {
    cudaEvent_t e;
    CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    ctx->chunk_events.push_back(e);
  }
  // the staging buffer may still be read by work enqueued earlier on the compute stream
  CK(cudaEventRecord(ctx->compute_done, ctx->stream));
  CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->compute_done, 0));
  uint8_t *d_frames = ctx->d_frames.as<uint8_t>();
  for (int c = 0; c < n_chunks; ++c) {
    const int f0 = c * chunk, nf = std::min(chunk, n - f0);
    CK(cudaMemcpyAsync(d_frames + frame_bytes * f0, rgba + frame_bytes * f0, frame_bytes * nf, cudaMemcpyHostToDevice,
                       ctx->copy_stream));
    CK(cudaEventRecord(ctx->chunk_events[c], ctx->copy_stream));
  }
  *chunk_out = chunk;
  *n_chunks_out = n_chunks;
  return HT_OK;
}

}  // namespace

// ================================================================================================
extern "C" {

uint32_t ht_version(void) { return (1u << 16) | 0u; }

const char *ht_last_error(const ht_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int ht_max_rects(const ht_ctx *ctx) { return ctx ? ctx->K : 0; }

uint64_t ht_launch_count(const ht_ctx *ctx) { return ctx ? ctx->launches : 0; }

int ht_create(ht_ctx **out, const ht_config *cfg, const void *cascade_blob, size_t blob_len) {
  if (!out || !cfg) { g_create_error = "ht_create: NULL argument"; return HT_ERR_ARG; }
  *out = nullptr;
  if (cfg->max_width <= 0 || cfg->max_height <= 0 || cfg->max_frames <= 0) { g_create_error = "ht_create: bad maxima"; return HT_ERR_ARG; }
  int n_dev = 0;
  if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) {
    cudaGetLastError();
    g_create_error = "ht_create: no CUDA device (this library has no CPU fallback)";
    return HT_ERR_CUDA;
  }
  if (cfg->device < 0 || cfg->device >= n_dev) { g_create_error = "ht_create: bad device ordinal"; return HT_ERR_ARG; }
  cudaDeviceProp prop{};
  if (cudaGetDeviceProperties(&prop, cfg->device) != cudaSuccess) { g_create_error = "ht_create: cudaGetDeviceProperties failed"; return HT_ERR_CUDA; }
  if (prop.major != 10) {
    g_create_error = "ht_create: device is sm_" + std::to_string(prop.major * 10 + prop.minor) + ", this build is sm_100a only";
    return HT_ERR_CUDA;
  }
  if (cudaSetDevice(cfg->device) != cudaSuccess) { g_create_error = "ht_create: cudaSetDevice failed"; return HT_ERR_CUDA; }
  std::unique_ptr<ht_ctx> c(new ht_ctx());
  c->cfg = *cfg;
  c->K = cfg->max_rects_per_frame > 0 ? cfg->max_rects_per_frame : 64;
  c->raw_cap = cfg->max_raw_per_frame > 0 ? cfg->max_raw_per_frame : 1024;
  std::string err;
  int rc = parse_cascade(cascade_blob, blob_len, c->hc, err);
  if (rc != HT_OK) { g_create_error = "ht_create: " + err; return rc; }
  if (cfg->cuda_stream) c->stream = static_cast<cudaStream_t>(cfg->cuda_stream);
  else {
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) { g_create_error = "ht_create: stream"; return HT_ERR_CUDA; }
    c->own_stream = true;
  }
  if (const char *tc = getenv("HT_TRACK_CLUSTER")) c->track_cluster = atoi(tc);
  if (const char *dp = getenv("HT_DETECT_PIPE")) c->detect_pipe = std::max(0, atoi(dp));
  if (const char *tm2 = getenv("HT_TRACK_MEMO")) c->track_memo = atoi(tm2) != 0;
  if (const char *tt = getenv("HT_TRACK_TRACE")) c->track_trace = atoi(tt) != 0;
  if (const char *tl = getenv("HT_TRACK_LPT")) c->track_lpt = atoi(tl) != 0;
  if (const char *th = getenv("HT_TRACK_HEAVY")) {
    c->track_heavy_div = std::max(0, atoi(th));
    if (const char *comma = strchr(th, ',')) {
      const int hc = atoi(comma + 1);
      if (hc == 2 || hc == 4 || hc == 8) c->track_heavy_cluster = hc;
    }
  }
  if (const char *tmid = getenv("HT_TRACK_MID")) {
    c->track_mid_div = std::max(0, atoi(tmid));
    if (const char *comma = strchr(tmid, ',')) {
      const int mc = atoi(comma + 1);
      if (mc == 2 || mc == 4 || mc == 8) c->track_mid_cluster = mc;
    }
  }
  if (const char *wv = getenv("HT_WAVE")) c->wave_frames = std::max(4, atoi(wv));
  if (const char *wm = getenv("HT_WAVE_MB")) c->wave_mb = std::max(1, atoi(wm));
  if (const char *tm = getenv("HT_TMA")) c->use_tma = atoi(tm) != 0;
  if (const char *ov = getenv("HT_OVERLAP")) { c->overlap_track = atoi(ov) != 0 ? 1 : 0; c->overlap_parts = atoi(ov); }
  if (const char *hc2 = getenv("HT_H2D_CHUNK")) c->h2d_chunk = std::max(1, atoi(hc2));
  if (const char *pl = getenv("HT_PIPELINE")) c->pipeline = atoi(pl) != 0 ? 1 : 0;
  if (const char *tk = getenv("HT_TRACK_MASK")) {   // HT_TRACK_MASK=<min n_calls>[,<min frames swept>]  (0: off / 0: every stream)
    c->track_mask_min = std::max(0, atoi(tk));
    if (const char *comma = strchr(tk, ',')) c->track_mask_frames = std::max(0, atoi(comma + 1));
  }
  if (cudaEventCreateWithFlags(&c->compute_done, cudaEventDisableTiming) != cudaSuccess) { g_create_error = "ht_create: event"; return HT_ERR_CUDA; }
  // the cascade image is copied into __constant__ memory lazily by run_detect; the late-stage table lives in HBM
  if (c->d_casc.reserve(c->hc.late.size() * sizeof(LateFeat)) != cudaSuccess ||
      cudaMemcpy(c->d_casc.p, c->hc.late.data(), c->hc.late.size() * sizeof(LateFeat), cudaMemcpyHostToDevice) != cudaSuccess ||
      c->d_late_chunk0.reserve(c->hc.late_chunk0.size() * sizeof(int32_t)) != cudaSuccess ||
      cudaMemcpy(c->d_late_chunk0.p, c->hc.late_chunk0.data(), c->hc.late_chunk0.size() * sizeof(int32_t), cudaMemcpyHostToDevice) != cudaSuccess) {
    g_create_error = "ht_create: cascade upload failed"; return HT_ERR_CUDA;
  }
  if (set_kernel_attributes(c.get()) != HT_OK) { g_create_error = "ht_create: " + c->err; return HT_ERR_CUDA; }
  // per-frame result buffers
  const size_t mf = (size_t)cfg->max_frames;
  bool ok = c->raw_keys.reserve(mf * c->raw_cap * sizeof(uint32_t)) == cudaSuccess &&
            c->raw_conf.reserve(mf * c->raw_cap * sizeof(double)) == cudaSuccess &&
            c->raw_count.reserve(mf * sizeof(uint32_t)) == cudaSuccess &&
            c->sorted.reserve(mf * c->raw_cap * sizeof(Rect)) == cudaSuccess &&
            c->labels.reserve(mf * c->raw_cap * sizeof(int)) == cudaSuccess &&
            c->seq2.reserve(mf * c->raw_cap * sizeof(Rect)) == cudaSuccess &&
            c->d_out_rects.reserve(mf * c->K * sizeof(Rect)) == cudaSuccess &&
            c->d_out_counts.reserve(mf * sizeof(int32_t)) == cudaSuccess &&
            c->d_flags.reserve(256) == cudaSuccess;
  if (!ok) { g_create_error = "ht_create: cudaMalloc failed"; return HT_ERR_CUDA; }
  cudaMemset(c->d_flags.p, 0, 256);
  cudaMemset(c->raw_count.p, 0, mf * sizeof(uint32_t));
  *out = c.release();
  return HT_OK;
}

void ht_destroy(ht_ctx *ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->cfg.device);
  if (ctx->aux_stream) cudaStreamSynchronize(ctx->aux_stream);
  cudaStreamSynchronize(ctx->stream);
  for (auto &kv : ctx->plans) kv.second->dev.release();
  DevBuf *bufs[] = {&ctx->d_casc, &ctx->arena, &ctx->d_frames, &ctx->raw_keys, &ctx->raw_conf, &ctx->raw_count, &ctx->sorted,
                    &ctx->labels, &ctx->seq2, &ctx->d_out_rects, &ctx->d_out_counts, &ctx->d_flags, &ctx->model_hist,
                    &ctx->bins, &ctx->d_sched, &ctx->d_trace, &ctx->d_tmaps, &ctx->d_late_chunk0, &ctx->d_track_cost, &ctx->d_stream_mode, &ctx->d_stream_mask, &ctx->d_stream_cs, &ctx->d_stream_init, &ctx->d_stream_events, &ctx->d_head_state, &ctx->d_head_params, &ctx->d_head_events, &ctx->cur_hist, &ctx->track_state, &ctx->d_slots, &ctx->d_rects, &ctx->d_found, &ctx->d_objs,
                    &ctx->d_windows, &ctx->d_wb_sums, &ctx->d_wb_out, &ctx->d_scratch};
  for (DevBuf *b : bufs) b->release();
  for (auto &sp : ctx->prof_spans) { cudaEventDestroy(sp.a); cudaEventDestroy(sp.b); }
  for (cudaEvent_t e : ctx->prof_free) cudaEventDestroy(e);
  for (cudaEvent_t e : ctx->chunk_events) cudaEventDestroy(e);
  if (ctx->compute_done) cudaEventDestroy(ctx->compute_done);
  if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
  if (ctx->pipe_stream) cudaStreamDestroy(ctx->pipe_stream);
  if (ctx->pipe_start) cudaEventDestroy(ctx->pipe_start);
  for (cudaEvent_t e : ctx->pipe_events) if (e) cudaEventDestroy(e);
  for (int t = 0; t < 3; ++t) {
    if (ctx->tier_stream[t]) cudaStreamDestroy(ctx->tier_stream[t]);
    if (ctx->tier_done[t]) cudaEventDestroy(ctx->tier_done[t]);
  }
  if (ctx->sched_ready) cudaEventDestroy(ctx->sched_ready);
  if (ctx->aux_stream) cudaStreamDestroy(ctx->aux_stream);
  if (ctx->aux_done) cudaEventDestroy(ctx->aux_done);
  if (ctx->pipe_detect_done) cudaEventDestroy(ctx->pipe_detect_done);
  for (cudaEvent_t e : ctx->part_events) if (e) cudaEventDestroy(e);
  if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
  delete ctx;
}

int ht_sync(ht_ctx *ctx) {
  if (!ctx) return HT_ERR_ARG;
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  CK(cudaStreamSynchronize(ctx->stream));
  int32_t flags[2] = {0, 0};
  CK(cudaMemcpy(flags, ctx->d_flags.p, sizeof(flags), cudaMemcpyDeviceToHost));
  if (flags[0] || flags[1]) {
    CK(cudaMemset(ctx->d_flags.p, 0, sizeof(flags)));
    if (flags[1]) return ctx->fail(HT_ERR_STATE, "ht_track on a tracker slot that was never initialised");
    return ctx->fail(HT_WARN_OVERFLOW, "a per-frame detection list overflowed its capacity (raw %d / K %d) and was truncated",
                     ctx->raw_cap, ctx->K);
  }
  return HT_OK;
}

int ht_detect(ht_ctx *ctx, const uint8_t *rgba, int n, int w, int h, int interval, int min_neighbors,
              ht_rect *out_rects, int32_t *out_counts) {
  if (!ctx) return HT_ERR_ARG;
  if (!out_rects || !out_counts) return ctx->fail(HT_ERR_ARG, "output pointers are NULL");
  int rc = check_batch(ctx, n);
  if (rc != HT_OK) return rc;
  CK(cudaSetDevice(ctx->cfg.device));
  Plan *P = nullptr;
  rc = get_plan(ctx, w, h, interval, &P);
  if (rc != HT_OK) return rc;
  if (!rgba) return ctx->fail(HT_ERR_ARG, "rgba is NULL");
  if ((reinterpret_cast<uintptr_t>(rgba) & 3u) != 0) return ctx->fail(HT_ERR_ARG, "rgba must be 4-byte aligned");
  cudaStream_t st = ctx->stream;
  const bool rects_dev = is_device_ptr(out_rects), counts_dev = is_device_ptr(out_counts);
  Rect *d_rects = rects_dev ? reinterpret_cast<Rect *>(out_rects) : ctx->d_out_rects.as<Rect>();
  int32_t *d_counts = counts_dev ? out_counts : ctx->d_out_counts.as<int32_t>();
  if (is_device_ptr(rgba)) {
    rc = run_detect(ctx, P, rgba, 0, n, min_neighbors, d_rects, d_counts);
    if (rc != HT_OK) return rc;
  } else {
    // host frames: the H2D of chunk c+1 (copy stream) overlaps the kernels of chunk c
    int chunk = 0, n_chunks = 0;
    rc = upload_chunks(ctx, rgba, n, (size_t)w * h * 4, &chunk, &n_chunks);
    if (rc != HT_OK) return rc;
    for (int c = 0; c < n_chunks; ++c) {
      const int f0 = c * chunk, nf = std::min(chunk, n - f0);
      CK(cudaStreamWaitEvent(st, ctx->chunk_events[c], 0));
      rc = run_detect(ctx, P, ctx->d_frames.as<uint8_t>(), f0, nf, min_neighbors, d_rects, d_counts);
      if (rc != HT_OK) return rc;
    }
  }
  ctx->last_plan = P;
  ctx->last_n = n;
  if (!rects_dev) CK(cudaMemcpyAsync(out_rects, d_rects, sizeof(Rect) * (size_t)n * ctx->K, cudaMemcpyDeviceToHost, st));
  if (!counts_dev) CK(cudaMemcpyAsync(out_counts, d_counts, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st));
  if (!rects_dev || !counts_dev) return ht_sync(ctx);
  return HT_OK;
}

int ht_track_init(ht_ctx *ctx, const int32_t *slots, int n, const uint8_t *rgba, int w, int h, const int32_t *rects,
                  int calc_angles) {
  if (!ctx) return HT_ERR_ARG;
  if (!rects) return ctx->fail(HT_ERR_ARG, "rects is NULL");
  int rc = check_batch(ctx, n);
  if (rc != HT_OK) return rc;
  if (w <= 0 || h <= 0) return ctx->fail(HT_ERR_ARG, "bad frame size");
  CK(cudaSetDevice(ctx->cfg.device));
  rc = ensure_tracker_buffers(ctx);
  if (rc != HT_OK) return rc;
  const uint8_t *d_rgba = nullptr;
  rc = device_frames(ctx, rgba, n, w, h, &d_rgba);
  if (rc != HT_OK) return rc;
  const int32_t *d_rects = rects;
  if (!is_device_ptr(rects)) {
    for (int i = 0; i < n; ++i)
      if (rects[4 * i + 2] <= 0 || rects[4 * i + 3] <= 0)
        return ctx->fail(HT_ERR_ARG, "initTracker rectangle %d is empty (canvas getImageData would throw)", i);
    CK(cudaMemcpyAsync(ctx->d_rects.p, rects, sizeof(int32_t) * 4 * n, cudaMemcpyHostToDevice, ctx->stream));
    d_rects = ctx->d_rects.as<int32_t>();
  }
  return track_init_common(ctx, slots, n, d_rgba, w, h, d_rects, calc_angles, nullptr);
}

int ht_track_init_from_detect(ht_ctx *ctx, const int32_t *slots, int n, const uint8_t *rgba, int w, int h,
                              const ht_rect *det_rects, const int32_t *det_counts, int calc_angles, int32_t *out_found) {
  if (!ctx) return HT_ERR_ARG;
  if (!det_rects || !det_counts) return ctx->fail(HT_ERR_ARG, "detection outputs are NULL");
  int rc = check_batch(ctx, n);
  if (rc != HT_OK) return rc;
  if (w <= 0 || h <= 0) return ctx->fail(HT_ERR_ARG, "bad frame size");
  CK(cudaSetDevice(ctx->cfg.device));
  rc = ensure_tracker_buffers(ctx);
  if (rc != HT_OK) return rc;
  const uint8_t *d_rgba = nullptr;
  rc = device_frames(ctx, rgba, n, w, h, &d_rgba);
  if (rc != HT_OK) return rc;
  const Rect *d_det = reinterpret_cast<const Rect *>(det_rects);
  const int32_t *d_cnt = det_counts;
  if (!is_device_ptr(det_rects)) {
    CK(cudaMemcpyAsync(ctx->d_out_rects.p, det_rects, sizeof(Rect) * (size_t)n * ctx->K, cudaMemcpyHostToDevice, ctx->stream));
    d_det = ctx->d_out_rects.as<Rect>();
  }
  if (!is_device_ptr(det_counts)) {
    CK(cudaMemcpyAsync(ctx->d_out_counts.p, det_counts, sizeof(int32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
    d_cnt = ctx->d_out_counts.as<int32_t>();
  }
  ctx->prof_begin(HT_PROF_TRACK_INIT);
  k_pick_face<<<(n + 127) / 128, 128, 0, ctx->stream>>>(d_det, d_cnt, ctx->K, n, ctx->d_rects.as<int32_t>());
  ctx->prof_end();
  ++ctx->launches;
  CK(cudaGetLastError());
  return track_init_common(ctx, slots, n, d_rgba, w, h, ctx->d_rects.as<int32_t>(), calc_angles, out_found);
}

int ht_track(ht_ctx *ctx, const int32_t *slots, int n, const uint8_t *rgba, int w, int h, int n_calls,
             ht_trackobj *out_objs, ht_window *out_windows) {
  if (!ctx) return HT_ERR_ARG;
  if (!out_objs) return ctx->fail(HT_ERR_ARG, "out_objs is NULL");
  if (n_calls < 1) return ctx->fail(HT_ERR_ARG, "n_calls must be >= 1");
  int rc = check_batch(ctx, n);
  if (rc != HT_OK) return rc;
  if (w <= 0 || h <= 0) return ctx->fail(HT_ERR_ARG, "bad frame size");
  CK(cudaSetDevice(ctx->cfg.device));
  rc = ensure_tracker_buffers(ctx);
  if (rc != HT_OK) return rc;
  const uint8_t *d_rgba = nullptr;
  rc = device_frames(ctx, rgba, n, w, h, &d_rgba);
  if (rc != HT_OK) return rc;
  const int32_t *d_slots = nullptr;
  rc = upload_slots(ctx, slots, n, &d_slots);
  if (rc != HT_OK) return rc;
  CK(ctx->bins.reserve((size_t)n * w * h * sizeof(uint16_t)));
  rc = launch_hist(ctx, d_rgba, n, w, h, ctx->cur_hist.as<uint32_t>(), ctx->bins.as<uint16_t>());   // camshift.js:268
  if (rc != HT_OK) return rc;
  const bool objs_dev = is_device_ptr(out_objs), win_dev = out_windows && is_device_ptr(out_windows);
  int32_t *d_objs = objs_dev ? reinterpret_cast<int32_t *>(out_objs) : ctx->d_objs.as<int32_t>();
  int32_t *d_win = out_windows ? (win_dev ? reinterpret_cast<int32_t *>(out_windows) : ctx->d_windows.as<int32_t>()) : nullptr;
  ctx->prof_begin(HT_PROF_TRACK);
  rc = launch_track(ctx, n, 0, ctx->bins.as<uint16_t>(), w, h, d_slots, ctx->model_hist.as<uint32_t>(),
                    ctx->cur_hist.as<uint32_t>(), ctx->track_state.as<TrackState>(), n_calls, d_objs, d_win,
                    ctx->d_flags.as<int32_t>() + 1);
  if (rc != HT_OK) return rc;
  ctx->prof_end();
  CK(cudaGetLastError());
  if (!objs_dev) CK(cudaMemcpyAsync(out_objs, d_objs, sizeof(ht_trackobj) * n, cudaMemcpyDeviceToHost, ctx->stream));
  if (out_windows && !win_dev) CK(cudaMemcpyAsync(out_windows, d_win, sizeof(ht_window) * n, cudaMemcpyDeviceToHost, ctx->stream));
  if (!objs_dev || (out_windows && !win_dev)) return ht_sync(ctx);
  return HT_OK;
}

int ht_detect_track(ht_ctx *ctx, const uint8_t *rgba, int n, int w, int h, int interval, int min_neighbors,
                    int calc_angles, int n_calls, ht_rect *out_rects, int32_t *out_counts, int32_t *out_found,
                    ht_trackobj *out_objs, ht_window *out_windows) {
  if (!ctx) return HT_ERR_ARG;
  if (!out_rects || !out_counts || !out_objs) return ctx->fail(HT_ERR_ARG, "output pointers are NULL");
  if (n_calls < 0) return ctx->fail(HT_ERR_ARG, "n_calls must be >= 0");
  const bool rects_dev = is_device_ptr(out_rects), counts_dev = is_device_ptr(out_counts);
  const bool found_dev = out_found && is_device_ptr(out_found), objs_dev = is_device_ptr(out_objs);
  const bool win_dev = out_windows && is_device_ptr(out_windows);
  // pipelined call (ht_set_pipeline): everything stays on the device, so nothing forces this call to wait for its own
  // tracking - it is left on the aux stream and runs under the next call's detection
  const bool deferred = ctx->pipeline > 0 && n_calls > 0 && rgba && is_device_ptr(rgba) && rects_dev && counts_dev && objs_dev &&
                        (!out_found || found_dev) && (!out_windows || win_dev);
  int rc = check_batch(ctx, n, !deferred);
  if (rc != HT_OK) return rc;
  CK(cudaSetDevice(ctx->cfg.device));
  Plan *P = nullptr;
  rc = get_plan(ctx, w, h, interval, &P);
  if (rc != HT_OK) return rc;
  rc = ensure_tracker_buffers(ctx);
  if (rc != HT_OK) return rc;
  cudaStream_t st = ctx->stream;
  if (deferred) {
    const size_t plane_elems = (size_t)ctx->cfg.max_frames * w * h;     // one parity's bin planes
    if (ctx->bins.cap < 2 * plane_elems * sizeof(uint16_t)) {
      if (ctx->aux_stream) CK(cudaStreamSynchronize(ctx->aux_stream));   // the buffer about to be replaced may still be read
      CK(cudaStreamSynchronize(st));
      CK(ctx->bins.reserve(2 * plane_elems * sizeof(uint16_t)));
    }
    if (!ctx->aux_stream) {
      int prio_least = 0, prio_greatest = 0;
      CK(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
      CK(cudaStreamCreateWithPriority(&ctx->aux_stream, cudaStreamNonBlocking, prio_greatest));
      CK(cudaEventCreateWithFlags(&ctx->aux_done, cudaEventDisableTiming));
      for (int i = 0; i < 4; ++i) CK(cudaEventCreateWithFlags(&ctx->part_events[i], cudaEventDisableTiming));
    }
    if (!ctx->pipe_detect_done) CK(cudaEventCreateWithFlags(&ctx->pipe_detect_done, cudaEventDisableTiming));
    ctx->pipe_parity ^= 1;
    ctx->bins_off = (size_t)ctx->pipe_parity * plane_elems;
    ctx->hist_off = (size_t)ctx->pipe_parity * (size_t)ctx->cfg.max_frames * 4096;
    Rect *dr = reinterpret_cast<Rect *>(out_rects);
    rc = run_detect(ctx, P, rgba, 0, n, min_neighbors, dr, out_counts,
                    HistOut{ctx->cur_hist.as<uint32_t>() + ctx->hist_off, ctx->bins.as<uint16_t>() + ctx->bins_off}, nullptr,
                    ctx->aux_pending ? ctx->aux_done : nullptr);
    if (rc != HT_OK) return rc;
    CK(cudaEventRecord(ctx->pipe_detect_done, st));
    CK(cudaStreamWaitEvent(ctx->aux_stream, ctx->pipe_detect_done, 0));
    ctx->stream = ctx->aux_stream;
    rc = run_track_from_detect(ctx, rgba, w, h, 0, n, dr, out_counts, calc_angles, n_calls, out_found,
                               reinterpret_cast<int32_t *>(out_objs), reinterpret_cast<int32_t *>(out_windows));
    ctx->stream = st;
    if (rc != HT_OK) return rc;
    CK(cudaEventRecord(ctx->aux_done, ctx->aux_stream));
    ctx->aux_pending = true;
    ctx->last_plan = P;
    ctx->last_n = n;
    return HT_OK;
  }
  if (n_calls > 0) CK(ctx->bins.reserve((size_t)n * w * h * sizeof(uint16_t)));
  Rect *d_rects = rects_dev ? reinterpret_cast<Rect *>(out_rects) : ctx->d_out_rects.as<Rect>();
  int32_t *d_counts = counts_dev ? out_counts : ctx->d_out_counts.as<int32_t>();
  int32_t *d_found = out_found ? (found_dev ? out_found : ctx->d_found.as<int32_t>()) : nullptr;
  int32_t *d_objs = objs_dev ? reinterpret_cast<int32_t *>(out_objs) : ctx->d_objs.as<int32_t>();
  int32_t *d_win = out_windows ? (win_dev ? reinterpret_cast<int32_t *>(out_windows) : ctx->d_windows.as<int32_t>()) : nullptr;
  if (n_calls == 0) CK(cudaMemsetAsync(d_objs, 0, sizeof(ht_trackobj) * n, st));
  if (!rgba) return ctx->fail(HT_ERR_ARG, "rgba is NULL");
  if ((reinterpret_cast<uintptr_t>(rgba) & 3u) != 0) return ctx->fail(HT_ERR_ARG, "rgba must be 4-byte aligned");
  const size_t frame_bytes = (size_t)w * h * 4;
  // Detect and track have complementary bottlenecks (k_cascade: shared-memory load wavefronts; k_track: a latency
  // chain of fp64 window passes with < 20 % LSU use), so the batch is cut into parts and the tracking of part p
  // runs on a second stream while part p+1 is being detected.
  // (Tracking host-frame parts on the main stream as their chunks arrive was also measured: e2e 27.3k vs 33.6k fps
  // for one k_track over the whole batch — every k_track launch costs at least its slowest stream.)
  const bool use_aux = n_calls > 0 && (ctx->overlap_track > 0 || (ctx->overlap_track < 0 && !is_device_ptr(rgba)));
  int parts = use_aux ? ((n >= 512) ? 4 : (n >= 128 ? 2 : 1)) : 1;
  if (use_aux && ctx->overlap_parts > 1) parts = std::min(ctx->overlap_parts, std::max(1, n / 32));
  auto part_begin = [&](int p) { return (int)(((long long)n * p) / parts); };
  auto hist_out = [&](int f0) {
    return n_calls > 0 ? HistOut{ctx->cur_hist.as<uint32_t>() + ctx->hist_off + (size_t)f0 * 4096,
                                 ctx->bins.as<uint16_t>() + ctx->bins_off + (size_t)f0 * w * h}
                       : HistOut{nullptr, nullptr};
  };
  if (use_aux && parts > 1 && !ctx->aux_stream) {
    CK(cudaStreamCreateWithFlags(&ctx->aux_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&ctx->aux_done, cudaEventDisableTiming));
    for (int i = 0; i < 4; ++i) CK(cudaEventCreateWithFlags(&ctx->part_events[i], cudaEventDisableTiming));
  }
  // run tracking for frames [f0, f0+nf) — on the aux stream when overlapping
  auto track_part = [&](const uint8_t *d_frames_batch, int f0, int nf) -> int {
    if (parts == 1 || !use_aux) return run_track_from_detect(ctx, d_frames_batch, w, h, f0, nf, d_rects, d_counts, calc_angles, n_calls, d_found, d_objs, d_win);
    const int pi = ctx->part_seq++ & 3;
    CK(cudaEventRecord(ctx->part_events[pi], st));
    CK(cudaStreamWaitEvent(ctx->aux_stream, ctx->part_events[pi], 0));
    cudaStream_t saved = ctx->stream;
    ctx->stream = ctx->aux_stream;
    const int r = run_track_from_detect(ctx, d_frames_batch, w, h, f0, nf, d_rects, d_counts, calc_angles, n_calls, d_found, d_objs, d_win);
    ctx->stream = saved;
    return r;
  };
  if (is_device_ptr(rgba)) {
    for (int p = 0; p < parts; ++p) {
      const int f0 = part_begin(p), nf = part_begin(p + 1) - f0;
      rc = run_detect(ctx, P, rgba, f0, nf, min_neighbors, d_rects, d_counts, hist_out(f0));
      if (rc != HT_OK) return rc;
      rc = track_part(rgba, f0, nf);
      if (rc != HT_OK) return rc;
    }
  } else {
    // host frames: upload in chunks on a copy stream so the H2D of chunk c+1 overlaps the kernels of chunk c
    int chunk = 0, n_chunks = 0;
    rc = upload_chunks(ctx, rgba, n, frame_bytes, &chunk, &n_chunks);
    if (rc != HT_OK) return rc;
    uint8_t *d_frames = ctx->d_frames.as<uint8_t>();
    // detect per uploaded chunk; tracking per PART (a k_track launch costs at least its slowest stream, so it is
    // not launched per chunk)
    int next_part = 0, tracked_to = 0;
    for (int c = 0; c < n_chunks; ++c) {
      const int f0 = c * chunk, nf = std::min(chunk, n - f0);
      CK(cudaStreamWaitEvent(st, ctx->chunk_events[c], 0));
      rc = run_detect(ctx, P, d_frames, f0, nf, min_neighbors, d_rects, d_counts, hist_out(f0));
      if (rc != HT_OK) return rc;
      const int done_to = f0 + nf;
      while (next_part < parts && part_begin(next_part + 1) <= done_to) {
        const int pb = part_begin(next_part), pe = part_begin(next_part + 1);
        if (pe > pb) { rc = track_part(d_frames, pb, pe - pb); if (rc != HT_OK) return rc; }
        tracked_to = pe;
        ++next_part;
      }
    }
    if (tracked_to < n) { rc = track_part(d_frames, tracked_to, n - tracked_to); if (rc != HT_OK) return rc; }
  }
  if (use_aux && parts > 1) {   // join: results of the aux stream are complete before anything later on the main stream
    CK(cudaEventRecord(ctx->aux_done, ctx->aux_stream));
    CK(cudaStreamWaitEvent(st, ctx->aux_done, 0));
  }
  ctx->last_plan = P;
  ctx->last_n = n;
  bool any_host = false;
  if (!rects_dev) { CK(cudaMemcpyAsync(out_rects, d_rects, sizeof(Rect) * (size_t)n * ctx->K, cudaMemcpyDeviceToHost, st)); any_host = true; }
  if (!counts_dev) { CK(cudaMemcpyAsync(out_counts, d_counts, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st)); any_host = true; }
  if (out_found && !found_dev) { CK(cudaMemcpyAsync(out_found, d_found, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st)); any_host = true; }
  if (!objs_dev) { CK(cudaMemcpyAsync(out_objs, d_objs, sizeof(ht_trackobj) * n, cudaMemcpyDeviceToHost, st)); any_host = true; }
  if (out_windows && !win_dev) { CK(cudaMemcpyAsync(out_windows, d_win, sizeof(ht_window) * n, cudaMemcpyDeviceToHost, st)); any_host = true; }
  if (any_host) return ht_sync(ctx);
  return HT_OK;
}

static_assert(sizeof(ht_stream_event) == sizeof(StreamEvent) && sizeof(ht_stream_event) == 56, "ht_stream_event layout");
static_assert(sizeof(ht_head_event) == sizeof(HeadEvent) && sizeof(ht_head_event) == 64, "ht_head_event layout");
static_assert(sizeof(ht_head_params) == 48, "ht_head_params layout");

__global__ void k_head_reset(HeadState *s, int first, int n) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) head_new_state(s[first + k]);
}

static HeadParams make_head_params(const ht_head_params *p) {
  HeadParams hp{};
  hp.smoothing = p->smoothing; hp.head_position = p->head_position; hp.edgecorrection = p->edgecorrection;
  hp.alpha = p->alpha; hp.fov_deg = p->fov_deg; hp.camera_offset = p->camera_offset; hp.distance_to_screen = p->distance_to_screen;
  const double head_width_cm = 16, head_height_cm = 19;                       // src/headposition.js:53-63
  const double hsa = std::atan(head_width_cm / head_height_cm);
  hp.head_diag_cm = std::sqrt((head_width_cm * head_width_cm) + (head_height_cm * head_height_cm));
  hp.sin_hsa = std::sin(hsa); hp.cos_hsa = std::cos(hsa); hp.tan_hsa = std::tan(hsa);
  return hp;
}

int ht_stream_head_config(ht_ctx *ctx, const ht_head_params *params) {
  if (!ctx) return HT_ERR_ARG;
  CK(cudaSetDevice(ctx->cfg.device));
  if (!params) { ctx->head_on = false; return HT_OK; }
  if (!(params->alpha >= 0.0 && params->alpha <= 1.0) || !(params->distance_to_screen > 0.0)) return ctx->fail(HT_ERR_ARG, "bad head parameters");
  const size_t mf = (size_t)ctx->cfg.max_frames;
  if (!ctx->d_head_state.p) {
    CK(ctx->d_head_state.reserve(mf * sizeof(HeadState)));
    CK(ctx->d_head_params.reserve(sizeof(HeadParams)));
    CK(ctx->d_head_events.reserve(mf * sizeof(HeadEvent)));
    k_head_reset<<<(unsigned)((mf + 127) / 128), 128, 0, ctx->stream>>>(ctx->d_head_state.as<HeadState>(), 0, (int)mf);
  }
  const HeadParams hp = make_head_params(params);
  CK(cudaMemcpyAsync(ctx->d_head_params.p, &hp, sizeof(hp), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));    // `hp` is a local
  ctx->head_on = true;
  return HT_OK;
}


static int ensure_stream_buffers(ht_ctx *ctx) {
  const size_t mf = (size_t)ctx->cfg.max_frames;
  if (!ctx->d_stream_mode.p) {
    CK(ctx->d_stream_mode.reserve(mf * sizeof(int32_t)));
    CK(cudaMemsetAsync(ctx->d_stream_mode.p, 0, mf * sizeof(int32_t), ctx->stream));   // every stream starts in "VJ"
    CK(ctx->d_stream_mask.reserve((mf + 3) / 4 + 16));
    CK(ctx->d_stream_cs.reserve(mf));
    CK(ctx->d_stream_init.reserve(mf));
    CK(ctx->d_stream_events.reserve(mf * sizeof(StreamEvent)));
  }
  return HT_OK;
}

int ht_stream_reset(ht_ctx *ctx, int first, int n) {
  if (!ctx) return HT_ERR_ARG;
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  if (first < 0 || n <= 0 || first + n > ctx->cfg.max_frames) return ctx->fail(HT_ERR_ARG, "stream range outside [0,%d)", ctx->cfg.max_frames);
  CK(cudaSetDevice(ctx->cfg.device));
  int rc = ensure_stream_buffers(ctx);
  if (rc != HT_OK) return rc;
  CK(cudaMemsetAsync(ctx->d_stream_mode.as<int32_t>() + first, 0, (size_t)n * sizeof(int32_t), ctx->stream));
  if (ctx->d_head_state.p)   // a new headtrackr.Tracker: smoother, head diagonals, fov estimate start over too
    k_head_reset<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ctx->d_head_state.as<HeadState>(), first, n);
  return HT_OK;
}

// One frame of n independent streams through facetrackr's state machine, entirely on the device:
//   streams in "VJ": gray + pyramid + cascade + grouping on their frame (masked frame quads), max-confidence pick,
//                    confidence gate, initTracker on the same frame, switch to "CS"        src/facetrackr.js:67-126,137-175
//   streams in "CS": histogram + one camshift track() on their frame; a 0-sized result switches the stream back to
//                    "VJ" for the next frame                                                src/facetrackr.js:178-209, src/main.js:230-244
// No host round trip between the kernels; the host only drains the event records.
int ht_stream_step(ht_ctx *ctx, const uint8_t *rgba, int n, int w, int h, int interval, int min_neighbors, int calc_angles,
                   ht_stream_event *out_events) {
  return ht_stream_step_head(ctx, rgba, n, w, h, interval, min_neighbors, calc_angles, out_events, nullptr);
}

int ht_stream_step_head(ht_ctx *ctx, const uint8_t *rgba, int n, int w, int h, int interval, int min_neighbors, int calc_angles,
                        ht_stream_event *out_events, ht_head_event *out_head) {
  if (!ctx) return HT_ERR_ARG;
  if (!out_events) return ctx->fail(HT_ERR_ARG, "out_events is NULL");
  if (out_head && !ctx->head_on) return ctx->fail(HT_ERR_STATE, "ht_stream_head_config has not been called");
  int rc = check_batch(ctx, n);
  if (rc != HT_OK) return rc;
  CK(cudaSetDevice(ctx->cfg.device));
  Plan *P = nullptr;
  rc = get_plan(ctx, w, h, interval, &P);
  if (rc != HT_OK) return rc;
  rc = ensure_tracker_buffers(ctx);
  if (rc != HT_OK) return rc;
  rc = ensure_stream_buffers(ctx);
  if (rc != HT_OK) return rc;
  const uint8_t *d_rgba = nullptr;
  rc = device_frames(ctx, rgba, n, w, h, &d_rgba);
  if (rc != HT_OK) return rc;
  CK(ctx->bins.reserve((size_t)n * w * h * sizeof(uint16_t)));
  cudaStream_t st = ctx->stream;
  int32_t *mode = ctx->d_stream_mode.as<int32_t>();
  uint8_t *vj_mask = ctx->d_stream_mask.as<uint8_t>(), *cs_en = ctx->d_stream_cs.as<uint8_t>(), *init_en = ctx->d_stream_init.as<uint8_t>();
  k_stream_plan<<<(n + 127) / 128, 128, 0, st>>>(mode, n, vj_mask, cs_en, init_en);
  ++ctx->launches;
  // detection for the streams in "VJ" (frame quads without such a stream exit at once)
  rc = run_detect(ctx, P, d_rgba, 0, n, min_neighbors, ctx->d_out_rects.as<Rect>(), ctx->d_out_counts.as<int32_t>(),
                  HistOut{nullptr, nullptr}, vj_mask);
  if (rc != HT_OK) return rc;
  // one track() for the streams in "CS" (src/camshift.js:213-312; the whole-frame histogram is :268)
  rc = launch_hist(ctx, d_rgba, n, w, h, ctx->cur_hist.as<uint32_t>(), ctx->bins.as<uint16_t>(), cs_en);
  if (rc != HT_OK) return rc;
  ctx->prof_begin(HT_PROF_TRACK);
  rc = launch_track(ctx, n, 0, ctx->bins.as<uint16_t>(), w, h, nullptr, ctx->model_hist.as<uint32_t>(),
                    ctx->cur_hist.as<uint32_t>(), ctx->track_state.as<TrackState>(), 1, ctx->d_objs.as<int32_t>(), nullptr,
                    ctx->d_flags.as<int32_t>() + 2, cs_en);
  if (rc != HT_OK) return rc;
  ctx->prof_end();
  // events + transitions, then initTracker for the streams that just found their face
  StreamEvent *d_ev = is_device_ptr(out_events) ? reinterpret_cast<StreamEvent *>(out_events) : ctx->d_stream_events.as<StreamEvent>();
  HeadEvent *d_he = nullptr;
  if (ctx->head_on) d_he = (out_head && is_device_ptr(out_head)) ? reinterpret_cast<HeadEvent *>(out_head) : ctx->d_head_events.as<HeadEvent>();
  k_stream_update<<<(n + 127) / 128, 128, 0, st>>>(mode, n, ctx->d_out_rects.as<Rect>(), ctx->d_out_counts.as<int32_t>(), ctx->K,
                                                   ctx->d_objs.as<int32_t>(), ctx->d_rects.as<int32_t>(), init_en, d_ev,
                                                   ctx->head_on ? ctx->d_head_state.as<HeadState>() : nullptr,
                                                   ctx->d_head_params.as<HeadParams>(), d_he, w, h);
  ctx->prof_begin(HT_PROF_TRACK_INIT);
  k_track_init<<<n, 256, 0, st>>>(d_rgba, (size_t)w * h * 4, w, h, nullptr, ctx->d_rects.as<int32_t>(), calc_angles ? 1 : 0,
                                  ctx->model_hist.as<uint32_t>(), ctx->track_state.as<TrackState>(), nullptr, init_en);
  ctx->prof_end();
  ctx->launches += 2;
  CK(cudaGetLastError());
  ctx->last_plan = P;
  ctx->last_n = n;
  bool any_host = false;
  if (!is_device_ptr(out_events)) { CK(cudaMemcpyAsync(out_events, d_ev, sizeof(StreamEvent) * (size_t)n, cudaMemcpyDeviceToHost, st)); any_host = true; }
  if (out_head && !is_device_ptr(out_head)) { CK(cudaMemcpyAsync(out_head, d_he, sizeof(HeadEvent) * (size_t)n, cudaMemcpyDeviceToHost, st)); any_host = true; }
  if (any_host) return ht_sync(ctx);
  return HT_OK;
}

// canvasContext.drawImage(video, 0, 0, canvas.width, canvas.height) for n frames (src/main.js:170)
int ht_ingest(ht_ctx *ctx, const uint8_t *src_rgba, int n, int sw, int sh, uint8_t *dst_rgba, int dw, int dh) {
  if (!ctx) return HT_ERR_ARG;
  if (!src_rgba || !dst_rgba || n <= 0 || sw <= 0 || sh <= 0) return ctx->fail(HT_ERR_ARG, "bad argument");
  if (dw <= 0 || dh <= 0) return ctx->fail(HT_ERR_SIZE, "0-sized canvas (a browser draws nothing; the detector then throws)");
  if ((reinterpret_cast<uintptr_t>(src_rgba) & 3u) || (reinterpret_cast<uintptr_t>(dst_rgba) & 3u)) return ctx->fail(HT_ERR_ARG, "frames must be 4-byte aligned");
  if (sw > 16384 || sh > 16384 || dw > 16384 || dh > 16384) return ctx->fail(HT_ERR_SIZE, "frame too large");
  IngestGeom g{sw, sh, dw, dh, 0, 0, 0};
  if (!bilinear_division_constants(4ull * dw * dh, g.magic, g.shift)) return ctx->fail(HT_ERR_SIZE, "canvas too large for 32-bit bilinear numerators");
  g.half = (uint32_t)(2ull * dw * dh);
  CK(cudaSetDevice(ctx->cfg.device));
  const size_t sbytes = (size_t)n * sw * sh * 4, dbytes = (size_t)n * dw * dh * 4;
  const uint8_t *d_src = src_rgba;
  if (!is_device_ptr(src_rgba)) {
    CK(ctx->d_frames.reserve(sbytes));
    CK(cudaMemcpyAsync(ctx->d_frames.p, src_rgba, sbytes, cudaMemcpyHostToDevice, ctx->stream));
    d_src = ctx->d_frames.as<uint8_t>();
  }
  const bool out_dev = is_device_ptr(dst_rgba);
  uint8_t *d_dst = dst_rgba;
  if (!out_dev) { CK(ctx->d_scratch.reserve(dbytes)); d_dst = ctx->d_scratch.as<uint8_t>(); }
  if (sw == dw && sh == dh) {   // a 1:1 draw is a copy (oracle/ht_oracle.h)
    CK(cudaMemcpyAsync(d_dst, d_src, dbytes, cudaMemcpyDeviceToDevice, ctx->stream));
  } else {
    k_ingest<<<dim3((unsigned)(dw + 63) / 64, (unsigned)(dh + 3) / 4, (unsigned)n), 256, 0, ctx->stream>>>(d_src, d_dst, g);
    ++ctx->launches;
    CK(cudaGetLastError());
  }
  if (!out_dev) {
    CK(cudaMemcpyAsync(dst_rgba, d_dst, dbytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return HT_OK;
}

int ht_backprojection(ht_ctx *ctx, int slot, const uint8_t *rgba, int w, int h, uint8_t *out_rgba) {
  if (!ctx) return HT_ERR_ARG;
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  if (!out_rgba || slot < 0 || slot >= ctx->cfg.max_frames || w <= 0 || h <= 0) return ctx->fail(HT_ERR_ARG, "bad argument");
  CK(cudaSetDevice(ctx->cfg.device));
  int rc = ensure_tracker_buffers(ctx);
  if (rc != HT_OK) return rc;
  const uint8_t *d_rgba = nullptr;
  rc = device_frames(ctx, rgba, 1, w, h, &d_rgba);
  if (rc != HT_OK) return rc;
  const size_t bytes = (size_t)w * h * 4;
  CK(ctx->d_scratch.reserve(bytes + 4096 * sizeof(uint32_t)));
  uint32_t *hist = reinterpret_cast<uint32_t *>(ctx->d_scratch.as<uint8_t>() + bytes);
  rc = launch_hist(ctx, d_rgba, 1, w, h, hist, nullptr);
  if (rc != HT_OK) return rc;
  const bool out_dev = is_device_ptr(out_rgba);
  uint8_t *d_out = out_dev ? out_rgba : ctx->d_scratch.as<uint8_t>();
  k_backproj<<<(w * h + 255) / 256, 256, 0, ctx->stream>>>(d_rgba, w * h, ctx->model_hist.as<uint32_t>() + (size_t)slot * 4096,
                                                          hist, d_out);
  ++ctx->launches;
  CK(cudaGetLastError());
  if (!out_dev) {
    CK(cudaMemcpyAsync(out_rgba, d_out, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return HT_OK;
}

int ht_whitebalance(ht_ctx *ctx, const uint8_t *rgba, int n, int w, int h, double *out) {
  if (!ctx) return HT_ERR_ARG;
  if (!out || w <= 0 || h <= 0) return ctx->fail(HT_ERR_ARG, "bad argument");
  int rc = check_batch(ctx, n);
  if (rc != HT_OK) return rc;
  CK(cudaSetDevice(ctx->cfg.device));
  const uint8_t *d_rgba = nullptr;
  rc = device_frames(ctx, rgba, n, w, h, &d_rgba);
  if (rc != HT_OK) return rc;
  const size_t mf = (size_t)ctx->cfg.max_frames;
  CK(ctx->d_wb_sums.reserve(mf * 3 * sizeof(unsigned long long)));
  CK(ctx->d_wb_out.reserve(mf * sizeof(double)));
  CK(cudaMemsetAsync(ctx->d_wb_sums.p, 0, (size_t)n * 3 * sizeof(unsigned long long), ctx->stream));
  const int chunks = std::min(64, std::max(1, 1184 / n));
  k_wb_sums<<<dim3(chunks, n), 256, 0, ctx->stream>>>(d_rgba, (size_t)w * h * 4, w * h, ctx->d_wb_sums.as<unsigned long long>(), chunks);
  const bool out_dev = is_device_ptr(out);
  double *d_out = out_dev ? out : ctx->d_wb_out.as<double>();
  k_wb_final<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->d_wb_sums.as<unsigned long long>(), n, w * h, d_out);
  ctx->launches += 2;
  CK(cudaGetLastError());
  if (!out_dev) {
    CK(cudaMemcpyAsync(out, d_out, sizeof(double) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
  }
  return HT_OK;
}

int ht_profile(ht_ctx *ctx, int enable) {
  if (!ctx) return HT_ERR_ARG;
  ctx->prof_on = enable != 0;
  return HT_OK;
}

int ht_profile_read(ht_ctx *ctx, double *ms, uint64_t *launches, int reset) {
  if (!ctx) return HT_ERR_ARG;
  CK(cudaSetDevice(ctx->cfg.device));
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  CK(cudaStreamSynchronize(ctx->stream));
  for (auto &sp : ctx->prof_spans) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, sp.a, sp.b) == cudaSuccess) {
      ctx->prof_ms[sp.cls] += t;
      ctx->prof_launches[sp.cls] += 1;
    } else cudaGetLastError();
    ctx->prof_free.push_back(sp.a);
    ctx->prof_free.push_back(sp.b);
  }
  ctx->prof_spans.clear();
  for (int i = 0; i < HT_PROF_N; ++i) {
    if (ms) ms[i] = ctx->prof_ms[i];
    if (launches) launches[i] = ctx->prof_launches[i];
    if (reset) { ctx->prof_ms[i] = 0; ctx->prof_launches[i] = 0; }
  }
  return HT_OK;
}

// ---- introspection for the parity tests ----

int ht_plan_info(ht_ctx *ctx, int w, int h, int interval, int32_t *n_slots, int32_t *scale_upto, int32_t *slot_w,
                 int32_t *slot_h, int cap) {
  if (!ctx) return HT_ERR_ARG;
  CK(cudaSetDevice(ctx->cfg.device));
  Plan *P = nullptr;
  int rc = get_plan(ctx, w, h, interval, &P);
  if (rc != HT_OK) return rc;
  if (n_slots) *n_slots = P->n_slots;
  if (scale_upto) *scale_upto = P->scale_upto;
  for (int i = 0; i < P->n_slots && i < cap; ++i) {
    if (slot_w) slot_w[i] = P->slot_w[i];
    if (slot_h) slot_h[i] = P->slot_h[i];
  }
  return HT_OK;
}

int ht_debug_plane(ht_ctx *ctx, int frame, int slot, int q, uint8_t *out, int cap_bytes, int32_t *w, int32_t *h) {
  if (!ctx) return HT_ERR_ARG;
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  Plan *P = ctx->last_plan;
  if (!P) return ctx->fail(HT_ERR_STATE, "no ht_detect call yet");
  if (frame < 0 || frame >= ctx->last_n || slot < 0 || slot >= P->n_slots || q < 0 || q > 3) return ctx->fail(HT_ERR_ARG, "bad frame/slot/q");
  const int id = P->plane_id[(size_t)slot * 4 + q];
  if (id < 0) return ctx->fail(HT_ERR_ARG, "plane (%d,%d) does not exist", slot, q);
  const DevPlane &pl = P->planes[id];
  if (w) *w = pl.w;
  if (h) *h = pl.h;
  if (!out || cap_bytes < pl.w * pl.h) return ctx->fail(HT_ERR_ARG, "output too small");
  if (frame < ctx->last_wave_f0 || frame >= ctx->last_wave_f0 + ctx->last_wave_n || !ctx->last_wave_arena)
    return ctx->fail(HT_ERR_STATE, "the pyramid of frame %d is no longer resident (only the last wave of %d frames is; see HT_WAVE)",
                     frame, ctx->last_wave_n);
  CK(cudaSetDevice(ctx->cfg.device));
  CK(cudaStreamSynchronize(ctx->stream));
  // the arena is frame-quad-interleaved: one word per pixel, byte f = frame within its quad
  const int rel = frame - ctx->last_wave_f0;
  std::vector<uint32_t> words((size_t)pl.pitch * pl.h);
  CK(cudaMemcpy(words.data(), ctx->last_wave_arena + (size_t)(rel / 4) * P->arena_stride + pl.off, words.size() * 4,
                cudaMemcpyDeviceToHost));
  for (int y = 0; y < pl.h; ++y)
    for (int x = 0; x < pl.w; ++x) out[(size_t)y * pl.w + x] = (uint8_t)(words[(size_t)y * pl.pitch + x] >> (8 * (rel & 3)));
  return HT_OK;
}

int ht_debug_raw(ht_ctx *ctx, int frame, ht_rect *out, int cap, int32_t *count) {
  if (!ctx) return HT_ERR_ARG;
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  if (!ctx->last_plan || frame < 0 || frame >= ctx->last_n || !count) return ctx->fail(HT_ERR_ARG, "bad frame");
  CK(cudaSetDevice(ctx->cfg.device));
  CK(cudaStreamSynchronize(ctx->stream));
  uint32_t c = 0;
  CK(cudaMemcpy(&c, ctx->raw_count.as<uint32_t>() + frame, sizeof(c), cudaMemcpyDeviceToHost));
  *count = (int32_t)c;
  const int ncopy = std::min<int>(std::min<uint32_t>(c, (uint32_t)ctx->raw_cap), cap);
  if (out && ncopy > 0)
    CK(cudaMemcpy(out, ctx->sorted.as<Rect>() + (size_t)frame * ctx->raw_cap, sizeof(Rect) * ncopy, cudaMemcpyDeviceToHost));
  return HT_OK;
}

int ht_debug_set_exactness(ht_ctx *ctx, int flags) {
  if (!ctx) return HT_ERR_ARG;
  ctx->force_ties = flags;
  return HT_OK;
}

int ht_set_track_memo(ht_ctx *ctx, int enable) {
  if (!ctx) return HT_ERR_ARG;
  ctx->track_memo = enable != 0;
  return HT_OK;
}

int ht_set_pipeline(ht_ctx *ctx, int enable) {
  if (!ctx) return HT_ERR_ARG;
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  ctx->pipeline = enable ? 1 : 0;
  return HT_OK;
}

int ht_join(ht_ctx *ctx) {
  if (!ctx) return HT_ERR_ARG;
  return join_aux(ctx);
}

int ht_debug_track_stats(ht_ctx *ctx, uint64_t *out5, int reset) {
  if (!ctx || !out5) return HT_ERR_ARG;
  CK(cudaSetDevice(ctx->cfg.device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(out5, ctx->d_flags.as<unsigned long long>() + 8, 5 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  if (reset) CK(cudaMemset(ctx->d_flags.as<unsigned long long>() + 8, 0, 5 * sizeof(uint64_t)));
  return HT_OK;
}

int ht_debug_track_trace(ht_ctx *ctx, uint64_t *out, int n) {
  if (!ctx || !out) return HT_ERR_ARG;
  if (!ctx->track_trace || !ctx->d_trace.p || n < 0 || n > ctx->cfg.max_frames)
    return ctx->fail(HT_ERR_ARG, "track timeline is not enabled (HT_TRACK_TRACE=1 at ht_create) or n is out of range");
  CK(cudaSetDevice(ctx->cfg.device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(out, ctx->d_trace.p, 4 * sizeof(uint64_t) * (size_t)n, cudaMemcpyDeviceToHost));
  return HT_OK;
}

int ht_debug_track_phases(ht_ctx *ctx, uint64_t *out, int n) {
  if (!ctx) return HT_ERR_ARG;
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  if (!ctx->track_trace || !ctx->d_trace.p || n < 0 || n > ctx->cfg.max_frames)
    return ctx->fail(HT_ERR_ARG, "no track trace (create the context with HT_TRACK_TRACE=1)");
  CK(cudaSetDevice(ctx->cfg.device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(out, ctx->d_trace.as<unsigned long long>() + 4 * (size_t)ctx->cfg.max_frames, 8 * sizeof(uint64_t) * (size_t)n, cudaMemcpyDeviceToHost));
  return HT_OK;
}

int ht_debug_model_hist(ht_ctx *ctx, int slot, uint32_t *out4096) {
  if (!ctx) return HT_ERR_ARG;
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  { const int jr = join_aux(ctx); if (jr != HT_OK) return jr; }
  if (!out4096 || slot < 0 || slot >= ctx->cfg.max_frames || !ctx->model_hist.p) return ctx->fail(HT_ERR_ARG, "bad slot");
  CK(cudaSetDevice(ctx->cfg.device));
  CK(cudaStreamSynchronize(ctx->stream));
  CK(cudaMemcpy(out4096, ctx->model_hist.as<uint32_t>() + (size_t)slot * 4096, 4096 * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  return HT_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// Host-only self-test of the cascade parser and the late-stage schedule (no device needed):
//   nvcc -DHT_HOST_SELFTEST -o ht_selftest ht_api.cu && ./ht_selftest ../data/cascade_face.bin
// Prints one JSON line; tests/test_late_schedule.py checks it.
#ifdef HT_HOST_SELFTEST
// ---- CPU emulation of k_cascade's tile evaluation (tests/test_cascade_host.py) ----
// Same generated stage code (cascade_face_gen.inc, compiled for the host), same tile layout (point_word), same
// staging index arithmetic, same bank-class bookkeeping, same late-stage schedule and integer thresholds as the
// kernel; only the parallel execution is replaced by loops.  The arena is one frame quad in the device layout.
extern "C" int ht_selftest_planes(int w, int h, int interval, int32_t *out, int cap) {
  Plan P;
  std::string err;
  if (build_plan(P, w, h, interval, 24, 24, err, false) != HT_OK) return -1;
  if ((int)P.planes.size() * 6 + 2 > cap) return -2;
  out[0] = (int32_t)P.planes.size();
  out[1] = (int32_t)P.arena_stride;
  for (size_t i = 0; i < P.planes.size(); ++i) {
    int slot = -1, q = -1;
    for (size_t k = 0; k < P.plane_id.size(); ++k) if (P.plane_id[k] == (int)i) { slot = (int)(k / 4); q = (int)(k % 4); }
    int32_t *o = out + 2 + 6 * i;
    o[0] = (int32_t)P.planes[i].off; o[1] = P.planes[i].pitch; o[2] = P.planes[i].w; o[3] = P.planes[i].h; o[4] = slot; o[5] = q;
  }
  return 0;
}

// the head-position epilogue of k_stream_update (head_step) over a sequence of CS results of one stream
extern "C" int ht_selftest_head(const ht_head_params *params, int n, const double *cs /* [n][5]: is_cs, x, y, w, h */, int camw,
                                int camh, ht_head_event *out) {
  const HeadParams hp = make_head_params(params);
  HeadState s;
  head_new_state(s);
  for (int i = 0; i < n; ++i) {
    const double *c = cs + 5 * i;
    HeadEvent he;
    head_step(s, hp, c[0] != 0.0, c[1], c[2], c[3], c[4], c[0] != 0.0 && (c[3] == 0.0 || c[4] == 0.0), (double)camw, (double)camh, he);
    memcpy(out + i, &he, sizeof(he));
  }
  return 0;
}

// k_ingest's per-pixel code over a whole frame batch
extern "C" int ht_selftest_ingest(const uint8_t *src, int n, int sw, int sh, uint8_t *dst, int dw, int dh) {
  IngestGeom g{sw, sh, dw, dh, 0, 0, 0};
  if (!bilinear_division_constants(4ull * dw * dh, g.magic, g.shift)) return -1;
  g.half = (uint32_t)(2ull * dw * dh);
  for (int f = 0; f < n; ++f)
    for (int Y = 0; Y < dh; ++Y)
      for (int X = 0; X < dw; ++X) ingest_pixel(src, dst, g, X, Y, f);
  return 0;
}

// gray + pyramid of one frame quad with the kernels' own per-thread code (gray_item, resample_thread), thread by thread
extern "C" int ht_selftest_pyramid(int w, int h, int interval, const uint8_t *rgba, int n_frames, uint32_t *arena, size_t arena_words) {
  Plan P;
  std::string err;
  if (build_plan(P, w, h, interval, 24, 24, err, false) != HT_OK) return -1;
  if (arena_words < P.arena_stride || n_frames < 1 || n_frames > 4) return -2;
  DevPlan dp{};
  dp.planes = P.planes.data(); dp.jobs = P.jobs.data(); dp.taps = P.taps.data(); dp.pyr_tiles = P.pyr_tiles.data();
  dp.scales = P.scales.data(); dp.casc_tiles = P.casc_tiles.data();
  dp.n_planes = (int)P.planes.size(); dp.n_jobs = (int)P.jobs.size();
  dp.n_scales = (int)P.scales.size(); dp.n_casc_tiles = (int)P.casc_tiles.size();
  const unsigned fmask = (1u << n_frames) - 1u;
  const int pitch0 = P.planes[0].pitch, gpr = pitch0 >> 2;
  const bool vec = (w % 4 == 0) && ((reinterpret_cast<uintptr_t>(rgba) & 15u) == 0);
  for (int it = 0; it < gpr * h; ++it) {
    if (vec) gray_item<true, false>(rgba, (size_t)w * h * 4, 0, fmask, arena, w, pitch0, gpr, it, nullptr, nullptr, w * h);
    else gray_item<false, false>(rgba, (size_t)w * h * 4, 0, fmask, arena, w, pitch0, gpr, it, nullptr, nullptr, w * h);
  }
  for (size_t g = 1; g + 1 < P.gen_tile_begin.size(); ++g)
    for (int t = P.gen_tile_begin[g]; t < P.gen_tile_begin[g + 1]; ++t)
      for (int tid = 0; tid < 256; ++tid) resample_thread(dp, P.gen_tile_begin[g], arena, P.arena_stride, t - P.gen_tile_begin[g], 0, tid);
  return 0;
}

extern "C" int ht_selftest_cascade(const void *blob, size_t blob_len, int w, int h, int interval, const uint32_t *arena,
                                   int n_frames, int force_ties, int quad_stages, double *out /* [4][cap][4] x,y,width,conf */,
                                   int32_t *counts, int cap) {
  if (quad_stages != HT_GEN_QUAD_STAGES) return -4;   // the dense group evaluates stages {0,1} in quad form, as k_cascade
  static HostCascade hc;   // (ConstCascade is 63 KB: keep it off the stack)
  std::string err;
  if (parse_cascade(blob, blob_len, hc, err) != HT_OK) { fprintf(stderr, "%s\n", err.c_str()); return -1; }
  if (!hc.fast) return -3;
  Plan P;
  if (build_plan(P, w, h, interval, hc.width, hc.height, err, false) != HT_OK) { fprintf(stderr, "%s\n", err.c_str()); return -2; }
  g_host_casc = &hc.cc;
  const ConstCascade &cc = hc.cc;
  const int late_first = cc.group_first[cc.n_groups];
  struct Hit { uint32_t key; double x, y, width, conf; };
  std::vector<Hit> hits[4];
  std::vector<uint32_t> tile((size_t)TILE_WORDS);
  const unsigned fmask = n_frames >= 4 ? 15u : (1u << n_frames) - 1u;
  for (const DevCascTile &tl : P.casc_tiles) {
    const DevScale &sc = P.scales[tl.scale];
    const int x0 = tl.tx * TW, y0 = tl.ty * TH;
    // staging: what the kernel's loops write, through the same layout functions (tile_l0 / tile_l1 / tile_l2)
    std::fill(tile.begin(), tile.end(), 0u);
    {
      const DevPlane pl = P.planes[sc.p0];
      const uint32_t *src = arena + pl.off;
      const int X0 = 4 * x0, Y0 = 4 * y0;
      for (int r = 0; r < L0_ROWS; ++r)
        for (int X = 0; X < L0_COLS; ++X) {
          const bool ok = (Y0 + r < pl.h) && (X0 + X < pl.pitch);
          tile[(size_t)tile_l0(r, X)] = ok ? src[(size_t)(Y0 + r) * pl.pitch + X0 + X] : 0u;
        }
    }
    {
      const DevPlane pl = P.planes[sc.p1];
      const uint32_t *src = arena + pl.off;
      const int X0 = 2 * x0, Y0 = 2 * y0;
      for (int r = 0; r < L1_ROWS; ++r)
        for (int c = 0; c < P1; ++c) {
          const bool ok = (Y0 + r < pl.h) && (X0 + c < pl.pitch);
          tile[(size_t)tile_l1(r, c)] = ok ? src[(size_t)(Y0 + r) * pl.pitch + X0 + c] : 0u;
        }
    }
    for (int rr = 0; rr < 2 * L2_ROWS; ++rr)
      for (int c2 = 0; c2 < P2; ++c2) {
        const int q = (c2 & 1) | ((rr & 1) << 1), r = rr >> 1, c = c2 >> 1;
        const DevPlane pl = P.planes[sc.p2[q]];
        const uint32_t *src = arena + pl.off;
        const bool ok = (y0 + r < pl.h) && (x0 + c < pl.pitch);
        tile[(size_t)tile_l2(rr, c2)] = ok ? src[(size_t)(y0 + r) * pl.pitch + x0 + c] : 0u;
      }
    const uint8_t *tile_b = reinterpret_cast<const uint8_t *>(tile.data());
    auto bases = [&](int e, const uint8_t *&tA, const uint8_t *&tB) {
      const int u = e & 63, v = (e >> 6) & 31, f = e >> 11;
      tA = tile_b + 4 * (v * VA + u) + f;
      tB = tile_b + 4 * (v * VB + u) + f;
    };
    // dense group (quad form)
    std::vector<int> list[32];
    for (int v = 0; v < 2 * TH; ++v)
      for (int u = 0; u < 2 * TW; ++u) {
        const int lx = u >> 1, ly = v >> 1;
        const uint32_t *tA = tile.data() + v * VA + u, *tB = tile.data() + v * VB + u;
        uint32_t a_lo = 0, a_hi = 0;
        if (x0 + lx < sc.qw && y0 + ly < sc.qh) {
          a_lo = ((fmask & 1u) ? 0x8000u : 0u) | ((fmask & 4u) ? 0x80000000u : 0u);
          a_hi = ((fmask & 2u) ? 0x8000u : 0u) | ((fmask & 8u) ? 0x80000000u : 0u);
        }
        for (int J = 0; J < HT_GEN_QUAD_STAGES; ++J) {
          uint32_t p_lo = 0, p_hi = 0, t_lo = 0, t_hi = 0;
          if (J == 0) gen_q_stage0(tA, tB, p_lo, p_hi, t_lo, t_hi);
          else gen_q_stage1(tA, tB, p_lo, p_hi, t_lo, t_hi);
          t_lo &= a_lo; t_hi &= a_hi;
          for (int f = 0; f < 4; ++f) {
            const uint32_t bit = (f & 2) ? 0x80000000u : 0x8000u;
            uint32_t &tt = (f & 1) ? t_hi : t_lo, &pp = (f & 1) ? p_hi : p_lo;
            if (tt & bit) {
              const uint8_t *bA = reinterpret_cast<const uint8_t *>(tA) + f, *bB = reinterpret_cast<const uint8_t *>(tB) + f;
              if (!stage_pass_ordered(bA, bB, J)) pp &= ~bit;
            }
          }
          a_lo &= p_lo; a_hi &= p_hi;
        }
        const uint32_t m = ((a_lo >> 15) & 1u) | ((a_hi >> 14) & 2u) | ((a_lo >> 29) & 4u) | ((a_hi >> 28) & 8u);
        for (int f = 0; f < 4; ++f)
          if (m & (1u << f)) list[bank_class(u, v)].push_back((v << 6) | u | (f << 11));
      }
    // survivor lists, then late stages
    for (int c = 0; c < 32; ++c)
      for (int e : list[c]) {
        const uint8_t *tA, *tB;
        bases(e, tA, tB);
        bool alive = true;
        for (int j = HT_GEN_QUAD_STAGES; j < late_first && alive; ++j) {
          int r = gen_stage(j, tA, tB);
          if (force_ties & 1) r = -1;
          if (r < 0) r = stage_pass_ordered(tA, tB, j) ? 1 : 0;
          alive = r != 0;
        }
        for (int j = late_first; j < cc.n_stages && alive; ++j) {
          long long acc = 0;
          for (int ch = hc.late_chunk0[j]; ch < hc.late_chunk0[j + 1]; ++ch)
            for (int lane = 0; lane < 32; ++lane) {
              const LateFeat &lf = hc.late[(size_t)ch * 32 + lane];
              unsigned pm = 255u, nm = 0u;
              for (int s = 0; s < 10; ++s) {
                if (lf.off[s] == LATE_UNUSED) continue;
                const unsigned v8 = px_at(tA, tB, late_decode(lf.off[s]));
                if (s < 5) pm = std::min(pm, v8); else nm = std::max(nm, v8);
              }
              acc += (pm > nm) ? (long long)lf.a_int : -(long long)lf.a_int;
            }
          if (acc == cc.thr_int[j] || (force_ties & 2)) alive = stage_pass_ordered(tA, tB, j);
          else alive = acc > cc.thr_int[j];
        }
        if (!alive) continue;
        const int u = e & 63, v = (e >> 6) & 31, f = e >> 11;
        const int lx = u >> 1, ly = v >> 1, q = (u & 1) | ((v & 1) << 1);
        Hit hit;
        hit.key = sc.win_base + (uint32_t)((q * sc.qh + (y0 + ly)) * sc.qw + (x0 + lx));
        hit.x = (double)((x0 + lx) * 4 + (q & 1) * 2) * sc.scale_x;          // k_group's decoding, src/ccv.js:228-233
        hit.y = (double)((y0 + ly) * 4 + (q >> 1) * 2) * sc.scale_x;
        hit.width = 24.0 * sc.scale_x;
        hit.conf = stage_sum_ordered(tA, tB, cc.n_stages - 1);
        hits[f].push_back(hit);
      }
  }
  for (int f = 0; f < 4; ++f) {
    std::sort(hits[f].begin(), hits[f].end(), [](const Hit &a, const Hit &b) { return a.key < b.key; });
    counts[f] = (int32_t)hits[f].size();
    for (size_t i = 0; i < hits[f].size() && (int)i < cap; ++i) {
      double *o = out + ((size_t)f * cap + i) * 4;
      o[0] = hits[f][i].x; o[1] = hits[f][i].y; o[2] = hits[f][i].width; o[3] = hits[f][i].conf;
    }
  }
  return 0;
}

int main(int argc, char **argv) {
  if (argc < 2) { fprintf(stderr, "usage: %s cascade.bin\n", argv[0]); return 2; }
  FILE *f = fopen(argv[1], "rb");
  if (!f) { perror("open"); return 2; }
  std::vector<uint8_t> blob;
  uint8_t buf[4096];
  size_t got;
  while ((got = fread(buf, 1, sizeof(buf), f)) > 0) blob.insert(blob.end(), buf, buf + got);
  fclose(f);
  HostCascade hc;
  std::string err;
  const int rc = parse_cascade(blob.data(), blob.size(), hc, err);
  if (rc != HT_OK) { fprintf(stderr, "parse_cascade: %s\n", err.c_str()); return 1; }
  const ConstCascade &cc = hc.cc;
  const int late_first = cc.group_first[cc.n_groups];
  // every feature of a late stage appears exactly once, with its points and its alpha
  long long bad = 0, used_slots = 0, used_instr = 0, conflicts = 0;
  for (int j = late_first; j < hc.n_stages; ++j) {
    std::vector<int> seen((size_t)cc.stage[j].count, 0);
    for (int ch = hc.late_chunk0[j]; ch < hc.late_chunk0[j + 1]; ++ch) {
      for (int s = 0; s < 10; ++s) {
        int bank_word[32];
        for (int &v : bank_word) v = -1;
        bool any = false;
        for (int lane = 0; lane < 32; ++lane) {
          const uint16_t o = late_decode(hc.late[(size_t)ch * 32 + lane].off[s]);
          if (o == 0xFFFF) continue;
          any = true; ++used_slots;
          const int word = o & 0x7fff;
          if (bank_word[word & 31] >= 0 && bank_word[word & 31] != word) ++conflicts;
          bank_word[word & 31] = word;
        }
        used_instr += any ? 1 : 0;
      }
      for (int lane = 0; lane < 32; ++lane) {
        const LateFeat &lf = hc.late[(size_t)ch * 32 + lane];
        std::vector<uint16_t> p, n;
        for (int s = 0; s < 5; ++s) if (lf.off[s] != LATE_UNUSED) p.push_back(late_decode(lf.off[s]));
        for (int s = 5; s < 10; ++s) if (lf.off[s] != LATE_UNUSED) n.push_back(late_decode(lf.off[s]));
        if (p.empty() && n.empty()) { if (lf.a_int != 0) ++bad; continue; }
        std::sort(p.begin(), p.end()); std::sort(n.begin(), n.end());
        int match = -1;
        for (int k = cc.stage[j].first; k < cc.stage[j].first + cc.stage[j].count && match < 0; ++k) {
          if (seen[(size_t)(k - cc.stage[j].first)]) continue;
          std::vector<uint16_t> kp(cc.off[k], cc.off[k] + (cc.np_nn[k] & 15)), kn(cc.off[k] + 5, cc.off[k] + 5 + (cc.np_nn[k] >> 4));
          std::sort(kp.begin(), kp.end()); std::sort(kn.begin(), kn.end());
          if (kp == p && kn == n && llround(cc.alpha[k] * 1e8) == lf.a_int) match = k;
        }
        if (match < 0) ++bad; else seen[(size_t)(match - cc.stage[j].first)] = 1;
      }
    }
    for (int v : seen) if (!v) ++bad;
  }
  printf("{\"n_stages\": %d, \"n_features\": %d, \"fast\": %d, \"n_groups\": %d, \"late_first\": %d, \"chunks\": %d, "
         "\"bad\": %lld, \"point_loads\": %lld, \"load_instr_with_traffic\": %lld, \"bank_conflicts\": %lld, \"late_conflicts\": %d}\n",
         hc.n_stages, hc.n_features, hc.fast ? 1 : 0, cc.n_groups, late_first, hc.late_chunk0[hc.n_stages], bad, used_slots,
         used_instr, conflicts, hc.late_conflicts);
  return bad ? 1 : 0;
}
#endif
