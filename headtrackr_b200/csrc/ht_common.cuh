// ht_common.cuh — structures shared by the host planner and the sm_100a kernels.
//
// Data layout in HBM (see DESIGN.md §3):
//   frames   : caller-owned RGBA8, n contiguous frames of w*h*4 bytes (the "canvas" of the reference).
//   arena    : per frame, every pyramid plane of src/ccv.js:113-147 as a single-channel u8 plane
//              (the reference only ever reads channel 0 of its gray canvases, src/ccv.js:171).
//              Plane pitch is the width rounded up to 16 B so tile staging can use 16 B vector loads;
//              plane offsets are 256 B aligned.  Planes are indexed densely; plane 0 is the gray image.
//   plan     : immutable per (w,h,interval): plane table, resample jobs + their column/row tap tables,
//              per-scale window geometry, tile lists.  Built once on the host (ht_plan.cuh).
//   cascade  : immutable device copy of the BBF cascade (features as shared-memory byte offsets).
#pragma once
#include <cstddef>
#include <cstdint>

namespace ht {

// ------------------------------------------------------------------------------------------------
// Frame quads.  The pyramid arena is stored FRAME-QUAD-INTERLEAVED: one 32-bit word per pixel holds the gray
// value of that pixel in four consecutive frames of the batch (byte f = frame & 3).  One LDS.32 / LDG.32 therefore
// serves the same window of four frames, the resampler's tap arithmetic is shared by four frames, and a window's
// base address never splits a bank word (round 1 lost 23 % of its shared-memory wavefronts to that).
// Arena of quad g starts at g * quad_stride words; plane offsets and pitches are in WORDS (pitch % 4 == 0).
//
// Cascade-tile geometry (k_cascade).  A tile is TW x TH quarter-resolution window positions x 4 phases x 4 frames.
// With u = 2*lx + dx in [0, 2*TW) and v = 2*ly + dy in [0, 2*TH) the three pyramid levels a window reads are staged
// in shared memory so that EVERY feature point is  base + constant  with two per-window bases
//     baseA = v * (2*P0) + u          (level 0)            baseB = v * P1 + u      (levels 1 and 2)
//   level 0 (full res), pixel (X,Y)      : word  Y*P0 + (X&1)*H0 + (X>>1)            (columns split by parity, so that
//                                           the 32 windows u..u+31 of a warp read 32 consecutive words)
//   level 1 (half res), pixel (X,Y)      : word  W1 + Y*P1 + X
//   level 2 (quarter res), phase copy q  : word  W2 + (2*Y + dy)*P2 + 2*X + dx       (the four copies interleaved)
// A window's level-0 origin is (2u, 2v), its level-1 origin (u, v), its level-2 origin (lx, ly) in copy q
// (src/ccv.js:179-180,235-241).  2*P0 == P1 == P2 (mod 32), so bank(baseA) == bank(baseB) == (u + 12 v) & 31: the
// "bank class" of the window.  Lane L only ever evaluates class-L windows -> conflict-free loads in every stage.
constexpr int TW = 32;
constexpr int TH = 8;                         // quarter-res rows of a tile
constexpr int NV = 2 * TH;                    // v values of a tile
constexpr int L0_COLS = 4 * TW + 22;          // 150 level-0 columns
constexpr int L0_ROWS = 4 * TH + 22;
constexpr int H0 = L0_COLS / 2;               // 75: word offset of the odd-column half of a level-0 row
constexpr int P0 = L0_COLS;                   // 150 words per level-0 row
constexpr int L1_ROWS = 2 * TH + 11;
constexpr int L1_COLS = 2 * TW + 11;          // 75
constexpr int P1 = 76;
constexpr int L2_ROWS = TH + 5;               // per copy
constexpr int L2_COLS = TW + 5;               // 37 per copy
constexpr int P2 = 76;
// The three levels are separate blocks (level 1 a dense box that the TMA engine can write), with two per-window bases.
constexpr int W1 = (L0_ROWS * P0 + 31) / 32 * 32;   // 128-byte aligned: the level-1 box can be written by TMA
constexpr int W2 = W1 + L1_ROWS * P1;
constexpr int TILE_WORDS = W2 + 2 * L2_ROWS * P2;
// word of level-0 pixel (row r, column X), level-1 pixel (r, c), interleaved level-2 entry (row rr = 2Y+dy, column c2 = 2X+dx)
__host__ __device__ constexpr int tile_l0(int r, int X) { return r * P0 + (X & 1) * H0 + (X >> 1); }
__host__ __device__ constexpr int tile_l1(int r, int c) { return W1 + r * P1 + c; }
__host__ __device__ constexpr int tile_l2(int rr, int c2) { return W2 + rr * P2 + c2; }
// words per unit of v of the two window bases: baseA = v * VA + u (level 0), baseB = v * VB + u (levels 1, 2)
constexpr int VA = 2 * P0;
constexpr int VB = P1;
static_assert((VA - VB) % 32 == 0 && P1 == P2, "bank classes of the two bases must coincide");
static_assert(2 * L2_COLS <= P2 && L1_COLS <= P1, "tile pitches");
constexpr int BANK_K = VA % 32;               // bank(baseA) = bank(baseB) = (u + BANK_K * v) & 31
static_assert(VB % 32 == BANK_K, "bank_class");
constexpr int NWIN = TW * TH * 4 * 4;         // windows per tile (4 phases x 4 frames)
// Survivors are kept as BIT MASKS per bank class: class c owns, for every v, the two windows u = ((c - BANK_K v) & 31)
// + 32 uh, each in 4 frames -> bit 8 v + 4 uh + f of the class's mask (NV / 4 words).  masks[word][class].
constexpr int MASK_WORDS = NV / 4;
static_assert(NV % 4 == 0, "TH must be even");
constexpr int CASCADE_THREADS = 256;
constexpr int CASCADE_WARPS = CASCADE_THREADS / 32;
constexpr int CASCADE_MIN_BLOCKS = 4;         // resident k_cascade CTAs per SM the register allocation aims at
// shared-memory WORD offset of point (z, x, y) of the 24x24 window relative to baseA (z == 0) or baseB (z > 0)
__host__ __device__ constexpr int point_word(int z, int x, int y) {
  return z == 0 ? tile_l0(y, x) : z == 1 ? tile_l1(y, x) : tile_l2(2 * y, 2 * x);
}
__host__ __device__ constexpr int bank_class(int u, int v) { return (u + BANK_K * v) & 31; }
// the window of class c at (v, uh)
__host__ __device__ constexpr int class_u(int c, int v, int uh) { return ((c - BANK_K * v) & 31) + 32 * uh; }

// survivor groups of the generated cascade after the dense group {0,1}: {2} {3} {4,5} {6,7}.  A split costs a CTA barrier
// and repacks the survivors (tools/early_exit_model.py: 9 live lanes per warp iteration in stage 5 and 6 in stage 7).
constexpr int MAX_STAGES = 64;
constexpr int MAX_GROUPS = 16;

struct DevPlane {
  uint32_t off;   // WORD offset inside the per-quad arena (one word = the pixel in 4 frames)
  int32_t pitch;  // words per row (multiple of 4 -> rows are 16 B aligned)
  int32_t w, h;
};

// one canvas-shim drawImage(src, sx,sy,sw,sh, 0,0,dw,dh) producing plane `dst` (oracle/ht_oracle.h)
struct alignas(16) DevJob {   // 64 B, read by k_resample as four 16 B vectors (field order matters)
  uint32_t src_off, dst_off;  // plane byte offsets inside the per-frame arena
  int32_t src_pitch, dst_pitch;
  int32_t dst_h;
  int32_t dw, dh;             // painted destination size; the rest of the plane is 0
  uint32_t col_off;           // first entry of the column tap table (even)
  uint32_t row_off;           // first entry of the row tap table
  uint32_t magic, shift;      // floor(n / (4 dw dh)) == (uint64(n) * magic) >> shift   for n <= 255.5 * 4 dw dh
  uint32_t half;              // 2 dw dh (round half up)
  int32_t src, dst;           // plane ids (host bookkeeping)
  uint32_t pad_[2];
};
static_assert(sizeof(DevJob) == 64, "DevJob is four 16-byte loads");

// bilinear taps for one destination column (or row): source indices a,b (already clamped and
// offset by sx/sy) and the numerator f of the fractional weight, 0 <= f < 2*dw (2*dh).
struct alignas(8) TapEnt {
  uint16_t a, b, f, pad_;
};

struct alignas(8) DevPyrTile {  // 32 x 32 pixels of a destination plane
  uint16_t job, tx, ty, pad_;
};

struct DevScale {  // one iteration i of src/ccv.js:154
  int32_t p0, p1, p2[4];  // plane ids: level 0, level 1, four quarter-res phase copies
  int32_t qw, qh;         // src/ccv.js:155-156
  uint32_t win_base;      // index of window (q=0,y=0,x=0) in the reference's (i,q,y,x) visiting order
  int32_t pad_;
  double scale_x;         // src/ccv.js:150,244 (repeated multiplication, computed on the host)
};

struct DevCascTile {
  uint16_t scale, tx, ty, pad_;
};

// The active cascade lives in __constant__ memory (ht_detect.cuh: c_casc): every lane of a warp
// evaluates the same feature at the same time, so all table reads are uniform and go through the
// constant cache / uniform datapath instead of the LSU pipe that the pixel loads saturate.
constexpr int MAX_FEATS = 2112;

struct DevStage {
  int32_t first, count;
  double threshold;
};

struct ConstCascade {
  // shared-memory WORD offsets (point_word) relative to baseA, or to baseB when bit 15 is set; valid p points first
  // (np of them), then repeats of slot 0; same for n.  Layout [feature][p0..p4, n0..n4].
  uint16_t off[MAX_FEATS][10];
  double alpha[MAX_FEATS];     // alpha[2k+1] (pass); alpha[2k] == -alpha[2k+1] is checked on the host
  uint8_t np_nn[MAX_FEATS];    // np | nn << 4   (1..5 each)
  DevStage stage[MAX_STAGES];
  int32_t n_stages;
  int32_t n_groups;                     // lane-per-window stage groups (survivor lists between them)
  int32_t group_first[MAX_GROUPS + 1];  // their stage boundaries; stages >= group_first[n_groups] are "late"
  int32_t late_int;                     // 1: late stages run warp-per-window with exact integer sums
  int64_t thr_int[MAX_STAGES];          // stage thresholds x 1e8 (exact, see LateFeat)
};

// Late stages (few windows, hundreds of features): one WARP per window, one feature per lane.
// Stage sums are accumulated as exact integers: every alpha / threshold of the cascade is a decimal
// literal with <= 8 fractional digits, so alpha * 1e8 is an integer (checked on the host).  The
// fp64 sequential sum of the reference differs from the exact decimal sum by < 1e-11, while two
// distinct decimal sums differ by >= 1e-8: `sum < threshold` (src/ccv.js:222) is therefore decided
// exactly by the integers unless they are EQUAL, in which case the stage is re-evaluated with the
// reference's ordered fp64 adds.  The confidence of a surviving window is always the ordered fp64 sum.
//
// Because an exact integer sum may be taken in any order, the features of a late stage are re-arranged on the
// host (build_late_schedule) into chunks of 32 records - lane L of the warp takes record L of every chunk - such
// that within a chunk the 32 offsets of each load slot fall into different shared-memory banks (all lanes add the
// same per-window base, so conflicts depend only on the offsets).  Unused slots hold 0xFFFF and cost no access.
struct alignas(16) LateFeat {
  // slots 0-4: p points, 5-9: n points.  An entry is the BYTE offset of the point (4 x point_word) with bit 31 set
  // when it is relative to baseB, or 0xFFFFFFFF when the slot is unused: the kernel forms the address with one
  // select and one add, `(int(o) < 0 ? sB - 2^31 : sA) + o` (round 2's first version unpacked 16-bit word offsets:
  // 9 instructions per slot, 25 % of the kernel's instructions).
  uint32_t off[10];
  int32_t a_int;     // alpha[2k+1] * 1e8 (0 for the padding records of a stage's last chunk)
  uint32_t pad_;
};
static_assert(sizeof(LateFeat) == 48, "LateFeat is three 16-byte loads");
constexpr uint32_t LATE_UNUSED = 0xFFFFFFFFu;
// ConstCascade::off encoding (u16: word offset, bit 15 = baseB, 0xFFFF = unused) <-> LateFeat::off encoding
__host__ __device__ constexpr uint32_t late_encode(uint16_t o) {
  return o == 0xFFFF ? LATE_UNUSED : (uint32_t)(o & 0x7fffu) * 4u | ((o & 0x8000u) ? 0x80000000u : 0u);
}
__host__ __device__ constexpr uint16_t late_decode(uint32_t o) {
  return o == LATE_UNUSED ? (uint16_t)0xFFFF : (uint16_t)(((o & 0x7fffffffu) >> 2) | ((o >> 31) ? 0x8000u : 0u));
}
static_assert(sizeof(ConstCascade) <= 65536 - 1024, "cascade must fit the constant bank");

struct DevPlan {  // pointers into one device allocation
  const DevPlane *planes;
  const DevJob *jobs;
  const TapEnt *taps;
  const DevPyrTile *pyr_tiles;
  const DevScale *scales;
  const DevCascTile *casc_tiles;
  int32_t n_planes, n_jobs, n_scales, n_casc_tiles;
};

// result record, identical to ht_rect in include/headtrackr_b200.h
struct Rect {
  double x, y, width, height, confidence;
  int32_t neighbors;
  int32_t pad_;
};

// per-slot camshift.Tracker state (src/camshift.js:153-160)
struct TrackState {
  int32_t sx, sy, sw, sh;  // _searchWindow
  int32_t tx, ty, tw, th;  // _trackObj
  double angle;
  int32_t calc_angles;
  int32_t initialised;
};

}  // namespace ht
