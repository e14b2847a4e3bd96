// Data structures of the scan matcher shared between scan_matcher.cu (single-match path, C ABI)
// and sm_sweep.cu (batched loop-closure sweep).
#pragma once
#include <cstdint>
#include <functional>
#include <utility>
#include <vector>

#include "common.cuh"
#include "sm_math.cuh"

namespace b200 {

constexpr int kMaxTies = 24;          // tie indices returned per pair; more -> host re-runs the pair
constexpr int kSweepThreads = 512;
constexpr int32_t kDevInvalid = -(1 << 30);   // device lookup sentinel: pos + it is always < 0

// CorrelationGrid geometry (M.h:1074-1313, K.h:4572-4965) + smear kernel
struct GridGeom {
  int width = 0, height = 0, stride = 0;
  int roi_x = 0, roi_y = 0, roi_w = 0, roi_h = 0;
  int data_size = 0;
  int ksize = 0;
  bool order_dependent = false;     // kernel has 100s off-centre (SURVEY.md 7, hard part 2)
  double scale = 0.0;
  double off_x = 0.0, off_y = 0.0;  // CoordinateConverter offset of the last raster
  std::vector<uint8_t> kernel;
};

// scratch of the host-side occupancy replay (host_cells)
struct CellScratch {
  std::vector<uint64_t> bits;
  std::vector<uint32_t> touched;
  std::vector<std::pair<int, int>> foot;
};

// One CorrelateScan pass prepared on the host (see build_plan)
struct CorrPlan {
  bool fine = false;
  int nX = 0, nY = 0, nA = 0, n = 0;
  double center[3] = {0, 0, 0}, sp_off[2] = {0, 0}, sp_res[2] = {0, 0}, ang_off = 0, ang_res = 0;
  std::vector<int32_t> offsets;            // nA x n, reference linear offsets (INVALID_SCAN kept)
  std::vector<int32_t> ogx, ogy;           // nA x n, the grid-cell offsets the linear offsets were built from
  std::vector<int32_t> xs, ys;             // grid column / row (ROI included) per x / y index
  std::vector<int32_t> px, py;             // search-space-probability grid cell per x / y index
  std::vector<double> xrel, yrel;          // m_xPoses / m_yPoses
  std::vector<double> newx, newy;          // searchCenter + x / y
  std::vector<double> sqx, sqy;            // Square(x) / Square(y)
  std::vector<double> angle, heading, angpen;   // raw angle, NormalizeAngle(angle), angle penalty
};

int build_plan(const GridGeom & g, int probs_side, const b200sm_params & prm, const b200_scan * q,
               const double center[3], const double sp_off[2], const double sp_res[2], double ang_off,
               double ang_res, bool fine, CorrPlan & pl);

// tail of ComputePositionalCovariance (M.cpp:935-965) from the accumulated sums
inline void finish_positional_cov(double norm, double aXX, double aXY, double aYY, double best,
                                  const double sp_res[2], double ang_res, double cov[9])
{
  if (norm > kTolerance) {
    double vXX = aXX / norm, vXY = aXY / norm, vYY = aYY / norm;
    double vTT = 4 * square(ang_res);
    double minXX = 0.1 * square(sp_res[0]), minYY = 0.1 * square(sp_res[1]);
    vXX = maximum(vXX, minXX);
    vYY = maximum(vYY, minYY);
    double mult = 1.0 / best;
    cov[0] = vXX * mult; cov[1] = vXY * mult; cov[3] = vXY * mult; cov[4] = vYY * mult; cov[8] = vTT;
  }
  if (double_equal(cov[0], 0.0)) cov[0] = kMaxVariance;
  if (double_equal(cov[4], 0.0)) cov[4] = kMaxVariance;
}

// per-pair result of the device reduction
struct PairOut {
  double best;              // best response (before the <= 1 clamp)
  double avg_x, avg_y;      // mean position of the tied poses
  double norm, acc_xx, acc_xy, acc_yy;   // ComputePositionalCovariance accumulators
  int32_t best_sum;         // best integer correlation sum
  int32_t tie_count;
  int32_t ties[kMaxTies];   // flat pose indices (y*nX+x)*nA+a of the first ties, array order
};

// everything the sweep kernels read, by value
struct SweepDev {
  // geometry
  int stride, height, roi_x, roi_y, roi_w, roi_h, data_size, ksize, order_dependent;
  double scale;
  const uint8_t * kern;
  // search space (coarse pass; same for every query)
  int nX, nY, nA, n;
  double norm;                   // n * 100
  int do_penalize;
  double dist_var, min_dist_pen;
  // per query
  const int32_t * offsets;       // [nq][nA][n] device-form lookup
  const int32_t * posidx;        // [nq][nY*nX]
  const double * qgeom;          // [nq][4] viewpoint x,y, grid offset x,y
  const double * center;         // [nq][3]
  const double * xrel, * yrel, * newx, * newy, * sqx, * sqy;   // [nq][nX] / [nq][nY]
  const double * angpen;         // [nq][nA]
  // candidates
  const double * points;         // all candidate scans' unfiltered points, x,y interleaved
  const int32_t * scan_pt_start; // [nscans+1]
  // pairs / items (item = one scan of one pair's chain)
  int npairs, nitems, max_n;
  const int32_t * pair_query;    // [npairs]
  const int32_t * pair_item_start;   // [npairs+1]
  const int32_t * item_pair, * item_scan;   // [nitems]
  int32_t * cells;               // [nitems][max_n]
  int32_t * cell_count;          // [nitems]
  // per-CTA workspaces
  uint8_t * ws_grid; size_t ws_grid_pitch;
  int32_t * ws_sums; size_t ws_sums_pitch;
  double * ws_probs; size_t ws_probs_pitch;   // P probs + 4P covariance terms
  PairOut * out;
};

// Fast sweep path (k_sweep_fast): per-query beam lists in "parity sub-grid" form.
//   The coarse search steps 2 cells in x and y, so one beam only ever reads grid cells of ONE
//   (column parity, row parity) class: the grid is kept in shared memory as one parity sub-grid
//   at a time (4 phases), in which consecutive x-poses are consecutive BYTES -> one 32-bit shared
//   load serves 4 poses.  Beams are grouped by (angle, phase, column alignment m = sub-column & 3);
//   a FAST beam (whole 41x41 window inside the grid) is a 16-bit word offset into the sub-grid.
constexpr int kFastThreads = 1024;
constexpr int kSubPitchW = 76;      // words per sub-grid row: 8 rows x 4 words per warp hit 32 distinct banks
constexpr int kFastRowTiles = 6;    // rows per thread (y_l + 8 r), nY <= 48
constexpr int kFastChunk = 640;     // beams accumulated in 16-bit fields before a flush (640 * 100 < 65536)
struct FastDev {
  int enabled;
  int sub_rows;                  // allocated sub-grid rows (incl. padding rows)
  int xtiles;                    // ceil((nX + 3) / 16)
  const uint16_t * beams;        // FAST descriptors, grouped; per group: plain entries, then multi entries
  const uint16_t * mult;         // multiplicity of every entry (1 for plain entries)
  const int32_t * cls_start;     // [nq][nA][33]: group g = phase * 4 + m -> [2g] plain begin, [2g+1] multi begin, [2g+2] end
  const int32_t * edge;          // EDGE beams in word form, grouped like the FAST lists: sub-row | word << 16 (both signed 16 bit)
  const int32_t * edge_start;    // [nq][nA][17]
  const int32_t * wrap2;         // EDGE beams whose columns leave [0, stride): secondary entries (row parity flipped)
  const int32_t * wrap2_start;   // [nq][nA][4] + 1, per phase
  const int32_t * slow;          // FAR beams (column offsets >= one stride): device-form linear offsets
  const int32_t * slow_start;    // [nq][nA + 1]
};

// Tiled sweep path (k_sweep_tile, sm_tile.cu): the generalisation of the fast path to any search
// dimension / range threshold.  A pair's pose volume is cut into V angle CHUNKS (accumulators of one
// chunk in shared memory) that are spread over the C CTAs of a thread-block cluster; the parity
// sub-grid is cut into row BANDS so that one band + one chunk fit an SM.  The per-(chunk, phase,
// band) beam-descriptor blocks are streamed into shared memory with cp.async.bulk + mbarrier.
constexpr int kTileThreads = 1024;
constexpr int kTileMaxCluster = 8;
struct TileSeq {                 // one descriptor block of a query's schedule (16 bytes)
  int32_t off;                   // byte offset in the descriptor blob (16-byte aligned)
  int32_t bytes;                 // size, multiple of 16
  int16_t chunk, stage;          // angle chunk; stage = phase * nbands + band
  int16_t a0, na;                // angles [a0, a0 + na) of this block (global indices)
  uint32_t flags;                // kSeq* bits
};
constexpr uint32_t kSeqNewChunk = 1, kSeqNewStage = 2, kSeqEndChunk = 4, kSeqHasEdge = 8, kSeqHasWrap = 16;
struct TileDev {
  int enabled;
  int C, V, nAc;                 // cluster size, angle chunks, angles per chunk
  int nbands, band_rows, alloc_rows, pitch_w;   // sub-grid banding (rows of one parity), allocated rows, row pitch in words
  int xtiles, ytiles;             // EDGE-beam items: x-tiles of 16 poses, y-tiles of 48 rows
  int ygroups, wranges;          // FAST-beam items: 16-row slot groups, ranges of kTileSlots sub-grid words
  int stage_bytes;               // size of one descriptor staging buffer
  int nlevels;                   // distinct non-zero smear-kernel values if <= 4 (levelled raster without atomics), else 0
  uint32_t level[4];             // ... ascending
  int int_ties;                  // responses are monotone in the integer sum with spacing > tolerance: integer arg-max / ties
  size_t off_A, off_probs, off_stage, off_cells;   // byte offsets into dynamic shared memory (S at 0)
  int cell_cap;                  // entries of one cell-list staging buffer (= max_n), 0 = cells are read from global memory
  const uint8_t * desc;          // descriptor blob
  const TileSeq * seq;           // schedules
  const int32_t * seq_start;     // [nq * C + 1]
  const int32_t * edge;          // EDGE beams: band-relative sub-row | word << 16
  const int32_t * edge_start;    // CSR over ((q * nA + a) * 4 * nbands + stage) * 4 + m
  const int32_t * wrap2;         // EDGE beams whose columns wrap into a neighbouring row
  const int32_t * wrap2_start;   // CSR over (q * nA + a) * 4 * nbands + stage
  const int32_t * slow;          // FAR beams (device-form linear offsets)
  const int32_t * slow_start;    // [nq][nA + 1]
};

struct FineDev {
  int P, nA;
  const int32_t * offsets;   // [npairs][nA][n]
  const int32_t * posidx;    // [npairs][P]
  int32_t * sums;            // [npairs][P*nA]
};

// host state of an uploaded sweep
struct SweepHost {
  bool uploaded = false, ran = false;
  int nq = 0, npairs = 0, nitems = 0, nscans = 0, max_n = 0, n = 0, blocks = 0;
  bool do_penalize = false;
  std::vector<CorrPlan> plans;             // one coarse plan per query
  std::vector<int32_t> pair_query, pair_chain;
  // copies of what the fine pass / fallbacks need from the caller's arrays
  std::vector<b200_scan> queries, scans;
  std::vector<int32_t> chain_start;
  DevBuf<int32_t> d_offsets, d_posidx, d_scan_pt_start, d_pair_query, d_pair_chain, d_pair_item_start, d_item_pair, d_item_scan,
    d_cells, d_cell_count, d_ws_sums, d_fine_off, d_fine_pos, d_fine_sums;
  DevBuf<double> d_qgeom, d_center, d_qd, d_angpen, d_points, d_ws_probs;
  DevBuf<uint8_t> d_ws_grid, d_kernel, d_win_flag;
  DevBuf<uint16_t> d_fast_beams, d_fast_mult;
  DevBuf<int32_t> d_fast_cls, d_fast_slow, d_fast_slow_start, d_fast_wrap2, d_fast_wrap2_start, d_fast_edge, d_fast_edge_start;
  FastDev fast{};
  size_t fast_smem = 0;
  TileDev tile{};
  size_t tile_smem = 0;
  int tile_grid = 0;
  int32_t tile_info[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // enabled, C, V, nbands, band rows, refusal reason, clusters, smem KB
  DevBuf<uint8_t> d_tile_desc;
  DevBuf<TileSeq> d_tile_seq;
  DevBuf<int32_t> d_tile_seq_start, d_tile_edge, d_tile_edge_start, d_tile_wrap2, d_tile_wrap2_start, d_tile_slow, d_tile_slow_start;
  int32_t fast_info[5] = {0, 0, 0, 0, 0};   // enabled, FAST descriptors, CLIP beams, WRAP beams, reason the fast path was refused
  int fast_blocks = 0;
  DevBuf<PairOut> d_out;
  PinBuf<PairOut> h_out;
  PinBuf<uint8_t> arena;    // pinned staging of the upload's tables (sweep_stage_h2d)
  size_t arena_used = 0;
  PinBuf<int32_t> h_i;
  PinBuf<double> h_d;
  SweepDev dev{};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  int64_t h2d_bytes = 0, d2h_bytes = 0;   // bytes moved by upload / fetch since the last reset
  // pairs of the last fetch finished by the all-poses-tie closed form / handed to the single-match path
  int zero_pairs = 0, fallback_pairs = 0;
  double upload_ms[3] = {0, 0, 0};   // host wall time of the last upload: lookup tables (plans), kernel tables, whole call
  std::vector<char> zero_done, zero_exp_done;
  std::vector<double> zero_mean, zero_cov, zero_exp_mean, zero_exp_cov;   // ... and of the widest response-expansion pass
  void release();
};

}  // namespace b200

// the opaque handle of include/b200slam.h
struct b200sm {
  b200sm_params p{};
  b200::GridGeom g;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int64_t launches = 0;
  double phase_ms[6] = {0, 0, 0, 0, 0, 0};   // host-side phase times of the single-match path (b200sm_match_timing)
  int probs_side = 0;   // Grid<double> m_pSearchSpaceProbs side (M.cpp:513)

  // single-match device state
  b200::DevBuf<uint8_t> d_grid, d_kernel;
  b200::DevBuf<int32_t> d_cells, d_offsets, d_sums, d_extra;
  b200::PinBuf<int32_t> h_stage_i, h_sums;
  bool have_raster = false;
  b200::CellScratch cell_scratch;
  bool no_dedup = false;        // testing: keep one descriptor per beam in the fast sweep lists
  bool force_generic = false;   // testing: run sweeps on the generic kernel even when the fast path applies
  int sweep_kernel = 0;         // 0 = auto, 1 = legacy single-CTA fast kernel when it applies, 2 = tiled cluster kernel
  int tile_cluster = 0;         // 0 = auto, else forced cluster size (1, 2, 4, 8)
  int tile_chunks = 0;          // 0 = auto, else forced number of angle chunks

  b200::SweepHost sweep;

  void ensure_stream()
  {
    if (!stream) {
      B200_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
      own_stream = true;
    }
  }
};

namespace b200 {
// single-match entry used by the sweep for pairs the device reduction cannot finish
// (tie-list overflow, response expansion)
double do_match(b200sm * h, const b200_scan * query, const b200_scan * base, int nbase, bool pen, bool refine,
                double mean[3], double cov[9]);
int32_t device_offset(int32_t off, int data_size);
void set_grid_offset(GridGeom & g, const b200_scan * query);
double normalize_angle_difference(double minuend, double subtrahend);
}  // namespace b200

namespace b200 {
// ScanMatcher::CorrelateScan's reduction + covariance (M.cpp:775-1025) on the host from an integer volume
bool build_tile_tables(b200sm * h, SweepHost & S, cudaStream_t st);
void sweep_stage_h2d(void * dst, const void * src, size_t bytes, cudaStream_t s);
void launch_sweep_tile(b200sm * h, SweepHost & S, cudaStream_t st);
double host_epilogue(const b200sm_params & prm, const GridGeom & geom, int probs_side, const CorrPlan & pl,
                     const int32_t * sums, bool do_penalize, double mean[3], double cov[9],
                     const std::function<bool(int, int, int32_t *)> * extra_cell = nullptr);
}  // namespace b200
