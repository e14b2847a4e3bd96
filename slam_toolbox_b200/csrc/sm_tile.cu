// b200slam scan matcher, batched loop-closure sweep: the TILED CLUSTER kernel.
//
// Reference path: ScanMatcher::MatchScan -> CorrelateScan -> operator()(y) -> GetResponse
// (lib/karto_sdk/src/Mapper.cpp:534-1208, "M.cpp"), called once per candidate chain by
// MapperGraph::TryCloseLoop (M.cpp:1500-1561).
//
// k_sweep_fast (sm_sweep.cu) keeps one parity sub-grid and the whole (x, y, theta) accumulator volume of
// a pair in ONE SM's shared memory, which only holds for BASELINE's 4 m / 12 m geometry.  This kernel lifts
// both limits so that the reference's shipped geometries (loop_search_space_dimension 8 m -> 81 x 81 x 21
// poses = 551 KB of accumulators; max_laser_range 20 m -> 881..965-cell grids) run on the same word-load
// scheme:
//   * the pose volume is cut into V angle CHUNKS; a thread-block CLUSTER of C CTAs shares one pair and CTA r
//     owns chunks r, r + C, ... (perfectly balanced: every angle has the same beams);
//   * the parity sub-grid is cut into row BANDS (band rows + a halo of one pose-window height), one band is
//     resident at a time, FAST beams form one stream per (angle, parity phase, band);
//   * the beam-descriptor block of every (chunk, phase, band) STAGE is streamed into shared memory by
//     cp.async.bulk (TMA, 1-D) completing on an mbarrier, double buffered: the block of stage s + 1 lands
//     while stage s is being correlated; the hot loop reads descriptors with broadcast LDS.128;
//   * the FAST beam loop runs on the integer tensor cores (mma.sync m16n8k32 u8): the word loads are the A fragments, the beams'
//     weights and byte alignments form B;
//   * warp items (FAST: angle, slot group, word range; EDGE: angle, alignment, y-tile, x-tile) come from a dynamic shared-memory queue;
//   * the reduction (CorrelateScan M.cpp:775-829, ComputePositionalCovariance M.cpp:893-933) is distributed:
//     every CTA reduces its chunks to (best, tie list, per-cell max image), the images and tie lists are
//     combined through DISTRIBUTED SHARED MEMORY by a leader CTA that rotates from pair to pair, and a split
//     cluster barrier (arrive ... wait) lets the other CTAs start the next pair while the leader runs the
//     order-preserving (sequential) covariance sums.
// Integer sums are exact in any order, the FP64 parts keep the reference's operation order: results are bit
// identical to the reference (tests/test_matcher_gpu.py).
// Compile with -fmad=false / -ffp-contract=off.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <type_traits>
#include <vector>

#include "common.cuh"
#include "sm_math.cuh"
#include "sm_types.cuh"
#include "sm_device.cuh"
#include "sm_sweep_dev.cuh"

namespace b200 {

constexpr int kRowTiles = 6;           // row tiles of 8 rows per thread: one y-tile = 48 poses
constexpr int kYTile = 8 * kRowTiles;
constexpr int kChunkBeams = 640;       // EDGE beams accumulated in 16-bit fields before a flush (640 * 100 < 65536)
constexpr int kTileSlots = 6;          // FAST items: sub-grid words W (MMA slot groups of 16 poses) per warp item

// ------------------------------------------------------------------------------------------
// PTX helpers: mbarrier, bulk async copy (TMA 1-D), cluster barrier, distributed shared memory
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void * p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void * src, uint32_t bytes, uint32_t bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
               "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
  uint32_t done = 0;
  while (!done) {
    asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(done)
      : "r"(bar), "r"(parity)
      : "memory");
  }
}
__device__ __forceinline__ uint32_t cluster_rank()
{
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t dsmem_addr(const void * local, uint32_t rank)
{
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(local)), "r"(rank));
  return r;
}
__device__ __forceinline__ void dsmem_st_f64(uint32_t a, double v) { asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ void dsmem_st_s32(uint32_t a, int v) { asm volatile("st.shared::cluster.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ int dsmem_ld_s32(uint32_t a)
{
  int v;
  asm volatile("ld.shared::cluster.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory");
  return v;
}
__device__ __forceinline__ double dsmem_ld_f64(uint32_t a)
{
  double v;
  asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory");
  return v;
}

// 32-bit shared-memory load from a shared-window byte address (keeps the window base folded into the per-lane base register)
__device__ __forceinline__ uint32_t lds_u32(uint32_t a)
{
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}

// D += A B on the integer tensor cores: m16n8k32, A (16 x 32) and B (32 x 8) unsigned bytes, s32 accumulators
__device__ __forceinline__ void mma_u8(int (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1)
{
  asm("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
      : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
      : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ uint32_t even_bytes_t(uint32_t w) { return __byte_perm(w, 0, 0x4240); }   // [b0, 0, b2, 0]
__device__ __forceinline__ uint32_t odd_bytes_t(uint32_t w) { return __byte_perm(w, 0, 0x4341); }    // [b1, 0, b3, 0]

// best / tie summary of a set of poses (one chunk, one CTA, or the whole pair)
struct TieRes {
  double L;        // best response
  double L2;       // highest chunk best strictly below L (ambiguity test: DoubleEqual(L2, L) -> the host decides)
  int cnt;         // number of poses with DoubleEqual(response, L)
  int sum0;        // integer sum of the first tie
  int ties[kMaxTies];
};

// folds b into a (both lists ascending in the flat pose index)
__device__ void tie_merge(TieRes & a, const double bL, const double bL2, const int bcnt, const int bsum0, const int * bties)
{
  if (bL == a.L) {
    int out[kMaxTies];
    const int na = a.cnt < kMaxTies ? a.cnt : kMaxTies, nb = bcnt < kMaxTies ? bcnt : kMaxTies;
    int i = 0, j = 0, k = 0;
    while (k < kMaxTies && (i < na || j < nb)) {
      if (j >= nb || (i < na && a.ties[i] < bties[j])) out[k++] = a.ties[i++];
      else out[k++] = bties[j++];
    }
    if (nb > 0 && (na == 0 || bties[0] < a.ties[0])) a.sum0 = bsum0;
    for (int t = 0; t < k; ++t) a.ties[t] = out[t];
    a.cnt += bcnt;
    a.L2 = bL2 > a.L2 ? bL2 : a.L2;
  } else if (bL > a.L) {
    double l2 = a.L > a.L2 ? a.L : a.L2;
    l2 = bL2 > l2 ? bL2 : l2;
    a.L = bL; a.L2 = l2; a.cnt = bcnt; a.sum0 = bsum0;
    const int nb = bcnt < kMaxTies ? bcnt : kMaxTies;
    for (int t = 0; t < nb; ++t) a.ties[t] = bties[t];
  } else {
    double l2 = bL > a.L2 ? bL : a.L2;
    a.L2 = bL2 > l2 ? bL2 : l2;
  }
}

struct TileShared {
  unsigned long long bar[4];       // [0..1] descriptor staging buffers, [2..3] cell-list staging buffers
  uint8_t kern[256];               // the smear kernel's taps (when ksize^2 <= 256)
  int ctr[2];
  double dscratch[32];
  int iscratch[32];
  TieRes chunk;                    // result of the chunk just reduced
  TieRes res;                      // this CTA's running result over its chunks
  // written by the other CTAs of the cluster when this CTA is the pair's leader
  double rankL[kTileMaxCluster], rankL2[kTileMaxCluster];
  int rankCnt[kTileMaxCluster], rankSum0[kTileMaxCluster];
  int rankTies[kTileMaxCluster][kMaxTies];
  double avg[2];
  double acc[4];
  int ok;
};

// ------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------
// kPitchW = the sub-grid row pitch in words as a compile-time constant (0 = take it from TileDev): with a constant pitch the 24
// loads of a 4-beam step address as [descriptor register + immediate]; with a run-time pitch every load costs an extra IMAD
// (20 % of the beam loop).  The pitches of the four shipped geometry combinations are instantiated.
template <int kPitchW>
__global__ void __launch_bounds__(kTileThreads, 1) k_sweep_tile(SweepDev d, TileDev f)
{
  extern __shared__ __align__(128) unsigned char s_raw[];
  __shared__ TileShared sh;
  uint32_t * S = reinterpret_cast<uint32_t *>(s_raw);
  uint8_t * S8 = s_raw;
  int32_t * A = reinterpret_cast<int32_t *>(s_raw + f.off_A);
  double * probs = reinterpret_cast<double *>(s_raw + f.off_probs);      // per-cell max response image (FP64 path) ...
  int32_t * iprobs = reinterpret_cast<int32_t *>(s_raw + f.off_probs);   // ... or per-cell max integer sum (integer path: half the bytes)
  const int C = f.C;
  const uint32_t rank = C > 1 ? cluster_rank() : 0u;
  const int cluster_id = blockIdx.x / C, nclusters = gridDim.x / C;
  const int nX = d.nX, nY = d.nY, nA = d.nA, P = nX * nY;
  const int half = d.ksize / 2, taps = d.ksize * d.ksize;
  const int tid = threadIdx.x, lane = tid & 31;
  const int y_l = lane >> 2, j_l = lane & 3;
  const int pitch_w = kPitchW ? kPitchW : f.pitch_w, pitchB = pitch_w * 4;
  const int sub_words = f.alloc_rows * pitch_w;
  const int nb = f.nbands;
  const uint32_t bar0 = smem_u32(&sh.bar[0]);
  const uint32_t stg0 = smem_u32(s_raw + f.off_stage);

  if (tid == 0) {
    mbar_init(bar0, 1);
    mbar_init(bar0 + 8, 1);
    mbar_init(bar0 + 16, 1);
    mbar_init(bar0 + 24, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    sh.ctr[0] = 0; sh.ctr[1] = 0;
  }
  const bool kern_smem = taps <= 256;
  if (kern_smem && tid < taps) sh.kern[tid] = d.kern[tid];
  const uint8_t * kern = kern_smem ? sh.kern : d.kern;
  __syncthreads();
  if (C > 1) { cluster_arrive(); cluster_wait(); }   // every CTA of the cluster is running before any remote access

  uint32_t cnt = 0;          // descriptor blocks consumed so far (buffer = cnt & 1, mbarrier parity = (cnt >> 1) & 1)
  bool pending_wait = false; // a cluster barrier arrive without its wait yet (split barrier across pairs)
  auto issue = [&](const TileSeq * e, uint32_t buf) {
    mbar_expect_tx(bar0 + 8 * buf, (uint32_t)e->bytes);
    bulk_g2s(stg0 + buf * (uint32_t)f.stage_bytes, f.desc + e->off, (uint32_t)e->bytes, bar0 + 8 * buf);
  };
  // the valid-point cells of a pair's FIRST scan (what every stage's raster reads: 4.3 KB for 1081 beams) are staged in shared
  // memory by a bulk copy too, one pair ahead -- a stage then starts without a global-memory round trip
  const uint32_t cel0 = smem_u32(s_raw + f.off_cells);
  const uint32_t cell_bytes = (uint32_t)f.cell_cap * 4u;
  auto issue_cells = [&](int pr, uint32_t buf) {
    const int it = min(d.pair_item_start[pr], max(d.nitems - 1, 0));
    mbar_expect_tx(bar0 + 16 + 8 * buf, cell_bytes);
    bulk_g2s(cel0 + buf * cell_bytes, d.cells + (size_t)it * d.max_n, cell_bytes, bar0 + 16 + 8 * buf);
  };
  if (cluster_id < d.npairs && tid == 0) {
    const int q0 = d.pair_query[cluster_id];
    issue(f.seq + f.seq_start[q0 * C + rank], 0);
    if (f.cell_cap) issue_cells(cluster_id, 0);
  }

  int iter = 0;
  for (int pair = cluster_id; pair < d.npairs; pair += nclusters, ++iter) {
    const int q = d.pair_query[pair];
    const uint32_t leader = (uint32_t)(iter % C);
    const TileSeq * seq = f.seq + f.seq_start[q * C + rank];
    const int nseq = f.seq_start[q * C + rank + 1] - f.seq_start[q * C + rank];
    const int it0 = d.pair_item_start[pair], it1 = d.pair_item_start[pair + 1];
    bool first_chunk = true;
    const int32_t * cells0 = d.cells + (size_t)it0 * d.max_n;
    const int ncell0 = it0 < it1 ? d.cell_count[it0] : 0;   // read once per pair, not once per stage
    if (f.cell_cap) {
      if (tid == 0 && pair + nclusters < d.npairs) issue_cells(pair + nclusters, (uint32_t)((iter + 1) & 1));
      mbar_wait(bar0 + 16 + 8 * (iter & 1), (uint32_t)((iter >> 1) & 1));
      cells0 = reinterpret_cast<const int32_t *>(s_raw + f.off_cells + (size_t)(iter & 1) * cell_bytes);
    }

    for (int si = 0; si < nseq; ++si) {
      const TileSeq e = seq[si];
      const int chunk_a0 = e.chunk * f.nAc;
      const int chunk_na = min(f.nAc, nA - chunk_a0);
      const int ph = e.stage / nb, band = e.stage - ph * nb;
      const int pp = ph & 1, pq = ph >> 1;
      const int band_r0 = band * f.band_rows;
      if (e.flags & kSeqNewChunk)
        for (int i = tid; i < chunk_na * P; i += kTileThreads) A[i] = 0;
      if (e.flags & kSeqNewStage) {
        {
          uint4 * S4 = reinterpret_cast<uint4 *>(s_raw);
          const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
          for (int i = tid; i < (sub_words >> 2); i += kTileThreads) S4[i] = zero;   // pitch_w is a multiple of 4
        }
        __syncthreads();
        // ---- raster: taps landing on (pp, pq) cells of this band (AddScan / SmearPoint, M.cpp:1080-1104, M.h:1152-1183);
        //      one thread per valid point, only the kernel rows / columns of this phase's parity ----
        // Max-stamp without atomics when the kernel has few distinct values (3 x 3: {6, 25, 100}): one pass per value in ascending
        // order, plain byte stores (all writers of a pass store the same value, a later pass overwrites with a larger one), a
        // barrier between passes.  Neighbouring beams end in neighbouring cells, so a CAS loop on the shared 32-bit words
        // serialises up to 8 lanes per word (3.4 us per stage measured); kernels with more values keep it.
        const int nlev = f.nlevels;
        for (int lv = 0; lv < (nlev > 0 ? nlev : 1); ++lv) {
          const uint32_t want = nlev > 0 ? f.level[lv] : 0u;
          for (int it = it0; it < it1; ++it) {
            const int32_t * cl = it == it0 ? cells0 : d.cells + (size_t)it * d.max_n;
            const int ncell = it == it0 ? ncell0 : d.cell_count[it];
            for (int t = tid; t < ncell; t += kTileThreads) {
              const int32_t cell = cl[t];
              if (cell < 0) continue;
              const int cx = (cell & 0xFFFF) + d.roi_x - half, cy = (cell >> 16) + d.roi_y - half;
              for (int ky = (cy ^ pq) & 1; ky < d.ksize; ky += 2) {
                const int rel = ((cy + ky) >> 1) - band_r0;
                if ((unsigned)rel >= (unsigned)f.alloc_rows) continue;
                for (int kx = (cx ^ pp) & 1; kx < d.ksize; kx += 2) {
                  const uint32_t kv = kern[ky * d.ksize + kx];
                  if (nlev > 0) { if (kv == want) S8[rel * pitchB + ((cx + kx) >> 1)] = (uint8_t)kv; }
                  else if (kv) atomic_max_u8(S8 + rel * pitchB + ((cx + kx) >> 1), kv);
                }
              }
            }
          }
          if (lv + 1 < nlev) __syncthreads();
        }
      }
      if (e.flags & (kSeqNewChunk | kSeqNewStage)) __syncthreads();
      // ---- prefetch the next descriptor block (this pair's, or the first of this cluster's next pair) ----
      if (tid == 0) {
        const TileSeq * nxt = nullptr;
        if (si + 1 < nseq) nxt = seq + si + 1;
        else if (pair + nclusters < d.npairs) nxt = f.seq + f.seq_start[d.pair_query[pair + nclusters] * C + rank];
        if (nxt) issue(nxt, (cnt + 1) & 1);
      }
      mbar_wait(bar0 + 8 * (cnt & 1), (cnt >> 1) & 1);
      const unsigned char * stg = s_raw + f.off_stage + (size_t)(cnt & 1) * f.stage_bytes;
      // block: [per angle (first step, end step, owns the angle's EDGE beams) | angles by descending stream length | 64-byte steps]
      const int32_t * tbl = reinterpret_cast<const int32_t *>(stg);
      const uint8_t * order = stg + (size_t)e.na * 12;
      const uint4 * steps = reinterpret_cast<const uint4 *>(stg + (((size_t)e.na * 13 + 15) & ~(size_t)15));
      // ---- warp items from the shared queue: FAST (angle, 16-row slot group, word range), then EDGE (angle, alignment,
      //      y-tile, x-tile) ----
      const int per_angle = f.ygroups * f.wranges;
      const int fast_items = e.na * per_angle;
      const int tiles = f.ytiles * f.xtiles;
      const int nitems = fast_items + ((e.flags & kSeqHasEdge) ? e.na * 4 * tiles : 0);
      for (;;) {
        int item = 0;
        if (lane == 0) item = atomicAdd(&sh.ctr[cnt & 1], 1);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= nitems) break;
        if (item < fast_items) {
          // FAST beams on the integer tensor cores: per 8-beam step one m16n8k32 u8 MMA per slot W of the item.  A row = pose
          // slot (rows g and g + 8 of the slot group at sub-grid word W), k = 4 * beam + byte: the lane's LDS.32 of a beam's
          // word IS its A fragment.  B[4b + j][n] = w_b * [j - m_b + 4 == n], so C[slot][n] = sum_b w_b * cell(c_b + 4W - 4 + n)
          // is the exact integer sum of pose x = 4W - 4 + n (n = 1..7; one stream serves every byte alignment m_b).
          const int gi = item / per_angle, ti = item - gi * per_angle;
          const int al = order[gi];
          const int s0 = tbl[3 * al], s1 = tbl[3 * al + 1];
          if (s0 == s1) continue;
          const int yg = ti / f.wranges, wr = ti - yg * f.wranges;
          const int g = lane >> 2, t4 = lane & 3;
          uint32_t base = smem_u32(S8) + (uint32_t)(((16 * yg + g) * pitch_w + kTileSlots * wr) * 4);
          asm volatile("" : "+r"(base));
          // B fragment (k = 4 t4 + j, column n = g) of a beam whose weight sits in byte m of V: byte j takes byte j + 4 - g of V
          uint32_t sel = 0;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int k = j + 4 - g;
            sel |= (uint32_t)((k >= 0 && k <= 3) ? k : 4) << (4 * j);
          }
          int acc[kTileSlots][4];
#pragma unroll
          for (int s = 0; s < kTileSlots; ++s) acc[s][0] = acc[s][1] = acc[s][2] = acc[s][3] = 0;
          // the lane's descriptor: byte offsets and V words of beams t4 and t4 + 4 (the 4 beams of a k-quad have distinct word
          // offsets mod 4, the row pitch is 4 x odd words: the 32 lanes of every load hit 32 distinct banks)
          const uint4 * de = steps + 4 * s1;
          for (const uint4 * dp = steps + 4 * s0 + t4; dp < de; dp += 4) {
            const uint4 dd = *dp;
            const uint32_t oa = base + dd.x, ob = base + dd.y;
            const uint32_t b0 = __byte_perm(dd.z, 0, sel), b1 = __byte_perm(dd.w, 0, sel);
#pragma unroll
            for (int s = 0; s < kTileSlots; ++s)
              mma_u8(acc[s], lds_u32(oa + 4 * s), lds_u32(oa + 4 * s + 8 * pitchB), lds_u32(ob + 4 * s), lds_u32(ob + 4 * s + 8 * pitchB),
                     b0, b1);
          }
          // once per item: C (rows g / g + 8, columns 2 t4 / 2 t4 + 1) into the accumulators; slots W and W + 1 share poses
          // 4W + 1 .. 4W + 3, the shared-memory atomics add both
          int32_t * Arow = A + (size_t)(e.a0 + al - chunk_a0) * P;
#pragma unroll
          for (int s = 0; s < kTileSlots; ++s) {
            const int x = 4 * (kTileSlots * wr + s) - 4 + 2 * t4;
#pragma unroll
            for (int hh = 0; hh < 2; ++hh) {
              const int y = 16 * yg + g + 8 * hh;
              if (y >= nY) continue;
              if (acc[s][2 * hh] && (unsigned)x < (unsigned)nX) atomicAdd(Arow + y * nX + x, acc[s][2 * hh]);
              if (acc[s][2 * hh + 1] && (unsigned)(x + 1) < (unsigned)nX) atomicAdd(Arow + y * nX + x + 1, acc[s][2 * hh + 1]);
            }
          }
          continue;
        }
        // EDGE beams (window partly outside the grid) of one (angle, alignment, tile): word loads with rows / words outside the
        // band allocation masked (they index outside [0, data_size) or wrap in the reference; the wrapped part is added from the
        // wrap2 list below).  Rows / words inside the allocation but beyond the valid cells are zero padding.
        const int ei = item - fast_items;
        const int gi = ei / tiles, ti = ei - gi * tiles;
        const int al = gi >> 2, m = gi & 3;
        if (!tbl[3 * al + 2]) continue;   // the angle's stream started in an earlier block, which took its EDGE beams
        const int a = e.a0 + al;
        const int32_t * es = f.edge_start + (((size_t)q * nA + a) * 4 * nb + e.stage) * 4 + m;
        int eb = es[0];
        const int ee = es[1];
        if (eb == ee) continue;
        const int yt = ti / f.xtiles, xt = ti - yt * f.xtiles;
        int32_t * Arow = A + (size_t)(a - chunk_a0) * P;
        const int ybase = y_l + kYTile * yt;
        const int x0 = 4 * (4 * xt + j_l) - m;
        while (eb < ee) {
          const int ce = min(ee, eb + kChunkBeams);
          uint32_t T0[kRowTiles], T1[kRowTiles];
#pragma unroll
          for (int r = 0; r < kRowTiles; ++r) { T0[r] = 0; T1[r] = 0; }
          for (int b0 = eb; b0 < ce; b0 += 32) {
            const int cn = min(32, ce - b0);
            const int32_t mine = (lane < cn) ? f.edge[b0 + lane] : 0;
            for (int k = 0; k < cn; ++k) {
              const int32_t ev = __shfl_sync(0xffffffffu, mine, k);
              const int row0 = (int)(int16_t)(ev & 0xFFFF) + ybase, wq = (ev >> 16) + 4 * xt + j_l;
              const bool cv = (unsigned)wq < (unsigned)pitch_w;
#pragma unroll
              for (int r = 0; r < kRowTiles; ++r) {
                const int row = row0 + 8 * r;
                const uint32_t w = (cv && (unsigned)row < (unsigned)f.alloc_rows) ? S[row * pitch_w + wq] : 0u;
                T0[r] += even_bytes_t(w);
                T1[r] += odd_bytes_t(w);
              }
            }
          }
          eb = ce;
          // 16-bit fields into the accumulators
          uint32_t any = 0;
#pragma unroll
          for (int r = 0; r < kRowTiles; ++r) any |= T0[r] | T1[r];
          if (!__any_sync(0xffffffffu, any != 0)) continue;
#pragma unroll
          for (int r = 0; r < kRowTiles; ++r) {
            const int y = ybase + 8 * r;
            if (y >= nY || (T0[r] | T1[r]) == 0) continue;
            int32_t * dst = Arow + y * nX + x0;
            const int v0 = T0[r] & 0xFFFF, v1 = T1[r] & 0xFFFF, v2 = T0[r] >> 16, v3 = T1[r] >> 16;
            if (v0 && (unsigned)(x0 + 0) < (unsigned)nX) atomicAdd(dst + 0, v0);
            if (v1 && (unsigned)(x0 + 1) < (unsigned)nX) atomicAdd(dst + 1, v1);
            if (v2 && (unsigned)(x0 + 2) < (unsigned)nX) atomicAdd(dst + 2, v2);
            if (v3 && (unsigned)(x0 + 3) < (unsigned)nX) atomicAdd(dst + 3, v3);
          }
        }
      }
      if (e.flags & kSeqNewStage) {
        // ---- wrapped part of EDGE beams (row parity flipped list): poses whose column left [0, stride) by less than a
        //      stride read the neighbouring row at column -/+ stride (linear index, M.cpp:1192-1200) ----
        const int32_t * ws = f.wrap2_start + ((size_t)q * nA + chunk_a0) * 4 * nb + e.stage;
        const bool has_wrap = (e.flags & kSeqHasWrap) != 0;
        if (has_wrap) {
          for (int p = tid; p < P; p += kTileThreads) {
            const int ex = 2 * (p % nX), ey = 2 * (p / nX);
            for (int al = 0; al < chunk_na; ++al) {
              int acc = 0;
              for (int bi = ws[(size_t)al * 4 * nb]; bi < ws[(size_t)al * 4 * nb + 1]; ++bi) {
                const int32_t ev = f.wrap2[bi];
                const int Xb = (int)(int16_t)(ev & 0xFFFF), Yb = ev >> 16;
                const int col = Xb + ex;
                if ((unsigned)col < (unsigned)d.stride) continue;
                const int r2 = Yb + ey + (col < 0 ? -1 : 1);
                const int c2 = col + (col < 0 ? d.stride : -d.stride);
                if ((unsigned)r2 >= (unsigned)d.height) continue;
                const int rel = (r2 >> 1) - band_r0;
                if ((unsigned)rel >= (unsigned)f.alloc_rows) continue;
                acc += S8[rel * pitchB + (c2 >> 1)];
              }
              if (acc) atomicAdd(A + (size_t)al * P + p, acc);
            }
          }
        }
        // ---- FAR beams (column offsets of a stride or more): pose by pose on the linear index; a row belongs to the band
        //      whose own rows contain it ----
        const int32_t * ss = f.slow_start + (size_t)q * (nA + 1);
        if (ss[nA] - ss[0] > 0) {
          const int32_t * pos = d.posidx + (size_t)q * P;
          const int own_hi = (band == nb - 1) ? 0x7FFFFFFF : f.band_rows;
          for (int al = 0; al < chunk_na; ++al) {
            const int sb = ss[chunk_a0 + al], se = ss[chunk_a0 + al + 1];
            const int work = (se - sb) * P;
            for (int t = tid; t < work; t += kTileThreads) {
              const int bi = t / P, p = t - bi * P;
              const int idx = pos[p] + f.slow[sb + bi];
              if ((unsigned)idx >= (unsigned)d.data_size) continue;
              const int row = idx / d.stride, col = idx - row * d.stride;
              if ((col & 1) != pp || (row & 1) != pq) continue;
              const int rel = (row >> 1) - band_r0;
              if (rel < 0 || rel >= own_hi || rel >= f.alloc_rows) continue;
              const int v = S8[rel * pitchB + (col >> 1)];
              if (v) atomicAdd(A + (size_t)al * P + p, v);
            }
          }
        }
      }
      if (tid == 0) sh.ctr[(cnt + 1) & 1] = 0;
      __syncthreads();
      ++cnt;

      if (e.flags & kSeqEndChunk) {
        // ================= chunk reduction: per-cell max image, best response, ordered tie list =================
        if (pending_wait) { cluster_wait(); pending_wait = false; }   // the previous pair's leader has read our image
        double lbest = -1.0;
        int smax = -1;
        if (f.int_ties) {
          // responses are sum / norm: monotone in the sum and two different sums differ by more than the tie tolerance
          for (int p = tid; p < P; p += kTileThreads) {
            int sm = 0;
            for (int al = 0; al < chunk_na; ++al) { const int s = A[(size_t)al * P + p]; sm = s > sm ? s : sm; }
            smax = sm > smax ? sm : smax;                       // this chunk's best
            if (!first_chunk) { const int o = iprobs[p]; sm = o > sm ? o : sm; }
            iprobs[p] = sm;                                     // running per-cell maximum over the chunks so far
          }
          for (int o = 16; o > 0; o >>= 1) { const int t = __shfl_xor_sync(0xffffffffu, smax, o); smax = t > smax ? t : smax; }
          __syncthreads();
          if (lane == 0) sh.iscratch[tid >> 5] = smax;
          __syncthreads();
          for (int i = 0; i < kTileThreads / 32; ++i) smax = sh.iscratch[i] > smax ? sh.iscratch[i] : smax;
          __syncthreads();
          lbest = (double)smax;
          lbest /= d.norm;
        } else {
          for (int p = tid; p < P; p += kTileThreads) {
            const int x = p % nX, y = p / nX;
            double pm = first_chunk ? 0.0 : probs[p];   // Grid<double>::Clear() initial value, M.cpp:727
            for (int al = 0; al < chunk_na; ++al) {
              const double r = pose_response(d, q, A[(size_t)al * P + p], x, y, chunk_a0 + al);
              pm = r > pm ? r : pm;
              lbest = r > lbest ? r : lbest;
            }
            probs[p] = pm;
          }
          lbest = block_max(lbest, sh.dscratch);
        }
        // ordered tie list: poses with DoubleEqual(response, best) in array order (M.cpp:807-817); every thread owns a
        // contiguous run of cells so that ranks follow array order
        const int per = (P + kTileThreads - 1) / kTileThreads;
        int t_own;   // the thread index read here, not the kernel-wide one: ptxas kept tid * per live across the beam loop (a spill)
        asm volatile("mov.u32 %0, %%tid.x;" : "=r"(t_own));
        const int p0 = min(P, t_own * per), p1 = min(P, p0 + per);
        int c = 0;
        for (int p = p0; p < p1; ++p) {
          const int x = p % nX, y = p / nX;
          for (int al = 0; al < chunk_na; ++al) {
            const int s = A[(size_t)al * P + p];
            const bool tie = f.int_ties ? (s == smax) : double_equal(pose_response(d, q, s, x, y, chunk_a0 + al), lbest);
            if (tie) ++c;
          }
        }
        int total = 0;
        int rk = block_exclusive_scan(c, sh.iscratch, total);
        if (c > 0 && rk < kMaxTies) {
          for (int p = p0; p < p1 && rk < kMaxTies; ++p) {
            const int x = p % nX, y = p / nX;
            for (int al = 0; al < chunk_na && rk < kMaxTies; ++al) {
              const int s = A[(size_t)al * P + p];
              const bool tie = f.int_ties ? (s == smax) : double_equal(pose_response(d, q, s, x, y, chunk_a0 + al), lbest);
              if (tie) {
                if (rk == 0) sh.chunk.sum0 = s;
                sh.chunk.ties[rk++] = p * nA + chunk_a0 + al;
              }
            }
          }
        }
        __syncthreads();
        if (tid == 0) {
          if (first_chunk) {
            sh.res.L = lbest; sh.res.L2 = -1e300; sh.res.cnt = total; sh.res.sum0 = sh.chunk.sum0;
            for (int t = 0; t < kMaxTies; ++t) sh.res.ties[t] = sh.chunk.ties[t];
          } else {
            tie_merge(sh.res, lbest, -1e300, total, sh.chunk.sum0, sh.chunk.ties);
          }
        }
        first_chunk = false;
        __syncthreads();
      }
    }

    // ================= pair reduction across the cluster =================
    if (C > 1) {
      if (tid < 32) {
        const uint32_t base = dsmem_addr(&sh, leader);
        const uint32_t off = smem_u32(&sh);
        if (tid == 0) {
          dsmem_st_f64(base + (smem_u32(&sh.rankL[rank]) - off), sh.res.L);
          dsmem_st_f64(base + (smem_u32(&sh.rankL2[rank]) - off), sh.res.L2);
          dsmem_st_s32(base + (smem_u32(&sh.rankCnt[rank]) - off), sh.res.cnt);
          dsmem_st_s32(base + (smem_u32(&sh.rankSum0[rank]) - off), sh.res.sum0);
        }
        if (tid < kMaxTies) dsmem_st_s32(base + (smem_u32(&sh.rankTies[rank][tid]) - off), sh.res.ties[tid]);
      }
      cluster_arrive();
      cluster_wait();
    }
    if (rank == leader) {
      PairOut & out = d.out[pair];
      if (tid == 0) {
        TieRes r = sh.res;
        if (C > 1) {
          r.L = sh.rankL[0]; r.L2 = sh.rankL2[0]; r.cnt = sh.rankCnt[0]; r.sum0 = sh.rankSum0[0];
          for (int t = 0; t < kMaxTies; ++t) r.ties[t] = sh.rankTies[0][t];
          for (int s = 1; s < C; ++s) tie_merge(r, sh.rankL[s], sh.rankL2[s], sh.rankCnt[s], sh.rankSum0[s], sh.rankTies[s]);
        }
        // a chunk best within the tie tolerance of (but not equal to) the pair's best could hold further ties: leave the
        // pair to the single-match path (tie_count -1).  Cannot happen on the integer path.
        const bool ambiguous = double_equal(r.L2, r.L);
        const int m = r.cnt < kMaxTies ? r.cnt : kMaxTies;
        out.best = r.L;
        out.best_sum = r.cnt > 0 ? r.sum0 : 0;
        out.tie_count = ambiguous ? -1 : r.cnt;
        for (int t = 0; t < m; ++t) out.ties[t] = r.ties[t];
        double ax = 0.0, ay = 0.0;
        for (int t = 0; t < m; ++t) {   // averagePosition += pose position, in order (M.cpp:809)
          const int p = r.ties[t] / nA;
          ax += d.newx[q * nX + p % nX];
          ay += d.newy[q * nY + p / nX];
        }
        if (r.cnt > 0) { ax /= r.cnt; ay /= r.cnt; }
        out.avg_x = ax; out.avg_y = ay;
        sh.avg[0] = ax; sh.avg[1] = ay;
        // the covariance sums are only used for an unambiguous, non-overflowing tie set with best >= tolerance (M.cpp:886-891)
        sh.ok = (!ambiguous && r.cnt > 0 && r.cnt <= kMaxTies && !(r.L < kTolerance)) ? 1 : 0;
        sh.acc[0] = sh.acc[1] = sh.acc[2] = sh.acc[3] = 0.0;
        sh.res.L = r.L;
      }
      __syncthreads();
      if (sh.ok && C > 1) {
        // per-cell max over the other CTAs' images, through distributed shared memory
        for (uint32_t s = 0; s < (uint32_t)C; ++s) {
          if (s == rank) continue;
          const uint32_t rp = dsmem_addr(probs, s);
          if (f.int_ties) {
            for (int p = tid; p < P; p += kTileThreads) {
              const int v = dsmem_ld_s32(rp + 4u * (uint32_t)p);
              if (v > iprobs[p]) iprobs[p] = v;
            }
          } else {
            for (int p = tid; p < P; p += kTileThreads) {
              const double v = dsmem_ld_f64(rp + 8u * (uint32_t)p);
              if (v > probs[p]) probs[p] = v;
            }
          }
        }
      }
    }
    if (C > 1) { cluster_arrive(); pending_wait = true; }   // the others may reuse their images once the leader has arrived
    if (rank == leader) {
      __syncthreads();
      PairOut & out = d.out[pair];
      if (sh.ok) {
        // positional covariance accumulators (M.cpp:893-933): cells with response >= best - 0.1, summed in (y, x) order.
        // Terms are formed in parallel, compacted in order, then added sequentially so the additions happen in the
        // reference's order.  The term buffer reuses S and A (free now), a sub-range of cells at a time.
        const double best = sh.res.L;
        const double dx = sh.avg[0] - d.center[q * 3 + 0], dy = sh.avg[1] - d.center[q * 3 + 1];
        double * terms = reinterpret_cast<double *>(s_raw);
        const int cap = (int)(f.off_probs / 32);
        for (int c0 = 0; c0 < P; c0 += cap) {
          const int c1 = min(P, c0 + cap), len = c1 - c0;
          const int per = (len + kTileThreads - 1) / kTileThreads;
          const int p0 = c0 + min(len, tid * per), p1 = min(c1, p0 + per);
          int c2 = 0;
          auto cell_max = [&](int p) -> double {   // the m_pSearchSpaceProbs value of cell p
            if (!f.int_ties) return probs[p];
            double v = (double)iprobs[p];
            v /= d.norm;
            return v;
          };
          for (int p = p0; p < p1; ++p) if (cell_max(p) >= (best - 0.1)) ++c2;
          int tot2 = 0;
          int r2 = block_exclusive_scan(c2, sh.iscratch, tot2);
          for (int p = p0; p < p1; ++p) {
            const double resp = cell_max(p);
            if (resp >= (best - 0.1)) {
              const double x = d.xrel[q * nX + p % nX], y = d.yrel[q * nY + p / nX];
              terms[4 * r2 + 0] = resp;
              terms[4 * r2 + 1] = (square(x - dx) * resp);
              terms[4 * r2 + 2] = ((x - dx) * (y - dy) * resp);
              terms[4 * r2 + 3] = (square(y - dy) * resp);
              ++r2;
            }
          }
          __syncthreads();
          if (tid == 0) {
            double norm = sh.acc[0], axx = sh.acc[1], axy = sh.acc[2], ayy = sh.acc[3];
            for (int t = 0; t < tot2; ++t) {
              norm += terms[4 * t + 0];
              axx += terms[4 * t + 1];
              axy += terms[4 * t + 2];
              ayy += terms[4 * t + 3];
            }
            sh.acc[0] = norm; sh.acc[1] = axx; sh.acc[2] = axy; sh.acc[3] = ayy;
          }
          __syncthreads();
        }
      }
      if (tid == 0) { out.norm = sh.acc[0]; out.acc_xx = sh.acc[1]; out.acc_xy = sh.acc[2]; out.acc_yy = sh.acc[3]; }
      __syncthreads();
    }
  }
  if (pending_wait) cluster_wait();   // nobody leaves while a leader may still read its shared memory
}

// ------------------------------------------------------------------------------------------
// host side: plan (chunks, bands, cluster size), descriptor blocks, launch
// ------------------------------------------------------------------------------------------
// the instantiation for a row pitch: 4 m / 12 m -> 76 words, 8 m / 12 m -> 92, 4 m / 20 m -> 116, 8 m / 20 m -> 132; anything else
// runs the run-time-pitch version
static const void * tile_kernel_for(int pitch_w)
{
  switch (pitch_w) {
    case 76: return (const void *)k_sweep_tile<76>;
    case 92: return (const void *)k_sweep_tile<92>;
    case 116: return (const void *)k_sweep_tile<116>;
    case 132: return (const void *)k_sweep_tile<132>;
    default: return (const void *)k_sweep_tile<0>;
  }
}

static int env_int(const char * name, int dflt)
{
  const char * v = std::getenv(name);
  return (v && *v) ? std::atoi(v) : dflt;
}

// the first scan's cell list is staged when one list is small enough and its stride keeps the bulk copy 16-byte aligned
static inline bool d_max_n_ok(int max_n) { return max_n > 0 && (max_n & 3) == 0 && max_n <= 4096; }

static inline int floor_div(int a, int b) { return a >= 0 ? a / b : -((-a + b - 1) / b); }

bool build_tile_tables(b200sm * h, SweepHost & S, cudaStream_t st)
{
  const GridGeom & g = h->g;
  const CorrPlan & p0 = S.plans[0];
  const int nX = p0.nX, nY = p0.nY, nA = p0.nA, n = p0.n, nq = S.nq, P = nX * nY;
  TileDev & T = S.tile;
  T = TileDev{};
  for (int i = 0; i < 8; ++i) S.tile_info[i] = 0;
  auto bail = [&](int why) { S.tile_info[5] = why; return false; };
  if (g.order_dependent) return bail(1);                 // AddScan's occupancy test makes the raster sequential (generic kernel)
  if ((g.stride & 1) || nA < 1 || nA > 4096) return bail(2);
  for (int q = 0; q < nq; ++q) {
    const CorrPlan & pl = S.plans[q];
    for (int k = 1; k < nX; ++k) if (pl.xs[k] != pl.xs[0] + 2 * k) return bail(6);   // coarse step must be exactly 2 cells
    for (int k = 1; k < nY; ++k) if (pl.ys[k] != pl.ys[0] + 2 * k) return bail(7);
  }
  // ---- geometry of one parity sub-grid ----
  // Row pitch: a sub-grid row (stride / 2 bytes) + 16 bytes, rounded up to 4 x odd words so that the 8 rows x 4 words of an
  // EDGE load, and the 8 rows x 4 word residues of a FAST k-quad load, hit 32 distinct banks (76 / 92 / 116 / 132 words at the
  // shipped geometries).  A FAST item reads kTileSlots * wranges words from a beam's word on (an EDGE item 4 * xtiles, masked
  // to the pitch), which can run past the row's end: those bytes only feed poses x >= nX, which the flush drops, and past
  // the last allocated row they stay inside the allocation by the overrun below.
  int pitch_w = (g.stride / 2 + 16 + 3) / 4;
  while ((pitch_w & 7) != 4) ++pitch_w;
  const int xtiles = (nX + 3 + 15) / 16, ytiles = (nY + kYTile - 1) / kYTile;
  // FAST slots: word W serves poses 4W - 3 .. 4W + 3, so words 0 .. (nX + 2) / 4 cover x = 0 .. nX - 1
  const int ygroups = (nY + 15) / 16, wranges = ((nX + 2) / 4 + 1 + kTileSlots - 1) / kTileSlots;
  const int rows_valid = (g.height + 1) / 2;
  const int halo = nY + 2;                               // rows a beam window reaches below its base row (idle row tiles are clamped) + the wrapped row
  const int base_rows = std::max(1, rows_valid - nY + 1);   // distinct base rows of beams whose window is inside the grid
  // ---- choose the number of angle chunks V and of bands ----
  int sms = 148, dev = 0;
  B200_CUDA(cudaGetDevice(&dev));
  B200_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  int want_c = h->tile_cluster > 0 ? h->tile_cluster : env_int("B200_SWEEP_CLUSTER", 0);
  if (want_c <= 0) {
    // throughput mode (one CTA per pair) once the batch fills the GPU, otherwise spread a pair over a cluster
    want_c = 1;
    while (want_c < kTileMaxCluster && S.npairs * want_c * 2 <= sms) want_c *= 2;
  }
  int Cc = 1;
  while (Cc * 2 <= std::min(want_c, kTileMaxCluster)) Cc *= 2;
  Cc = std::min(Cc, nA);
  while (Cc & (Cc - 1)) --Cc;
  const int budget = 227 * 1024 - (int)sizeof(TileShared) - 256;
  const int int_ties = (!S.do_penalize && (double)n * kOccupied < 0.9e6) ? 1 : 0;
  const int probs_bytes = (P * (int_ties ? 4 : 8) + 15) & ~15;   // per-cell maximum image: integer sums or FP64 responses
  int force_v = h->tile_chunks > 0 ? h->tile_chunks : env_int("B200_SWEEP_CHUNKS", 0);
  int bestV = 0, bestNb = 0, bestB = 0, bestStage = 0;
  long bestCost = -1;
  for (int V = Cc; V <= nA; ++V) {
    if (force_v > 0 && V < std::min(force_v, nA)) continue;   // "sweep_chunks" = at least this many chunks
    const int nAc = (nA + V - 1) / V;
    if ((nA + nAc - 1) / nAc != V || nAc > 63) continue;   // same chunk size as a smaller V; group ids are bytes
    const int a_bytes = (nAc * P * 4 + 15) & ~15;
    // staging buffer: header + about the descriptor bytes of a (chunk, phase, band) block (8 B per entry, n / 4 beams per phase
    // and band less the beams merged into weights, plus the residue padding); a longer block is split at a step boundary.  The
    // size depends on the number of bands and the bands on what the buffers leave: one refinement with the first pass's bands.
    int stage = 0, B = 0, nbv = 1;
    bool fits = true;
    for (int pass = 0; pass < 2 && fits; ++pass) {
      stage = 16 + nAc * 13 + (nAc * n * 3) / (2 * nbv) + 64 * nAc;
      stage = std::max(stage, 16 + 13 + 64 * 16);
      stage = (stage + 127) & ~127;
      const int s_avail = budget - a_bytes - probs_bytes - 2 * stage;
      B = s_avail / (pitch_w * 4) - halo;
      if (s_avail <= 0 || B < 8) { fits = false; break; }
      B = std::min(B, base_rows);
      nbv = (base_rows + B - 1) / B;
      B = (base_rows + nbv - 1) / nbv;                   // even bands
    }
    if (!fits) continue;
    // cost of one pair on one CTA, in thread-instructions: rasters (4 phases per chunk and band) + the beam loop per angle
    // the accumulator flush of every (angle, stage, slot group, word range) item (~100 warp instructions each, 32 warps) and the fixed
    // cost of a stage (clear + raster + three barriers, ~3 us) are what make extra bands expensive (measured: V 1 x 3 bands at
    // 4 m / 12 m runs 13 % slower than V 2 x 1 band).  0.4 per lookup: fitted to the tensor-core loop's kernel times at V = 2 ... 11
    // chunks, 4 m / 12 m (profiles/r3_tile_sweep.jsonl; the byte-unpack loop it replaced took 0.8)
    const long w_angle = (long)((double)P * n * 0.4 / kTileThreads) + 4L * nbv * ((long)ygroups * wranges * 100 / 32);
    const long w_raster = 4 * (700 + 3L * std::min(B + halo, rows_valid + halo - nY) * pitch_w / kTileThreads);
    const long cost = (long)((V + Cc - 1) / Cc) * (nbv * w_raster + nAc * w_angle);
    if (bestCost < 0 || cost < bestCost) { bestCost = cost; bestV = V; bestNb = nbv; bestB = B; bestStage = stage; }
  }
  if (bestCost < 0) return bail(4);
  const int V = bestV, nbands = bestNb, B = bestB, nAc = (nA + V - 1) / V, stage_bytes = bestStage;
  const int C = std::min(Cc, V);
  int alloc_rows = std::min(B + halo, rows_valid + halo - nY);
  alloc_rows = std::max(alloc_rows, 1);
  const size_t s_bytes = ((size_t)alloc_rows * pitch_w * 4 + 15) & ~(size_t)15;
  const size_t a_bytes = ((size_t)nAc * P * 4 + 15) & ~(size_t)15;
  T.C = C; T.V = V; T.nAc = nAc; T.nbands = nbands; T.band_rows = B; T.alloc_rows = alloc_rows; T.pitch_w = pitch_w;
  T.xtiles = xtiles; T.ytiles = ytiles; T.ygroups = ygroups; T.wranges = wranges; T.stage_bytes = stage_bytes;
  T.int_ties = int_ties;
  {
    // distinct non-zero smear values, ascending; up to 4 -> levelled (atomic-free) raster
    std::vector<uint8_t> lv(g.kernel.begin(), g.kernel.end());
    std::sort(lv.begin(), lv.end());
    lv.erase(std::unique(lv.begin(), lv.end()), lv.end());
    if (!lv.empty() && lv[0] == 0) lv.erase(lv.begin());
    T.nlevels = (!lv.empty() && lv.size() <= 4) ? (int)lv.size() : 0;
    for (int i = 0; i < 4; ++i) T.level[i] = i < T.nlevels ? lv[i] : 0;
  }
  T.off_A = s_bytes; T.off_probs = s_bytes + a_bytes; T.off_stage = (T.off_probs + probs_bytes + 127) & ~(size_t)127;
  T.off_cells = T.off_stage + 2 * (size_t)stage_bytes;
  // cell-list staging only where the chosen plan leaves room for it (it must not cost a band or a chunk: measured -17 % at 4 m / 20 m)
  int cell_cap = d_max_n_ok(S.max_n) ? S.max_n : 0;                     // entries per cell staging buffer (0 = read cells from global)
  if (T.off_cells + 2 * (size_t)cell_cap * 4 + sizeof(TileShared) + 64 > 227 * 1024) cell_cap = 0;
  T.cell_cap = cell_cap;
  size_t smem = T.off_cells + 2 * (size_t)cell_cap * 4;
  // reads past the last allocated row: idle lanes of the last y-tile read up to (48 ytiles - nY) rows past the band (EDGE), the
  // last slot group up to (16 ygroups - nY) rows plus the words of a word range (FAST): keep them inside the allocation even when
  // everything behind S is small (tiny search windows)
  const size_t overrun = std::max((size_t)(kYTile * ytiles - nY + 1) * pitch_w * 4,
                                  ((size_t)(16 * ygroups - nY + 1) * pitch_w + (size_t)kTileSlots * wranges) * 4);
  if (smem - s_bytes < overrun) smem = s_bytes + overrun;
  if (smem + sizeof(TileShared) + 64 > 227 * 1024) return bail(5);

  // ---- per-query descriptor blocks and schedules ----
  const int nstage = 4 * nbands;
  std::vector<uint8_t> blob;
  std::vector<TileSeq> seq;
  std::vector<int32_t> seq_start((size_t)nq * C + 1, 0);
  std::vector<int32_t> edge, edge_start((size_t)nq * nA * nstage * 4 + 1, 0);
  std::vector<int32_t> wrap2, wrap2_start((size_t)nq * nA * nstage + 1, 0);
  std::vector<int32_t> slow, slow_start((size_t)nq * (nA + 1), 0);
  int n_fast = 0, n_edge = 0;
  std::vector<std::vector<uint32_t>> grp((size_t)nA * nstage);   // FAST beams: band word offset << 2 | alignment
  std::vector<std::vector<int32_t>> egrp((size_t)nA * nstage * 4), wgrp((size_t)nA * nstage);
  blob.reserve((size_t)nq * nA * n * 2 + 4096);
  // one FAST stream per (angle, stage): 8-beam steps of 64 bytes, lane quad t4 reads {byte offset of beam t4, of beam t4 + 4,
  // V of beam t4, of beam t4 + 4} with V = weight << 8 * alignment
  struct Encoded { int steps; std::vector<uint32_t> pay; };
  std::vector<Encoded> enc((size_t)nA * nstage);
  std::vector<std::vector<int32_t>> slow_a(nA);
  std::vector<int> nfast_a(nA), nedge_a(nA);
  for (int q = 0; q < nq; ++q) {
    const CorrPlan & pl = S.plans[q];
    const int X0 = pl.xs[0], Y0 = pl.ys[0];
    // one host-pool task per angle: classify its beams, then sort / run-length encode its groups stage by stage
    auto one_angle = [&](int a) {
      for (int k = 0; k < nstage * 4; ++k) egrp[(size_t)a * nstage * 4 + k].clear();
      for (int k = 0; k < nstage; ++k) { grp[(size_t)a * nstage + k].clear(); wgrp[(size_t)a * nstage + k].clear(); }
      slow_a[a].clear();
      int nf = 0, ne = 0;
      for (int i = 0; i < n; ++i) {
        const int32_t off = pl.offsets[(size_t)a * n + i];
        if (off == kInvalidScan) continue;
        const int gx = pl.ogx[(size_t)a * n + i], gy = pl.ogy[(size_t)a * n + i];
        const int Xb = X0 + gx, Yb = Y0 + gy;
        const bool inside = Xb >= 0 && Xb + 2 * (nX - 1) < g.stride && Yb >= 0 && Yb + 2 * (nY - 1) < g.height;
        if (inside) {
          const int pp = Xb & 1, pq = Yb & 1, c = Xb >> 1, r = Yb >> 1;
          const int band = std::min(r / B, nbands - 1);
          const int wo = (r - band * B) * pitch_w + (c >> 2);
          grp[(size_t)a * nstage + (pq * 2 + pp) * nbands + band].push_back(((uint32_t)wo << 2) | (uint32_t)(c & 3));
          ++nf;
        } else if (Xb >= -g.stride && Xb + 2 * (nX - 1) < 2 * g.stride && Xb > -32768 && Xb < 32767 && Yb > -32768 && Yb < 32767) {
          // EDGE beam: at most one row wrap.  Primary entry in the beam's own phase; if some column leaves [0, stride), a
          // secondary entry in the phase with the row parity flipped.
          const bool rows_hit = Yb + 2 * (nY - 1) >= 0 && Yb < g.height;
          const bool cols_hit = Xb + 2 * (nX - 1) >= 0 && Xb < g.stride;
          if (rows_hit && cols_hit) {
            const int c = Xb >> 1, r = Yb >> 1;   // arithmetic shifts: floor for negative coordinates
            const int band = std::min(std::max(floor_div(r, B), 0), nbands - 1);
            const int rr = r - band * B;
            if (rr > -32768 && rr < 32767) {
              egrp[((size_t)a * nstage + ((Yb & 1) * 2 + (Xb & 1)) * nbands + band) * 4 + (c & 3)].push_back(
                (int32_t)((uint32_t)(rr & 0xFFFF) | ((uint32_t)(c >> 2) << 16)));
              ++ne;
            }
          }
          const bool wraps = Xb < 0 || Xb + 2 * (nX - 1) >= g.stride;
          if (wraps && Yb + 2 * (nY - 1) + 1 >= 0 && Yb - 1 < g.height) {
            const int r = (Yb - 1) >> 1;
            const int band = std::min(std::max(floor_div(r, B), 0), nbands - 1);
            wgrp[(size_t)a * nstage + (((Yb & 1) ^ 1) * 2 + (Xb & 1)) * nbands + band].push_back(
              (int32_t)((uint32_t)(Xb & 0xFFFF) | ((uint32_t)Yb << 16)));
          }
        } else {
          const int32_t dv = device_offset(off, g.data_size);
          if (dv != kDevInvalid) slow_a[a].push_back(dv);   // FAR: can still index [0, data_size) for some pose
        }
      }
      nfast_a[a] = nf; nedge_a[a] = ne;
      // the angle's stream of every stage.  Beams that land in the same cell become one entry whose weight is their count (entries
      // of at most 255: B holds bytes).  Entries are bucketed by word offset mod 4 and a k-quad takes one entry of each residue
      // (zero-weight entries at word `residue` of row 0 fill the shorter buckets); the stream is padded to whole 8-beam steps.
      for (int sg = 0; sg < nstage; ++sg) {
        std::vector<uint32_t> & gk = grp[(size_t)a * nstage + sg];
        std::sort(gk.begin(), gk.end());
        std::vector<uint32_t> bk[4][2];   // per residue: byte offsets, V words
        for (size_t i = 0; i < gk.size();) {
          size_t j = i;
          while (j < gk.size() && gk[j] == gk[i]) ++j;
          const uint32_t wo = gk[i] >> 2, m = gk[i] & 3;
          for (size_t t = i; t < j;) {
            const uint32_t w = h->no_dedup ? 1u : (uint32_t)std::min<size_t>(j - t, 255);
            bk[wo & 3][0].push_back(4u * wo);
            bk[wo & 3][1].push_back(w << (8 * m));
            t += w;
          }
          i = j;
        }
        size_t quads = 0;
        for (int r = 0; r < 4; ++r) quads = std::max(quads, bk[r][0].size());
        quads = (quads + 1) & ~(size_t)1;
        Encoded & E = enc[(size_t)a * nstage + sg];
        E.steps = (int)(quads / 2);
        E.pay.assign(quads * 8, 0u);
        for (size_t qd = 0; qd < quads; ++qd)
          for (int r = 0; r < 4; ++r) {
            const bool real = qd < bk[r][0].size();
            uint32_t * d = E.pay.data() + (qd / 2) * 16 + r * 4 + (qd & 1);
            d[0] = real ? bk[r][0][qd] : 4u * (uint32_t)r;
            d[2] = real ? bk[r][1][qd] : 0u;
          }
      }
    };
    host_parallel_for(nA, one_angle);
    for (int a = 0; a < nA; ++a) {
      slow_start[(size_t)q * (nA + 1) + a] = (int32_t)slow.size();
      slow.insert(slow.end(), slow_a[a].begin(), slow_a[a].end());
      n_fast += nfast_a[a]; n_edge += nedge_a[a];
    }
    slow_start[(size_t)q * (nA + 1) + nA] = (int32_t)slow.size();
    for (int a = 0; a < nA; ++a)
      for (int sg = 0; sg < nstage; ++sg) {
        wrap2_start[((size_t)q * nA + a) * nstage + sg] = (int32_t)wrap2.size();
        const auto & w = wgrp[(size_t)a * nstage + sg];
        wrap2.insert(wrap2.end(), w.begin(), w.end());
        for (int m = 0; m < 4; ++m) {
          edge_start[(((size_t)q * nA + a) * nstage + sg) * 4 + m] = (int32_t)edge.size();
          const auto & ev = egrp[((size_t)a * nstage + sg) * 4 + m];
          edge.insert(edge.end(), ev.begin(), ev.end());
        }
      }
    struct Seg { int a, k0, k1; };
    std::vector<Seg> segs;
    for (int r = 0; r < C; ++r) {
      seq_start[(size_t)q * C + r] = (int32_t)seq.size();
      for (int v = r; v < V; v += C) {
        const int ca0 = v * nAc, cna = std::min(nAc, nA - ca0);
        for (int sg = 0; sg < nstage; ++sg) {
          // sub-blocks: as many steps as fit one staging buffer; an angle's stream may continue in the next sub-block (the
          // accumulators are sums, the EDGE beams go with the angle's first part)
          int a = ca0, k = 0;
          bool first_sub = true;
          do {
            segs.clear();
            long used = 0;
            while (a < ca0 + cna) {
              const Encoded & E = enc[(size_t)a * nstage + sg];
              const long room = ((long)stage_bytes - (long)((((segs.size() + 1) * 13) + 15) & ~(size_t)15)) / 64 - used;
              if (room < 0 || (room == 0 && E.steps > k)) break;
              const int take = (int)std::min<long>(E.steps - k, room);
              segs.push_back({a, k, k + take});
              used += take;
              k += take;
              if (k < E.steps) break;
              ++a; k = 0;
            }
            if (segs.empty()) return bail(8);   // the staging buffer holds no step
            const int na = (int)segs.size();
            const size_t hdr = (((size_t)na * 13) + 15) & ~(size_t)15;
            const size_t bytes = hdr + (size_t)used * 64;
            TileSeq e{};
            e.off = (int32_t)blob.size();
            e.bytes = (int32_t)bytes;
            e.chunk = (int16_t)v; e.stage = (int16_t)sg; e.a0 = (int16_t)segs[0].a; e.na = (int16_t)na;
            e.flags = (first_sub ? kSeqNewStage : 0u) | ((first_sub && sg == 0) ? kSeqNewChunk : 0u);
            for (const Seg & sgm : segs)
              for (int m = 0; m < 4; ++m)
                if (sgm.k0 == 0 && !egrp[((size_t)sgm.a * nstage + sg) * 4 + m].empty()) e.flags |= kSeqHasEdge;
            if (first_sub)
              for (int aa = ca0; aa < ca0 + cna; ++aa)
                if (!wgrp[(size_t)aa * nstage + sg].empty()) e.flags |= kSeqHasWrap;
            blob.resize(blob.size() + bytes, 0);
            int32_t * tbl = reinterpret_cast<int32_t *>(blob.data() + e.off);
            uint8_t * order = blob.data() + e.off + (size_t)na * 12;
            uint32_t * steps = reinterpret_cast<uint32_t *>(blob.data() + e.off + hdr);
            std::vector<std::pair<int, int>> wt;   // angles by descending stream length: the shared queue hands out long items first
            int at = 0;
            for (int i = 0; i < na; ++i) {
              const Seg & sgm = segs[i];
              const int len = sgm.k1 - sgm.k0;
              tbl[3 * i + 0] = at; tbl[3 * i + 1] = at + len; tbl[3 * i + 2] = sgm.k0 == 0;
              if (len) std::memcpy(steps + (size_t)at * 16, enc[(size_t)sgm.a * nstage + sg].pay.data() + (size_t)sgm.k0 * 16, (size_t)len * 64);
              at += len;
              wt.emplace_back(-len, i);
            }
            std::sort(wt.begin(), wt.end());
            for (int i = 0; i < na; ++i) order[i] = (uint8_t)wt[i].second;
            seq.push_back(e);
            first_sub = false;
          } while (a < ca0 + cna);
        }
        seq.back().flags |= kSeqEndChunk;
      }
    }
  }
  seq_start[(size_t)nq * C] = (int32_t)seq.size();
  edge_start[(size_t)nq * nA * nstage * 4] = (int32_t)edge.size();
  wrap2_start[(size_t)nq * nA * nstage] = (int32_t)wrap2.size();
  edge.push_back(0); wrap2.push_back(0); slow.push_back(0);
  blob.resize(blob.size() + 16, 0);

  auto up = [&](auto & dst, const auto & src) {
    using TT = typename std::remove_reference<decltype(src)>::type::value_type;
    dst.reserve(src.size());
    sweep_stage_h2d(dst.p, src.data(), src.size() * sizeof(TT), st);   // pinned arena: no blocking, the vectors may go away
  };
  up(S.d_tile_desc, blob);
  up(S.d_tile_seq, seq);
  up(S.d_tile_seq_start, seq_start);
  up(S.d_tile_edge, edge);
  up(S.d_tile_edge_start, edge_start);
  up(S.d_tile_wrap2, wrap2);
  up(S.d_tile_wrap2_start, wrap2_start);
  up(S.d_tile_slow, slow);
  up(S.d_tile_slow_start, slow_start);
  T.desc = S.d_tile_desc.p; T.seq = S.d_tile_seq.p; T.seq_start = S.d_tile_seq_start.p;
  T.edge = S.d_tile_edge.p; T.edge_start = S.d_tile_edge_start.p;
  T.wrap2 = S.d_tile_wrap2.p; T.wrap2_start = S.d_tile_wrap2_start.p;
  T.slow = S.d_tile_slow.p; T.slow_start = S.d_tile_slow_start.p;
  T.enabled = 1;
  S.tile_smem = smem;

  // ---- grid: as many co-resident clusters as the device holds, one pair per cluster at a time ----
  const void * kfn = tile_kernel_for(pitch_w);
  B200_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int max_clusters = sms / C;
  {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)(C * std::max(1, sms / C)));
    cfg.blockDim = dim3(kTileThreads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int nc = 0;
    if (cudaOccupancyMaxActiveClusters(&nc, kfn, &cfg) == cudaSuccess && nc > 0) max_clusters = nc;
    else (void)cudaGetLastError();
  }
  const int clusters = std::max(1, std::min(S.npairs, max_clusters));
  S.tile_grid = clusters * C;
  S.tile_info[0] = 1; S.tile_info[1] = C; S.tile_info[2] = V; S.tile_info[3] = nbands; S.tile_info[4] = B; S.tile_info[5] = 0;
  S.tile_info[6] = clusters; S.tile_info[7] = (int32_t)(smem / 1024);
  S.fast_info[1] = n_fast; S.fast_info[2] = n_edge; S.fast_info[3] = (int32_t)slow.size() - 1;
  return true;
}

void launch_sweep_tile(b200sm * h, SweepHost & S, cudaStream_t st)
{
  (void)h;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)S.tile_grid);
  cfg.blockDim = dim3(kTileThreads);
  cfg.dynamicSmemBytes = S.tile_smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = (unsigned)S.tile.C; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  const void * kfn = tile_kernel_for(S.tile.pitch_w);
  B200_CUDA(cudaFuncSetAttribute(kfn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S.tile_smem));
  void * args[] = {(void *)&S.dev, (void *)&S.tile};
  B200_CUDA(cudaLaunchKernelExC(&cfg, kfn, args));
}

}  // namespace b200
