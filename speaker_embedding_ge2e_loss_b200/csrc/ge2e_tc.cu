// tcgen05 / TMA / TMEM path of the GE2E loss (TF32 operands, fp32 accumulators in tensor memory).
//
// One warp-specialised persistent kernel, two instantiations: the forward rows alone (contrast loss,
// forward-only calls) and the whole softmax step -- forward rows fused with the dE_hat contraction,
// then the dC_hat contraction (the tensor-core twin of ge2e_simt.cu's strip kernel).  An "owner" operand
// tile X[128, D] stays resident in shared memory, a "stream" operand Y is pulled through a TMA
// ring one work unit (128 rows) at a time:
//
//   MMA1   T[128 x n] = X . Y_unit^T            (SS, both K-major, K = D)            -> TMEM
//   FWD    epilogue: online log-sum-exp (softmax) / running arg-max (contrast) over T's columns;
//          S = w (cos + eps) + b is never written anywhere (reference s3:64-79, s3:27, s3:114-127)
//          n = 256 (two units per step) whenever two units are left in the CTA's range
//   STEP   two passes over S (n = 128), S computed ONCE per pass and never stored:
//          pass 1 (DE segments: X = E_hat rows, Y = C_hat): epilogue P = exp2(S log2e - m) with the
//            leave-one-out diagonal masked, m = |w| + b a FIXED shift (|cos| <= 1 bounds every logit,
//            so partial sums from different clusters simply add); the row sums give the log-sum-exp
//            (the forward's row loss) and P, rounded to TF32, is written back over T in TMEM;
//            MMA2  Acc[128 x D] += P . Y_unit  (A from TMEM, B MN-major from smem) -> un-normalised
//            dE_hat rows: the true row is g w exp(m - lse_r) times it (row_scale, applied by finalize)
//          -- per utterance tile: the segment that completes a tile's row sums closes its 128 rows --
//          pass 2 (DC segments: X = C_hat rows, Y = E_hat; a stream unit is one utterance tile, and its epilogue
//            waits for that tile's rows only, not for the grid): epilogue G = w g softmax(S) with the own
//            speaker's rows masked, written back over T; MMA2 Acc += G . Y_unit -> dC_hat = (wG)^T E_hat
//          the accumulator leaves through shared memory and a TMA store / TMA reduce-add.
//          Issued contraction work: 8 U N D (algorithmic 6: S is recomputed once, for pass 2).
//
// CG = 2 runs every MMA on a CTA pair (tcgen05 cta_group::2, UMMA M = 256): the two CTAs of a
// cluster own two consecutive owner tiles and each fetches HALF of every stream operand, which
// halves the L2 -> SM traffic and the shared-memory read rate per MMA (the limits of CG = 1: the
// probe in tests/probe/pipe_probe.cu measures 80 clk for a 128x128x8 TF32 MMA against 65 for
// the paired 256x128x8).  The leader CTA (cluster rank 0) issues the MMAs; every barrier the MMA
// warp waits on lives in the leader and is signalled by both CTAs.
//
// Work = (owner group, stream unit) pairs; a segment is a run of pairs inside one owner group.
//   FWD   the flat pair list is cut into equal contiguous ranges over the clusters (stream-K); a
//         cluster whose range covers only part of an owner group publishes (max, sum) per row and
//         the last cluster to finish that tile merges.
//   STEP  both passes in ONE launch: whole owner groups where that balances (plain store), else cut
//         groups whose partial accumulators are added into the zero-filled output at the L2
//         (cp.reduce.async.bulk).  The per-cluster ranges are computed on the host (make_step_sched) and
//         passed by value: pass 2 is cut against a model of when each cluster leaves pass 1 and when each
//         utterance tile's row sums are complete, and a cluster walks its pass-2 range rotated so that
//         the tiles completed last come last.  The TMA and MMA warps run straight from pass 1 into
//         pass 2 (their operands are inputs); only the epilogue waits, per stream unit.
//
// Warp roles (384 threads): warp 0 = TMA producer, warp 1 = MMA issuer, warp 2 = TMEM allocator,
// warps 4-11 = epilogue (TMEM lane quarter = warp % 4, column half = (warp - 4) / 4: two threads
// share a tile row).  Producer and MMA warps run their loops with all 32 lanes and issue through
// elect.sync: what looks like a detail is a 2.5x difference in MMA issue rate (see the probe).
#include <cuda.h>
#include <cuda_fp16.h>
#include <cudaTypedefs.h>
#include <limits.h>
#include <stdlib.h>

#include <algorithm>
#include <cstring>
#include <type_traits>
#include <vector>

#include "ge2e_common.cuh"
#include "ge2e_tc_ptx.cuh"

namespace ge2e {

namespace {

using namespace ptx;

constexpr int kTile = 128;            // owner rows per CTA (= UMMA M per CTA = TMEM lanes)
constexpr int kUnit = 128;            // stream rows per work unit
constexpr int kSlabCols = 32;         // fp32 columns per 128-byte swizzled row
constexpr int kSlabBytes = kTile * 128;       // one owner [128 x 32] K-major slab = 16 KB
constexpr int kMaxSlabs = 8;          // D <= 256
constexpr int kRingBytes = 96 * 1024;
constexpr int kBoxRows = 64;          // rows of one K-major stream TMA box
constexpr int kMma2Rows = 32;         // stream rows (K of MMA2) per ring stage
constexpr int kMaxStages = 6;
constexpr int kEpiWarp0 = 4;
constexpr int kEpiWarps = 8;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kThreadsTc = (kEpiWarp0 + kEpiWarps) * 32;
constexpr int kMaxClusters = 160;     // >= SM count / cluster size
constexpr int kMaxPeers = GE2E_MAX_PEERS;   // ranks of one NVSwitch domain (fused reduce-scatter)
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

enum { TC_FWD = 0, TC_STEP = 1 };
// operand precision: TF32 (one rounded fp32 plane) or SPLIT (fp32-class: every operand as two fp16 planes
// hi = fp16(x), lo = fp16(x - hi); a product is the three kind::f16 MMAs hi.hi + hi.lo + lo.hi)
// F16: ONE fp16 plane (hi only): 11-bit mantissas as TF32, twice its MMA rate -- the TF32-tolerance class for the
// shapes where the MMAs dominate (same kernels and row-closing order as SPLIT, one MMA per product)
// HYB: the TF32 flow (fixed shift, one launch, P and MMA2 in TF32) with MMA1 alone on fp16 COPIES of the operands
// (11-bit mantissas as TF32): MMA1 at n = 128 is bound by its shared-memory operand reads, an fp16 instruction reads
// the same bytes for twice the K -- half the instructions.  The copies are made by a conversion kernel in front
// of the step kernel and live in the workspace; chosen by tc_step for large shapes under GE2E_TF32.
enum { PREC_TF32 = 0, PREC_SPLIT = 1, PREC_F16 = 2, PREC_HYB = 3 };
// The probability planes carry p * 2^(14 + k): 2^14 keeps p <= 1 inside fp16, and k >= 0 lifts what is known to
// be small -- pass 1: k_r from q_r = 1 - p_jj >= every off-diagonal probability of utterance row r (per owner
// row, undone by row_scale); pass 2: k from the largest q of the whole batch (undone in the accumulator flush).
// Without the lift a confident batch (all off-diagonal p ~ 1e-8) would sit in the fp16 subnormals.
constexpr int kSplitLift = 14;
constexpr int kSplitMaxExtra = 96;
__device__ __forceinline__ int split_extra_lift(float q) {      // largest k in [0, 96] with q * 2^k <= 1
  if (!(q > 0.f)) return kSplitMaxExtra;
  return max(0, min(kSplitMaxExtra, -ilogbf(q) - 1));
}
enum { PASS_ROWS = 1, PASS_CENTROIDS = 2 };   // TcParams::phases
enum { SEG_DE = 0, SEG_DC = 1 };      // index into the per-segment-kind arrays (FWD uses index 0)

// barrier indices inside the shared barrier array
enum {
  BAR_FULL = 0,                         // [stages] TMA -> MMA                         (leader)
  BAR_EMPTY = BAR_FULL + kMaxStages,    // [stages] MMA -> TMA                         (every CTA)
  BAR_A_FULL = BAR_EMPTY + kMaxStages,  // [slabs]  owner slab landed                  (leader)
  BAR_A_EMPTY = BAR_A_FULL + kMaxSlabs, // owner tile no longer read by MMA1           (every CTA)
  BAR_S_FULL,                           // [2] MMA1 result in TMEM                     (every CTA)
  BAR_S_EMPTY = BAR_S_FULL + 2,         // [2] FWD: epilogue drained T                 (leader)
  BAR_G_FULL = BAR_S_EMPTY + 2,         // [2] BWD: G written back to TMEM             (leader)
  BAR_ACC_FULL = BAR_G_FULL + 2,        // BWD: accumulator complete for this segment  (every CTA)
  BAR_ACC_EMPTY,                        // BWD: accumulator drained                    (leader)
  BAR_A_FREE,                           // [slabs] STEP: the flush's TMA store has read owner slab k (own CTA)
  BAR_COUNT = BAR_A_FREE + kMaxSlabs
};

// tensor maps of one launch; index = segment kind (FWD: [SEG_DE] only)
struct TmSet {
  CUtensorMap own[2];    // owner tiles        box [128 rows][32 cols], 128B swizzle
  CUtensorMap strk[2];   // stream, K-major    box [64 rows][32 cols], 128B swizzle
  CUtensorMap strmn[2];  // stream, MN-major   box [D/32/CG][32 rows][32 cols], 32B-atom 128B swizzle
  CUtensorMap out[2];    // accumulator output box [128 rows][32 cols], 128B swizzle
  // STEP, speaker-sharded over peer memory: dC_hat rows [r * peer_rows, (r + 1) * peer_rows) live in rank r's
  // dC_local (mapped into this process, NVLink): pass 2 reduce-adds its accumulators THERE instead of into a
  // full-height local partial that a reduce-scatter would have to sum afterwards
  CUtensorMap out_peer[kMaxPeers];
};

// STEP: pair range [begin[c], begin[c + 1]) of cluster c in the dE_hat (pass 1) / dC_hat (pass 2) pair lists;
// cluster c walks its pass-2 range (one owner group whenever dc_rot[c] != 0) starting dc_rot[c] units in and
// wrapping around, so that the utterance tiles whose row sums are completed last are visited last
struct StepSched {
  int de[kMaxClusters + 1];
  int dc[kMaxClusters + 1];
  unsigned char dc_rot[kMaxClusters];
};

struct TcParams {
  int D, kslabs;              // kslabs = D / 32: 32-column fp32 slabs of an accumulator tile (and of a TF32 operand tile)
  int oslabs;                 // 128-byte slabs of an OPERAND tile: D / 32 (TF32), 2 D / 64 (SPLIT), D / 64 (F16)
  int M, spk_offset;
  int n_own[2], n_str[2];     // rows of the owner / stream matrix per segment kind
  int OT[2], ST[2];           // owner tiles, stream units
  long long GP;               // FWD: owner groups * ST (group, stream unit) pairs
  const float* cos_diag;      // [U_local]
  const float* row_stat;      // STEP, pass 2 alone: lse per local utterance row (written by an earlier launch)
  const float* row_aux;       // STEP, pass 2 alone: q = 1 - p_jj per local utterance row
  float* row_aux_out;         // FWD softmax / STEP pass 1
  int phases;                 // STEP: PASS_ROWS | PASS_CENTROIDS
  float* rowsum;              // STEP: [U_local] off-diagonal sums of P (workspace; zero-filled by the kernel)
  float* row_scale_out;       // STEP pass 1: w exp(m - lse_r), the factor of the un-normalised dE_hat rows
  const float* w;
  const float* b;
  const float* grad_out;
  const float* grad_rows;     // STEP pass 2 alone, RG instantiations: upstream gradient per local utterance row
  float eps;
  // FWD outputs
  float* row_stat_out;
  int32_t* kstar_out;
  float* loss_accum;
  float* per_row_out;
  int* seg_done;              // [OT] stream units finished per owner tile; STEP: per utterance tile, pass 1 (zero on entry and exit)
  float2* seg_part;           // [OT][maxseg][128] partial row state
  int maxseg;
  // BWD outputs (dE_hat / dC_hat go through the `out` tensor maps)
  float* dwdb;
  float4* zero_base;          // STEP: dC_hat, zero-filled by the kernel itself before any partial sum lands
  long long zero_n4;          //      (float4 count; 0 = nothing to clear)
  float4* zero2_base;         // STEP: dE_hat when some owner group is cut between clusters
  long long zero2_n4;
  int* ctr;                   // STEP: {CTAs done zero-filling, CTAs done, utterance tiles complete}: zero on entry and exit
  int peer_rows;              // STEP: > 0: centroid rows per rank, pass 2 flushes through tms.out_peer (see TmSet)
  unsigned long long* stamps; // STEP, nullable: [CTA]{start, end} globaltimer stamps (in-situ kernel time)
  unsigned long long* trace;  // debug: [CTA][3 roles][kTraceEvents] globaltimer stamps, or nullptr
  int dbg;                    // debug instantiation only: 8 = per-stage marks in the MMA warp's trace
};

constexpr int kTraceEvents = 64;
// DBG = false compiles every hook away: the MMA issue loop is instruction-bound (a ring stage must be
// issued in less than the ~520 clk its MMAs run), stray branches there cost real throughput.
template <bool DBG>
struct Tracer {
  unsigned long long* buf;
  int n, cap;
  // reserve: slots at the end of the record kept for put()
  __device__ __forceinline__ Tracer(unsigned long long* base, int role, int reserve = 0)
      : buf(DBG && base ? base + (static_cast<size_t>(blockIdx.x) * 3 + role) * kTraceEvents : nullptr), n(0),
        cap(kTraceEvents - reserve) {}
  __device__ __forceinline__ void mark() {
    if (DBG) {
      if (buf != nullptr && n < cap) buf[n++] = globaltimer_ns();
    }
  }
  // the step kernel's epilogue record reserves its last three slots: [61] pass 1 done (row sums counted),
  // [62] first pass-2 segment begins, [63] total ns spent waiting for pass-2 row sums
  __device__ __forceinline__ void put(int slot, unsigned long long v) {
    if (DBG) {
      if (buf != nullptr) buf[slot] = v;
    }
  }
};

struct SharedTail {
  uint64_t bars[BAR_COUNT];
  uint32_t tmem_base;
  int flag;
  int rows_all_done;                      // STEP: this CTA has seen ctr[2] == OT (every utterance tile complete)
  union {
    float red[2 * kEpiWarps];
    float red3[3 * kEpiWarps];
  };
  union {                                 // 1 KB either way: the budget above the ring is ~2 KB
    alignas(16) float lse_s[2][kUnit];    // DC segments: lse (log2 domain) of the current stream rows
    alignas(16) float2 xch[kTile];        // FWD: row state of the upper column half
  };
};
// RG instantiations (per-row upstream gradient): lse_s[buf][r] then holds lse2 - log2 |g_r| (/ gamma on the planes) and
// gsign[buf] the signs of g_r, one bit per stream row, staged by the same threads at the same points
struct SharedTailRG : SharedTail {
  uint32_t gsign[2][kUnit / 32];
};
constexpr size_t kWsHeaderBytes = 256;   // workspace: [header: BWD counters][FWD seg_done][FWD seg_part]
template <bool RG = false>
constexpr size_t kSmemBytesT = 1024 + kMaxSlabs * kSlabBytes + kRingBytes + (RG ? sizeof(SharedTailRG) : sizeof(SharedTail));
constexpr size_t kSmemBytes = kSmemBytesT<false>;
static_assert(kSmemBytesT<true> <= 232448, "dynamic shared memory over the 227 KB per-CTA limit");

__device__ __forceinline__ int cluster_of_pair(long long gp, long long GP, int NC) {
  // largest c with floor(c * GP / NC) <= gp
  return static_cast<int>(((gp + 1) * NC + GP - 1) / GP) - 1;
}

// The walk over a cluster's segments, identical in every warp role.
struct Walk {
  long long gp, end;      // remaining pair range of the current part
  long long gp2, end2;    // BWD: the other part, visited second
  int kind, kind2;        // kind of the current / of the second part (kind2 < 0: no second part left)
  int rot;                // STEP: first unit of a pass-2 segment, relative to s0 (StepSched::dc_rot)
  // unit visited i-th in the segment [s0, s1) returned by next()
  __device__ __forceinline__ int unit(int i, int s0, int s1) const {
    const int u = s0 + i + (kind == SEG_DC ? rot : 0);
    return u < s1 ? u : u - (s1 - s0);
  }
  __device__ __forceinline__ bool next(const TcParams& p, int& kind_out, int& og, int& s0, int& s1) {
    while (gp >= end) {
      if (kind2 < 0) return false;
      kind = kind2; gp = gp2; end = end2; kind2 = -1;
    }
    const int st = p.ST[kind];
    kind_out = kind;
    og = static_cast<int>(gp / st);
    s0 = static_cast<int>(gp % st);
    s1 = static_cast<int>(min(static_cast<long long>(st), s0 + (end - gp)));
    gp += s1 - s0;
    return true;
  }
};

// close_softmax_row (ge2e_common.cuh, reference s3:119-121) from LOG2-domain state: m2 >= every S_k log2e (the
// running maximum, or the fixed shift), loff = sum_{k != j} exp2(S_k log2e - m2), xd2 = the diagonal logit formed
// by the SAME affine map (w log2e, b log2e) as the off-diagonal ones -- the constant roundings of that map then
// cancel in q = 1 - p_j, which a natural-domain diagonal term against a log2-domain sum would not (measured at
// w = 30: -5e-6 relative in q).  Sd = the natural-domain diagonal logit for the large-q row loss.
// lse2 = log-sum-exp in the log2 domain, z = sum_k exp2(S_k log2e - m2) + eps 2^-m2 (only where m2 > -115).
struct RowClose { float stat, q, per, lse2, z; };
__device__ __forceinline__ RowClose close_softmax_row_log2(float m2, float loff, float xd2, float Sd, float eps) {
  RowClose r;
  if (m2 > -115.f) {      // -80 log2e
    const float em = eps * exp2f(-m2);
    r.z = loff + exp2f(xd2 - m2) + em;
    r.lse2 = m2 + log2f(r.z);
    r.stat = r.lse2 * kLn2;
    r.q = (loff + em) / r.z;
  } else {                // every logit below -80: eps dominates
    const float s = exp2f(m2);
    const float Z = eps + (loff + exp2f(xd2 - m2)) * s;
    r.stat = logf(Z);
    r.lse2 = r.stat * kLog2e;
    r.q = (eps + loff * s) / Z;
    r.z = Z / s;
  }
  r.per = (r.q < 0.5f) ? -log1pf(-r.q) : r.stat - Sd;
  return r;
}

// two fp32 values -> packed fp16 pair of their leading parts and of the remainders
__device__ __forceinline__ void split_pack(float p0, float p1, uint32_t& hi, uint32_t& lo) {
  const __half2 h = __floats2half2_rn(p0, p1);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(p0 - hf.x, p1 - hf.y);
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// RG (STEP, pass 2 alone): the upstream gradient is one value g_r per utterance row (p.grad_rows), not the scalar
// p.grad_out.  The tail above the ring has 608 bytes left, too few for a staged fp32 copy of g_r (1 KB double
// buffered), so |g_r| is folded into the staged log-sum-exp (exp2(S log2e - lse2 + log2 |g_r|) = p |g_r|, one more
// fp32 rounding of an exponent that already carries one) and its sign is staged as one bit per stream row (SharedTailRG).
// The fp16 planes carry p (g_r / gamma), gamma = max_r |g_r|, lifted by the largest q_r |g_r| / gamma; the flush
// applies w gamma.
template <int MODE, int VARIANT, int CG, int PREC, bool DBG, bool RG = false>
__global__ void __launch_bounds__(kThreadsTc, 1)
tc_strip_kernel(const __grid_constant__ TmSet tms, const __grid_constant__ StepSched sched, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  constexpr bool kBwd = (MODE != TC_FWD);
  constexpr bool kSplit = (PREC == PREC_SPLIT || PREC == PREC_F16);   // fp16 planes, rows closed by the forward kernel
  constexpr bool kHyb = (PREC == PREC_HYB);
  constexpr bool kOpF16 = kSplit || kHyb;           // MMA1 operands are fp16 (planes, or the workspace copies)
  constexpr int kPlanes = (PREC == PREC_SPLIT) ? 2 : 1;
  // stream rows (K of MMA2) per ring stage: a stage is 16 KB per CTA of a pair either way -- 32 rows of fp32 or of
  // two fp16 planes, 64 rows of ONE fp16 plane (with 32 the stages would be half empty and the ring would hold
  // barely one unit of look-ahead: the F16 kernel ran load-latency-bound)
  constexpr int kM2 = (PREC == PREC_F16) ? 64 : kMma2Rows;
  constexpr int kStageBytes = 32768 / CG;
  constexpr int kStages = 3 * CG;
  constexpr uint16_t kPairMask = (CG == 2) ? 3 : 1;
  constexpr uint32_t kEpiArrivals = kEpiWarps * CG;

  // carve: [owner slabs 8 x 16 KB][ring 96 KB][tail]; the dynamic window starts at the same
  // CTA-relative offset in both CTAs of a pair, so descriptors and multicast offsets line up
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_al = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t a_smem = smem_base;
  const uint32_t ring_smem = smem_base + kMaxSlabs * kSlabBytes;
  using Tail = std::conditional_t<RG, SharedTailRG, SharedTail>;
  Tail* tail = reinterpret_cast<Tail*>(smem_al + kMaxSlabs * kSlabBytes + kRingBytes);
  const uint32_t bars = smem_u32(&tail->bars[0]);
  auto bar = [&](int i) { return bars + 8u * i; };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NC = gridDim.x / CG, cl = blockIdx.x / CG;
  const int cr = (CG == 2) ? static_cast<int>(cluster_ctarank()) : 0;     // rank in the CTA pair
  const bool leader = (cr == 0);
  // barriers the MMA warp waits on live in the leader: address them through the cluster window
  auto lbar = [&](int i) { return (CG == 2) ? mapa(bar(i), 0) : bar(i); };
  const int kslabs = p.kslabs, oslabs = p.oslabs;
  // fp16 planes: slab s of an operand tile is [rows x 64 fp16] = chunk s % hs of plane s / hs (hi plane first)
  const int hs = p.D >> 6;
  const int dbg = DBG ? p.dbg : 0;      // compile-time 0 in the production instantiation

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tms.own[0]);
    prefetch_tmap(&tms.strk[0]);
    if (kBwd) {
      prefetch_tmap(&tms.own[1]); prefetch_tmap(&tms.strk[1]);
      prefetch_tmap(&tms.strmn[0]); prefetch_tmap(&tms.strmn[1]);
      prefetch_tmap(&tms.out[0]); prefetch_tmap(&tms.out[1]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(bar(BAR_FULL + i), 1); mbar_init(bar(BAR_EMPTY + i), 1); }
    for (int i = 0; i < kMaxSlabs; ++i) mbar_init(bar(BAR_A_FULL + i), 1);
    mbar_init(bar(BAR_A_EMPTY), 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar(BAR_S_FULL + i), 1);
      mbar_init(bar(BAR_S_EMPTY + i), kEpiArrivals);
      mbar_init(bar(BAR_G_FULL + i), kEpiArrivals);
    }
    mbar_init(bar(BAR_ACC_FULL), 1);
    mbar_init(bar(BAR_ACC_EMPTY), kEpiArrivals);
    for (int i = 0; i < kMaxSlabs; ++i) mbar_init(bar(BAR_A_FREE + i), 1);
    fence_mbar_init();
  }
  if (warp == 2) {
    if (CG == 1) tmem_alloc<512>(smem_u32(&tail->tmem_base));
    else tmem_alloc_2cta<512>(smem_u32(&tail->tmem_base));
  }
  tc_fence_before();
  __syncthreads();
  if (CG > 1) cluster_sync_all();     // the peer's barriers are initialised before any remote arrive
  tc_fence_after();
  const uint32_t tmem = tail->tmem_base;
  // Programmatic dependent launch: everything above overlapped the stream predecessor's tail.  Both
  // instantiations read what their predecessor (prep) wrote: wait, THEN let the successor go -- a
  // successor that starts early may therefore assume that everything before this kernel has completed.
  pdl_wait();
  pdl_trigger();
  if (kBwd && p.stamps != nullptr && tid == 0) p.stamps[2 * blockIdx.x] = globaltimer_ns();

  // ---- this cluster's work
  auto make_walk = [&]() {
    Walk wk;
    if (!kBwd) {
      wk.kind = SEG_DE; wk.kind2 = -1;
      wk.gp = (static_cast<long long>(cl) * p.GP) / NC;
      wk.end = (static_cast<long long>(cl + 1) * p.GP) / NC;
      wk.gp2 = wk.end2 = 0;
      wk.rot = 0;
    } else {
      // pass 1 (dE_hat segments), then pass 2 (dC_hat segments); a pass that is not in p.phases has empty ranges
      wk.kind = SEG_DE; wk.gp = sched.de[cl]; wk.end = sched.de[cl + 1];
      wk.kind2 = SEG_DC; wk.gp2 = sched.dc[cl]; wk.end2 = sched.dc[cl + 1];
      wk.rot = sched.dc_rot[cl];
    }
    return wk;
  };
  constexpr int kStepUnits = kBwd ? 1 : 2;

  if (warp == 0) {
    // ===================================================================== TMA producer
    Tracer<DBG> tr(lane == 0 ? p.trace : nullptr, 0);
    tr.mark();
    int stage = 0, phase = 0;
    auto advance = [&]() { if (++stage == kStages) { stage = 0; phase ^= 1; } };
    // one K-major stage: `nslab` slabs of [rows_cta x 32] starting at slab ks0, stream rows
    // [row0 + cr * rows_cta, + rows_cta) of a step that covers rows_cta * CG rows
    auto load_k = [&](const CUtensorMap* tm, int row0, int rows_cta, int ks0, int nslab) {
      mbar_wait(bar(BAR_EMPTY + stage), phase ^ 1);
      if (elect_one()) {
        const uint32_t bytes = static_cast<uint32_t>(nslab * rows_cta * 128);
        if (leader) mbar_expect_tx(bar(BAR_FULL + stage), bytes * CG);
        const uint32_t full = lbar(BAR_FULL + stage);
        uint32_t dst = ring_smem + stage * kStageBytes;
        for (int sl = 0; sl < nslab; ++sl)
          for (int r = 0; r < rows_cta; r += kBoxRows, dst += kBoxRows * 128) {
            const int s = ks0 + sl;
            if (kHyb) {
              if (CG == 1) tma_load_2d(dst, tm, s * 64, row0 + r, full);
              else tma_load_2d_2cta(dst, tm, s * 64, row0 + cr * rows_cta + r, full);
            } else if (kSplit) {
              if (CG == 1) tma_load_3d(dst, tm, (s % hs) * 64, row0 + r, s / hs, full);
              else tma_load_3d_2cta(dst, tm, (s % hs) * 64, row0 + cr * rows_cta + r, s / hs, full);
            } else {
              if (CG == 1) tma_load_2d(dst, tm, s * kSlabCols, row0 + r, full);
              else tma_load_2d_2cta(dst, tm, s * kSlabCols, row0 + cr * rows_cta + r, full);
            }
          }
      }
      __syncwarp();
      advance();
    };
    // one MN-major stage: kMma2Rows stream rows x this CTA's share of the D columns
    auto load_mn = [&](const CUtensorMap* tm, int row0) {
      mbar_wait(bar(BAR_EMPTY + stage), phase ^ 1);
      if (elect_one()) {
        const int slabs_c = (kSplit ? oslabs : kslabs) / CG;      // (HYB: the MN-major operand of MMA2 stays fp32)
        const uint32_t bytes = static_cast<uint32_t>(slabs_c * kM2 * 128);
        if (leader) mbar_expect_tx(bar(BAR_FULL + stage), bytes * CG);
        const uint32_t full = lbar(BAR_FULL + stage);
        const uint32_t dst = ring_smem + stage * kStageBytes;
        if (kSplit) {        // [plane][chunk][32 rows][64 fp16]: this CTA's chunks of both planes in one box
          if (CG == 1) tma_load_4d(dst, tm, 0, row0, 0, 0, full);
          else tma_load_4d_2cta(dst, tm, 0, row0, cr * (hs / CG), 0, full);
        } else {
          if (CG == 1) tma_load_3d(dst, tm, 0, row0, 0, full);
          else tma_load_3d_2cta(dst, tm, 0, row0, cr * slabs_c, full);
        }
      }
      __syncwarp();
      advance();
    };
    Walk wk = make_walk();
    int kind, og, s0, s1;
    for (int sg = 0; wk.next(p, kind, og, s0, s1); ++sg) {
      const CUtensorMap* tm_own = &tms.own[kind];
      const CUtensorMap* tm_k = &tms.strk[kind];
      const CUtensorMap* tm_mn = &tms.strmn[kind];
      const int ot = og * CG + cr;      // may be >= OT in the last group: TMA zero-fills, nothing is stored
      if (sg > 0) mbar_wait(bar(BAR_A_EMPTY), (sg - 1) & 1);      // every MMA1 of the previous segment has completed
      tr.mark();   // owner tile issue
      auto load_own = [&](int ks) {
        // STEP: the previous segment's accumulator leaves through the owner area, slab by slab; slab ks is
        // free again once the TMA store that took it out has read it
        if (kBwd && sg > 0) mbar_wait(bar(BAR_A_FREE + ks), (sg - 1) & 1);
        if (elect_one()) {
          if (leader) mbar_expect_tx(bar(BAR_A_FULL + ks), kSlabBytes * CG);
          const uint32_t dst = a_smem + ks * kSlabBytes;
          if (kHyb) {
            if (CG == 1) tma_load_2d(dst, tm_own, ks * 64, ot * kTile, bar(BAR_A_FULL + ks));
            else tma_load_2d_2cta(dst, tm_own, ks * 64, ot * kTile, lbar(BAR_A_FULL + ks));
          } else if (kSplit) {
            if (CG == 1) tma_load_3d(dst, tm_own, (ks % hs) * 64, ot * kTile, ks / hs, bar(BAR_A_FULL + ks));
            else tma_load_3d_2cta(dst, tm_own, (ks % hs) * 64, ot * kTile, ks / hs, lbar(BAR_A_FULL + ks));
          } else {
            if (CG == 1) tma_load_2d(dst, tm_own, ks * kSlabCols, ot * kTile, bar(BAR_A_FULL + ks));
            else tma_load_2d_2cta(dst, tm_own, ks * kSlabCols, ot * kTile, lbar(BAR_A_FULL + ks));
          }
        }
        __syncwarp();
      };
      // TF32 / HYB step: the first unit's MMA1 stages are requested right behind the two owner slabs each of them
      // meets, so MMA1 starts after ~48 KB have landed instead of after the whole 160 KB (every CTA fills at once:
      // the fill is bound by the aggregate L2 bandwidth)
      constexpr bool kInterleaveFill = kBwd && !kSplit;
      if (!kInterleaveFill) {
        for (int i = 0; i < oslabs; ++i)
          load_own((kPlanes == 2) ? (i & 1) * hs + (i >> 1) : i);   // SPLIT: hi chunk c, then lo chunk c
      }
      if (!kBwd) {
        for (int u = s0; u < s1; u += kStepUnits) {
          const int nu = min(kStepUnits, s1 - u);
          for (int ks = 0; ks < oslabs; ++ks) load_k(tm_k, u * kUnit, nu * kUnit / CG, ks, 1);
        }
      } else {
        auto load_mma1_unit = [&](int u) {       // stages of two slabs, n = 128
          for (int ks = 0; ks < oslabs; ks += 2) load_k(tm_k, u * kUnit, kUnit / CG, ks, min(2, oslabs - ks));
        };
        const int u0 = wk.unit(0, s0, s1), nun = s1 - s0;
        if (kInterleaveFill) {
          for (int ks = 0; ks < oslabs; ks += 2) {
            const int n = min(2, oslabs - ks);
            for (int q = 0; q < n; ++q) load_own(ks + q);
            load_k(tm_k, u0 * kUnit, kUnit / CG, ks, n);
          }
        } else {
          load_mma1_unit(u0);
        }
        for (int i = 0; i < nun; ++i) {
          const int u = wk.unit(i, s0, s1);
          if (i + 1 < nun) load_mma1_unit(wk.unit(i + 1, s0, s1));
          for (int kc = 0; kc < kUnit / kM2; ++kc) load_mn(tm_mn, u * kUnit + kc * kM2);
        }
      }
      tr.mark();   // all loads of the segment issued
    }
  } else if (warp == 1) {
    // ===================================================================== MMA issuer (leader CTA)
    if (leader) {
      const uint32_t idesc2 = kSplit ? idesc_f16(kTile * CG, p.D, 0, 1) : idesc_tf32(kTile * CG, p.D, 0, 1);
      // descriptor templates: only the 14-bit start-address field changes per MMA
      const uint64_t dk = smem_desc(0, 16, 1024, kLayoutSw128);                        // K-major
      // MN-major: TF32 needs the 32-byte-atom swizzle (4-row groups), fp16 the plain 128B swizzle (8-row groups)
      const uint64_t dmn = kSplit ? smem_desc(0, kM2 * 128, 1024, kLayoutSw128)
                                  : smem_desc(0, kMma2Rows * 128, 512, kLayoutSw128Base32);
      int stage = 0, phase = 0, sg = 0, it = 0;
      Tracer<DBG> tr(lane == 0 ? p.trace : nullptr, 1);
      tr.mark();
      auto advance = [&]() { if (++stage == kStages) { stage = 0; phase ^= 1; } };
      auto commit = [&](int b) {
        if (CG == 1) umma_commit(bar(b)); else umma_commit_2cta(bar(b), kPairMask);
      };
      // A stage is issued from one asm block (umma_stage_ss / umma_stage_ts) that first probes the
      // NEXT stage's FULL barrier: when the probe succeeded the blocking wait (~200 clk even on a
      // completed barrier) is skipped.  The loop is instruction-bound, see ge2e_tc_ptx.cuh.
      bool ready = false;          // FULL[stage] was seen complete by the previous stage's probe
      uint32_t leader = 0;         // lane elected to issue (same value in every lane)
      auto stage_wait = [&]() {
        if (DBG && (dbg & 8)) tr.mark();     // fine trace: before / after the wait for the stage's data
        if (!ready) mbar_wait(bar(BAR_FULL + stage), phase);
        if (DBG && (dbg & 8)) tr.mark();
        tc_fence_after();
      };
      auto next_bar = [&]() { return bar(BAR_FULL + (stage + 1 == kStages ? 0 : stage + 1)); };
      auto next_par = [&]() { return static_cast<uint32_t>(stage + 1 == kStages ? (phase ^ 1) : phase); };
      auto stage_done = [&](uint32_t probe) {
        __syncwarp();
        ready = __shfl_sync(0xffffffffu, probe, leader) != 0;
        advance();
      };
      // MMA1 over one stage holding `nslab` (1 or 2) K-slabs of [rows_cta x 32] starting at slab ks0
      auto mma1_stage = [&](uint32_t d_tmem, uint32_t idesc1, int rows_cta, int ks0, int nslab, bool first_of_seg) {
        if (kOpF16) {
          // stream slab s = (plane, chunk c): a hi slab meets the owner's hi AND lo chunk c (8 MMAs), a lo slab
          // the owner's hi chunk (4 MMAs); lo.lo is below fp32 resolution and is not formed
          if (first_of_seg) {
            for (int sl = 0; sl < nslab; ++sl) {
              const int s = ks0 + sl, c = s % hs;
              mbar_wait(bar(BAR_A_FULL + c), sg & 1);
              if (kPlanes == 2 && s < hs) mbar_wait(bar(BAR_A_FULL + hs + c), sg & 1);
            }
          }
          stage_wait();
          uint32_t probe = 0;
          if (elect_leader(leader)) {
            probe = mbar_test(next_bar(), next_par());
            for (int sl = 0; sl < nslab; ++sl) {
              const int s = ks0 + sl, c = s % hs;
              const uint64_t db = dk | ((ring_smem + stage * kStageBytes + sl * rows_cta * 128) >> 4);
              umma_f16_ss4<CG>(d_tmem, dk | ((a_smem + c * kSlabBytes) >> 4), db, idesc1, s != 0);
              if (kPlanes == 2 && s < hs)
                umma_f16_ss4<CG>(d_tmem, dk | ((a_smem + (hs + c) * kSlabBytes) >> 4), db, idesc1, 1);
            }
            commit(BAR_EMPTY + stage);
          }
          stage_done(probe);
          return;
        }
        if (first_of_seg) {
          for (int sl = 0; sl < nslab; ++sl) mbar_wait(bar(BAR_A_FULL + ks0 + sl), sg & 1);
        }
        stage_wait();
        uint32_t probe = 0;
        if (elect_leader(leader)) {
          const uint64_t da = dk | ((a_smem + ks0 * kSlabBytes) >> 4);
          const uint64_t db = dk | ((ring_smem + stage * kStageBytes) >> 4);
          const uint32_t eb = bar(BAR_EMPTY + stage);
          if (nslab == 2)
            probe = umma_stage_ss<CG, 2>(d_tmem, da, db, kSlabBytes >> 4, static_cast<uint32_t>(rows_cta * 128) >> 4,
                                         idesc1, ks0 != 0, eb, next_bar(), next_par());
          else
            probe = umma_stage_ss<CG, 1>(d_tmem, da, db, 0, 0, idesc1, ks0 != 0, eb, next_bar(), next_par());
        }
        stage_done(probe);
      };
      const uint32_t idesc_unit = kOpF16 ? idesc_f16(kTile * CG, kUnit, 0, 0) : idesc_tf32(kTile * CG, kUnit, 0, 0);
      auto mma1_unit = [&](int iter, bool first_of_seg) {   // BWD: n = 128 into T[iter & 1]
        const uint32_t d_tmem = tmem + (iter & 1) * kUnit;
        for (int ks = 0; ks < oslabs; ks += 2)
          mma1_stage(d_tmem, idesc_unit, kUnit / CG, ks, min(2, oslabs - ks), first_of_seg);
        if (elect_one()) commit(BAR_S_FULL + (iter & 1));
        __syncwarp();
      };
      auto mma2_unit = [&](int iter, bool first) {
        const uint32_t a_tmem = tmem + (iter & 1) * kUnit;
        const uint32_t d_tmem = tmem + 2 * kUnit;
        for (int kc = 0; kc < kUnit / kM2; ++kc) {
          stage_wait();
          uint32_t probe = 0;
          if (PREC == PREC_F16) {
            if (elect_leader(leader)) {
              probe = mbar_test(next_bar(), next_par());
              // the stage's 64 stream rows are column half kc of T: 32 cells of packed fp16 pairs = 4 K steps
              const uint32_t a_hi = a_tmem + 64 * kc;
              const uint64_t db_hi = dmn | ((ring_smem + stage * kStageBytes) >> 4);
              umma_f16_ts2<CG>(d_tmem, a_hi, db_hi, idesc2, !(first && kc == 0));
              umma_f16_ts2<CG>(d_tmem, a_hi + 16, db_hi + 256, idesc2, 1);      // rows 32..63: 4096 bytes further
              commit(BAR_EMPTY + stage);
            }
            stage_done(probe);
            continue;
          }
          if (kSplit) {
            if (elect_leader(leader)) {
              probe = mbar_test(next_bar(), next_par());
              // P / G planes in T (see the epilogue): column half h = kc / 2 holds [hi 32 cols | lo 32 cols] of
              // its 64 stream rows; the stage's 32 rows start 16 columns into the plane when kc is odd
              const uint32_t a_hi = a_tmem + 64 * (kc >> 1) + 16 * (kc & 1), a_lo = a_hi + 32;
              const uint32_t sb = ring_smem + stage * kStageBytes;
              const uint64_t db_hi = dmn | (sb >> 4);
              const uint64_t db_lo = dmn | ((sb + (hs / CG) * kMma2Rows * 128) >> 4);
              umma_f16_ts2<CG>(d_tmem, a_hi, db_hi, idesc2, !(first && kc == 0));
              if (kPlanes == 2) {
                umma_f16_ts2<CG>(d_tmem, a_hi, db_lo, idesc2, 1);
                umma_f16_ts2<CG>(d_tmem, a_lo, db_hi, idesc2, 1);
              }
              commit(BAR_EMPTY + stage);
            }
            stage_done(probe);
            continue;
          }
          if (elect_leader(leader)) {
            // MN-major TF32 operand: 32-byte-atom 128B swizzle, chunks of 32 columns kMma2Rows*128 B
            // apart (LBO), groups of 4 k-rows 512 B apart (SBO); one MMA consumes 8 k-rows = 1024 B
            const uint64_t db = dmn | ((ring_smem + stage * kStageBytes) >> 4);
            static_assert(kMma2Rows == 32, "umma_stage_ts issues 4 MMAs of 8 k-rows");
            probe = umma_stage_ts<CG>(d_tmem, a_tmem + kc * kMma2Rows, db, idesc2, !(first && kc == 0),
                                      bar(BAR_EMPTY + stage), next_bar(), next_par());
          }
          stage_done(probe);
        }
      };
      Walk wk = make_walk();
      int kind, og, s0, s1;
      for (; wk.next(p, kind, og, s0, s1); ++sg) {
        if (!kBwd) {
          for (int u = s0; u < s1; u += kStepUnits, ++it) {
            const int nu = min(kStepUnits, s1 - u);
            mbar_wait(bar(BAR_S_EMPTY + (it & 1)), ((it >> 1) & 1) ^ 1);
            tc_fence_after();
            const uint32_t d_tmem = tmem + (it & 1) * (kStepUnits * kUnit);
            const uint32_t idesc_step = kOpF16 ? idesc_f16(kTile * CG, nu * kUnit, 0, 0)
                                               : idesc_tf32(kTile * CG, nu * kUnit, 0, 0);
            for (int ks = 0; ks < oslabs; ++ks) mma1_stage(d_tmem, idesc_step, nu * kUnit / CG, ks, 1, u == s0);
            if (elect_one()) commit(BAR_S_FULL + (it & 1));
            __syncwarp();
            tr.mark();   // step issued
          }
          if (elect_one()) commit(BAR_A_EMPTY);
          __syncwarp();
        } else {
          mma1_unit(it, true);
          for (int i = 0; i < s1 - s0; ++i, ++it) {
            if (i + 1 < s1 - s0) {
              mma1_unit(it + 1, false);
            } else {
              if (elect_one()) commit(BAR_A_EMPTY);
              __syncwarp();
            }
            tr.mark();   // MMA1(next) issued
            if (i == 0 && sg > 0) { mbar_wait(bar(BAR_ACC_EMPTY), (sg - 1) & 1); tc_fence_after(); }
            mbar_wait(bar(BAR_G_FULL + (it & 1)), (it >> 1) & 1);
            tc_fence_after();
            tr.mark();   // G landed
            mma2_unit(it, i == 0);
            tr.mark();   // MMA2 issued
          }
          if (elect_one()) commit(BAR_ACC_FULL);
          __syncwarp();
        }
      }
    }
  } else if (warp >= kEpiWarp0) {
    // ===================================================================== epilogue
    const int ew = warp - kEpiWarp0;
    const int et = tid - kEpiWarp0 * 32;             // thread index among the epilogue threads
    const int quarter = ew & 3, half = ew >> 2;      // TMEM lanes [32 q, 32 q + 32); column half h
    const int trow = quarter * 32 + lane;            // row inside the owner tile
    const uint32_t lane_addr = static_cast<uint32_t>(quarter * 32) << 16;
    const float w = __ldg(p.w), b = __ldg(p.b), eps = p.eps;
    const float w2 = w * kLog2e, b2 = fmaf(w, eps, b) * kLog2e;   // log2-domain affine: S*log2e
    const float bb = fmaf(w, eps, b);
    const float g = (kBwd && !RG && p.grad_out != nullptr) ? __ldg(p.grad_out) : 1.f;
    const float wg = w * g;
    float gamma = 1.f, inv_gamma = 1.f;   // RG, SPLIT pass 2: max_r |g_r| and its inverse (0 when every g_r is 0)
    // RG: sign bits of g_r for stream rows [32 w, 32 w + 32) of the unit staged in buffer buf
    auto gsign_of = [&](int buf, int w) -> uint32_t {
      if constexpr (RG) return tail->gsign[buf][w]; else return 0u;
    };
    // STEP, pass 1: every logit is bounded by |w| + (w eps + b) because |cos| <= 1, so the exponentials are
    // taken against that FIXED shift (log2 domain: m2) instead of a running row maximum: P <= 1, partial row
    // sums and partial accumulators of different clusters simply add, nothing is ever rescaled.  The
    // smallest P is 2^(-2 |w| log2e), a normal fp32 number for |w| <= 43 (the reference's own exp(S) is
    // un-stabilised, s3:120, and overflows beyond w + b = 88).
    const float m2 = b2 + fabsf(w2), c0 = -fabsf(w2);
    float dw_acc = 0.f, db_acc = 0.f, loss_acc = 0.f;
    int it = 0;
    // STEP: the rows are closed in this launch (TF32: pass 1 produces the row sums) or were closed by the
    // forward kernel in front of it (SPLIT: the probabilities must be normalised BEFORE they are cut into
    // fp16 planes, so the log-sum-exp has to be known when pass 1 starts)
    const bool close_here = kBwd && !kSplit && (p.phases & PASS_ROWS);
    Tracer<DBG> tr((trow == 0 && half == 0) ? p.trace : nullptr, 2, kBwd ? 3 : 0);
    tr.mark();
    // epilogue -> MMA signals go to the leader CTA of the pair
    const uint32_t s_empty0 = lbar(BAR_S_EMPTY), g_full0 = lbar(BAR_G_FULL), acc_empty = lbar(BAR_ACC_EMPTY);
    auto arrive_leader = [&](uint32_t addr) {
      if (CG == 1) mbar_arrive(addr); else mbar_arrive_cluster(addr);
    };
    // spin until *ctr >= target (all CTAs of the persistent grid are co-resident); a counter that never
    // gets there is a bug: trap after 2 s instead of hanging the GPU
    auto spin_until = [&](const int* ctr, int target) {
      unsigned long long t0 = 0;
      for (unsigned spins = 0;; ++spins) {
        int v;
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
        if (v >= target) break;
        if ((spins & 1023u) == 1023u) {
          const unsigned long long t = globaltimer_ns();
          if (t0 == 0) t0 = t;
          else if (t - t0 > 2000000000ull) __trap();
        }
      }
    };
    bool zero_seen = false;      // (thread et 0) every CTA has finished its share of the zero-fill
    auto wait_zero_fill = [&]() {
      if (zero_seen) return;
      spin_until(p.ctr, static_cast<int>(gridDim.x));
      asm volatile("fence.proxy.async;" ::: "memory");    // the TMA reduce below is an async-proxy access
      zero_seen = true;
    };
    if (kBwd) {
      // Outputs that collect partial sums from many CTAs (dC_hat; dE_hat when its owner groups are cut; the
      // row sums) are zeroed here instead of with memset nodes in front of the kernel: every CTA clears a
      // slice while its pipeline fills and bumps ctr[0]; nobody adds before ctr[0] == gridDim.x.
      auto zfill = [&](float4* base, long long n4) {
        const long long z0 = n4 * blockIdx.x / gridDim.x, z1 = n4 * (blockIdx.x + 1) / gridDim.x;
        for (long long i = z0 + et; i < z1; i += kEpiThreads) base[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      };
      if (p.zero_n4 > 0) zfill(p.zero_base, p.zero_n4);
      if (p.zero2_n4 > 0) zfill(p.zero2_base, p.zero2_n4);
      if (close_here) zfill(reinterpret_cast<float4*>(p.rowsum), (p.n_own[SEG_DE] + 3) / 4);
      if (et == 0) tail->rows_all_done = 0;
      __threadfence();
      named_bar_sync(1, kEpiThreads);
      if (et == 0) atomicAdd(p.ctr, 1);
    }

    // STEP: closing a row -- log-sum-exp, row loss, q = 1 - p_jj, the factor of the un-normalised dE_hat row; the
    // diagonal terms of dw and the closed-form db (SURVEY 8(a-bis) items 8, 12) ride along.  close_here: once per
    // utterance tile, by the CTA whose pass-1 segment completes the tile's row sums (close_tile); otherwise every
    // CTA closes a grid-strided slice of rows whose statistics an earlier launch wrote (close_rows).
    int lift2 = kSplitLift;      // SPLIT pass 2: exponent of the probability planes (set by close_rows)
    auto close_row = [&](int r) {
      const float cdv = __ldg(p.cos_diag + r);
      float stat, q;
      if (close_here) {
        const RowClose rc = close_softmax_row_log2(m2, __ldcg(p.rowsum + r), fmaf(cdv, w2, b2),
                                                   fmaf(w, cdv + eps, b), eps);      // s3:120-121
        stat = rc.stat; q = rc.q;
        p.row_stat_out[r] = stat;
        p.row_aux_out[r] = q;
        p.row_scale_out[r] = w / rc.z;      // = w exp(m - lse_r)
        if (p.per_row_out != nullptr) p.per_row_out[r] = rc.per;
        loss_acc += rc.per;
      } else {
        stat = __ldg(p.row_stat + r);
        q = __ldg(p.row_aux + r);
        if (kSplit && (p.phases & PASS_ROWS))      // dE_hat row r was formed from p * 2^(14 + k_r)
          p.row_scale_out[r] = w * exp2f(static_cast<float>(-(kSplitLift + split_extra_lift(q))));
      }
      if (p.phases & PASS_CENTROIDS) {
        if (RG) {
          const float gr = __ldg(p.grad_rows + r);
          dw_acc = fmaf(-q * gr, cdv + eps, dw_acc);
          db_acc -= gr * eps * expf(-stat);
        } else {
          dw_acc = fmaf(-q, cdv + eps, dw_acc);     // diagonal element G_jj = -g q (uses cos_diag)
          db_acc -= eps * expf(-stat);              // item 12: db = -g sum eps / (sum exp + eps)
        }
      }
    };
    auto close_rows = [&]() {
      const int U = p.n_own[SEG_DE];
      if (kSplit && (p.phases & PASS_CENTROIDS)) {
        // pass 2's lift: every CTA takes the maximum of q over ALL rows (U floats out of the L2)
        if (RG) {
          // the planes carry p g_r / gamma: the lift comes from max_r q_r |g_r| / gamma
          float qm = 0.f, gm = 0.f;
          for (int r = et; r < U; r += kEpiThreads) {
            const float ga = fabsf(__ldg(p.grad_rows + r));
            qm = fmaxf(qm, __ldg(p.row_aux + r) * ga);
            gm = fmaxf(gm, ga);
          }
          qm = warp_max(qm);
          gm = warp_max(gm);
          if (lane == 0) { tail->red[ew] = qm; tail->red[kEpiWarps + ew] = gm; }
          named_bar_sync(1, kEpiThreads);
          qm = tail->red[0];
          gm = tail->red[kEpiWarps];
          for (int i = 1; i < kEpiWarps; ++i) { qm = fmaxf(qm, tail->red[i]); gm = fmaxf(gm, tail->red[kEpiWarps + i]); }
          gamma = gm;
          inv_gamma = gm > 0.f ? 1.f / gm : 0.f;
          lift2 = kSplitLift + split_extra_lift(qm * inv_gamma);
        } else {
          float qm = 0.f;
          for (int r = et; r < U; r += kEpiThreads) qm = fmaxf(qm, __ldg(p.row_aux + r));
          qm = warp_max(qm);
          if (lane == 0) tail->red[ew] = qm;
          named_bar_sync(1, kEpiThreads);
          qm = tail->red[0];
          for (int i = 1; i < kEpiWarps; ++i) qm = fmaxf(qm, tail->red[i]);
          lift2 = kSplitLift + split_extra_lift(qm);
        }
        named_bar_sync(1, kEpiThreads);      // red is reused by the scalar reductions
      }
      for (int r = blockIdx.x * kEpiThreads + et; r < U; r += gridDim.x * kEpiThreads) close_row(r);
      tr.mark();   // rows closed
    };
    // close_here, pass 2: stream unit u is utterance tile u (kUnit == kTile), its row sums are final once every
    // pass-1 segment of that tile has counted its units into seg_done[u].  No deadlock: pass-1 work never waits
    // on pass 2 (a CTA's pass-1 segments precede its pass-2 segments, the TMA and MMA warps need no row
    // statistics), and every CTA of the grid is co-resident (max_clusters).
    static_assert(kUnit == kTile, "a pass-2 stream unit must be exactly one pass-1 owner tile");
    unsigned long long ready_wait_ns = 0;      // DBG: time this thread spent waiting for row sums
    // ctr[2] counts complete tiles: once a CTA has seen all of them, its pass-2 units need no acquire load
    // in front of their row-sum loads (most of pass 2 at large shapes)
    auto tile_ready = [&](int u) {
      if (*reinterpret_cast<volatile int*>(&tail->rows_all_done) != 0) return true;
      int v;
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p.ctr + 2) : "memory");
      if (v >= p.OT[SEG_DE]) { tail->rows_all_done = 1; return true; }
      asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p.seg_done + u) : "memory");
      return v >= p.ST[SEG_DE];
    };
    auto wait_tile = [&](int u) {
      if (tile_ready(u)) return;
      const unsigned long long t0 = DBG ? globaltimer_ns() : 0ull;
      spin_until(p.seg_done + u, p.ST[SEG_DE]);
      if (DBG) ready_wait_ns += globaltimer_ns() - t0;
    };
    bool closed = false;
    int sg_dc0 = -1;             // DBG: first pass-2 segment

    Walk wk = make_walk();
    int kind, og, s0, s1;
    for (int sg = 0; wk.next(p, kind, og, s0, s1); ++sg) {
      const bool is_dc = kBwd && kind == SEG_DC;       // CTA-uniform
      if (kBwd && !close_here && is_dc && !closed) { close_rows(); closed = true; }
      if (DBG && is_dc && sg_dc0 < 0) { sg_dc0 = sg; tr.put(kTraceEvents - 2, globaltimer_ns()); }   // pass 2 begins
      const int n_str = p.n_str[kind];
      const int ot = og * CG + cr;
      const bool tile_valid = ot < p.OT[kind];         // CTA-uniform
      const int orow = ot * kTile + trow;              // owner row (utterance, or centroid in a DC segment)
      const bool ovalid = orow < p.n_own[kind];
      // per-owner-row metadata
      int jg = -1;            // FWD / DE: global speaker of this utterance row
      float cd = 0.f;
      int dlo = 0, dhi = 0;   // DC: local utterance rows [dlo, dhi) belong to this centroid
      if (!is_dc) {
        if (ovalid) {
          jg = p.spk_offset + orow / p.M;
          if (!kBwd) cd = __ldg(p.cos_diag + orow);
        }
      } else {
        const int jl = orow - p.spk_offset;
        if (ovalid && jl >= 0 && (long long)jl * p.M < n_str) { dlo = jl * p.M; dhi = dlo + p.M; }
      }
      // FWD softmax running state, log2 domain, OFF-diagonal columns only: the running max starts at
      // the diagonal logit (known from cos_diag) and the diagonal term joins when the row is closed
      const float xd2 = fmaf(cd, w2, b2);
      float m2r = xd2, lsum = 0.f;
      float best = -INFINITY; int bestk = INT_MAX;   // FWD contrast
      float rs_acc = 0.f;                            // STEP pass 1: this thread's share of the row sum
      float dw_seg = 0.f;                            // STEP pass 2: sum p (cos + eps) of this centroid row
      // STEP pass 2: lse (log2 domain) of stream row ur from its raw inputs -- the row sum of pass 1 when both
      // passes run in this launch (row_stat was written by other CTAs after the barrier), else row_stat
      auto lse2_of = [&](bool valid, float raw, float cdv) -> float {
        if (!valid) return INFINITY;
        if (!close_here) return raw * kLog2e;
        return close_softmax_row_log2(m2, raw, fmaf(cdv, w2, b2), fmaf(w, cdv + eps, b), eps).lse2;
      };
      auto lse2_raw = [&](int ur, float& raw, float& cdv) -> bool {
        if (ur >= n_str) return false;
        if (close_here) { raw = __ldcg(p.rowsum + ur); cdv = __ldg(p.cos_diag + ur); }
        else { raw = __ldg(p.row_stat + ur); cdv = 0.f; }
        return true;
      };
      // SPLIT pass 1: exponent offset of this owner row, P * 2^14 = exp2(S w2 + c0r); a row past the end gives 0
      float c0r = 0.f;
      if (kBwd && kSplit && !is_dc)
        c0r = ovalid ? (b2 + static_cast<float>(kSplitLift + split_extra_lift(__ldg(p.row_aux + orow)))) -
                           __ldg(p.row_stat + orow) * kLog2e
                     : -INFINITY;
      // lse_s[buf] of unit u, loaded when this unit's turn comes (close_here: once its row sums are final)
      // RG: g_r of stream row ur (0 past the end), loaded with the row's other inputs
      auto grad_of = [&](int ur) -> float { return (RG && ur < n_str) ? __ldg(p.grad_rows + ur) : 0.f; };
      // lse_s[buf][trow] (+ RG: |g_r| folded in, its sign into gsign); every lane of the warp takes part
      auto stage_row = [&](int buf, bool valid, float raw, float cdv, float gr) {
        float l = lse2_of(valid, raw, cdv);
        if constexpr (RG) {
          l -= log2f(fabsf(gr) * inv_gamma);      // exp2(. - l) = p |g_r| (/ gamma); g_r = 0: l = +inf, p = 0
          const uint32_t neg = __ballot_sync(0xffffffffu, gr < 0.f);
          if (lane == 0) tail->gsign[buf][quarter] = neg;
        }
        tail->lse_s[buf][trow] = l;
      };
      auto stage_lse = [&](int u, int buf) {
        if (close_here) wait_tile(u);
        float raw = 0.f, cdv = 0.f;
        const bool v = lse2_raw(u * kUnit + trow, raw, cdv);
        stage_row(buf, v, raw, cdv, grad_of(u * kUnit + trow));
      };
      if (is_dc && half == 0) stage_lse(wk.unit(0, s0, s1), it & 1);
      bool deferred = false;     // the next unit's row sums were not final at prefetch time: staged at its turn

      for (int i = 0; i < s1 - s0; i += kStepUnits, ++it) {
        const int u = wk.unit(i, s0, s1);
        const int nu = min(kStepUnits, s1 - s0 - i);
        const int buf = it & 1;
        float nraw = 0.f, ncd = 0.f, ngr = 0.f;
        bool nvalid = false;
        if (is_dc) {
          if (half == 0 && deferred) { stage_lse(u, buf); deferred = false; }
          named_bar_sync(1, kEpiThreads);      // lse_s[buf] staged (by the previous unit, above, or just now)
          // the next unit's raw inputs travel while this unit is processed -- if its row sums are final already:
          // a poll, never a wait, so that a late tile holds up its own unit only
          if (half == 0 && i + 1 < s1 - s0) {
            const int un = wk.unit(i + 1, s0, s1);
            if (!close_here || tile_ready(un)) {
              nvalid = lse2_raw(un * kUnit + trow, nraw, ncd);
              ngr = grad_of(un * kUnit + trow);
            }
            else deferred = true;
          }
        }
        mbar_wait(bar(BAR_S_FULL + buf), (it >> 1) & 1);
        tc_fence_after();
        tr.mark();   // T tile ready
        const uint32_t t_addr = tmem + lane_addr + buf * (kStepUnits * kUnit);
        const int nch = nu * (kUnit / 32) / 2;       // 32-column chunks per column half
        if (kBwd && kSplit) {
          // This thread's 64 columns of T become [hi plane: 32 cells | lo plane: 32 cells] of packed fp16 pairs
          // IN PLACE, so all 64 are read before the first cell is written.
          const uint32_t tb = t_addr + half * 64;
          uint32_t v0[32], v1[32];
          tmem_ld32(tb, v0);
          tmem_ld32(tb + 32, v1);
          tmem_ld_wait();
          auto plane_chunk = [&](const uint32_t (&v)[32], int c2) {
            const int ch = half * 2 + c2;
            const int cc = u * kUnit + ch * 32;
            uint32_t hi[16], lo[16];
            if (!is_dc) {
              const bool special = (cc + 32 > n_str) || (static_cast<unsigned>(jg - cc) < 32u);
              const bool any_special = __any_sync(0xffffffffu, special);
#pragma unroll
              for (int i = 0; i < 32; i += 2) {
                float p0 = ex2(fmaf(__uint_as_float(v[i]), w2, c0r));
                float p1 = ex2(fmaf(__uint_as_float(v[i + 1]), w2, c0r));
                if (any_special) {     // padding / own speaker (s3:78)
                  if (cc + i >= n_str || cc + i == jg) p0 = 0.f;
                  if (cc + i + 1 >= n_str || cc + i + 1 == jg) p1 = 0.f;
                }
                split_pack(p0, p1, hi[i >> 1], lo[i >> 1]);
              }
            } else {
              const float* ls = &tail->lse_s[buf][ch * 32];
              const bool special = (cc < dhi) && (cc + 32 > dlo);
              const bool any_special = __any_sync(0xffffffffu, special);
              const float b2s = b2 + static_cast<float>(lift2);
              const uint32_t neg = gsign_of(buf, ch);     // RG: signs of g_r (|g_r| / gamma is in ls)
#pragma unroll
              for (int i = 0; i < 32; i += 2) {
                const float2 l2 = *reinterpret_cast<const float2*>(ls + i);
                const float d0 = __uint_as_float(v[i]), d1 = __uint_as_float(v[i + 1]);
                float p0 = ex2(fmaf(d0, w2, b2s) - l2.x);       // lse = +inf past the end
                float p1 = ex2(fmaf(d1, w2, b2s) - l2.y);
                if (any_special) {     // own speaker's rows
                  if (cc + i >= dlo && cc + i < dhi) p0 = 0.f;
                  if (cc + i + 1 >= dlo && cc + i + 1 < dhi) p1 = 0.f;
                }
                if (RG) {
                  if ((neg >> i) & 1u) p0 = -p0;
                  if ((neg >> (i + 1)) & 1u) p1 = -p1;
                }
                dw_seg = fmaf(p0, d0 + eps, dw_seg);
                dw_seg = fmaf(p1, d1 + eps, dw_seg);
                split_pack(p0, p1, hi[i >> 1], lo[i >> 1]);
              }
            }
            tmem_st16(tb + 16 * c2, hi);
            if (kPlanes == 2) tmem_st16(tb + 32 + 16 * c2, lo);
          };
          plane_chunk(v0, 0);
          plane_chunk(v1, 1);
        } else
#pragma unroll 1
        for (int ch = half * nch; ch < (half + 1) * nch; ++ch) {
          const int cc = u * kUnit + ch * 32;        // first stream row (column of T) of this chunk
          uint32_t v[32];
          tmem_ld32(t_addr + ch * 32, v);
          tmem_ld_wait();
          if (!kBwd) {
            if (cc < n_str) {
              const bool tailc = cc + 32 > n_str;
              const bool diagc = static_cast<unsigned>(jg - cc) < 32u;
              if (VARIANT == GE2E_SOFTMAX) {
                float x[32];
#pragma unroll
                for (int i = 0; i < 32; ++i) x[i] = fmaf(__uint_as_float(v[i]), w2, b2);
                if (__any_sync(0xffffffffu, tailc || diagc)) {
#pragma unroll
                  for (int i = 0; i < 32; ++i)   // own-speaker column (s3:78) and padding leave the sum
                    if (cc + i == jg || cc + i >= n_str) x[i] = -INFINITY;
                }
                float cm = x[0];
#pragma unroll
                for (int i = 1; i < 32; ++i) cm = fmaxf(cm, x[i]);
                const float mn = fmaxf(m2r, cm);
                float sacc = 0.f;
#pragma unroll
                for (int i = 0; i < 32; ++i) sacc += ex2(x[i] - mn);
                lsum = fmaf(lsum, ex2(m2r - mn), sacc);
                m2r = mn;
              } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                  float sv = fmaf(__uint_as_float(v[i]), w, bb);
                  if (cc + i == jg || cc + i >= n_str) sv = -INFINITY;
                  if (sv > best) { best = sv; bestk = cc + i; }
                }
              }
            }
          } else {
            uint32_t gq[32];
            if (!is_dc) {
              // ---- pass 1: P tile (fixed shift), written back over T; row sums on the side
              const bool special = (cc + 32 > n_str) || (static_cast<unsigned>(jg - cc) < 32u);
              const bool any_special = __any_sync(0xffffffffu, special);
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                float pr = ex2(fmaf(__uint_as_float(v[i]), w2, c0));
                if (any_special && (cc + i >= n_str || cc + i == jg)) pr = 0.f;   // padding / own speaker (s3:78)
                rs_acc += pr;
                gq[i] = __float_as_uint(round_tf32(pr));
              }
            } else {
              // ---- pass 2: G tile = w g softmax(S), own speaker's rows masked, written back over T
              const float4* ls4 = reinterpret_cast<const float4*>(&tail->lse_s[buf][ch * 32]);
              const uint32_t neg = gsign_of(buf, ch);     // RG: signs of g_r (|g_r| is in ls4)
              const bool special = (cc < dhi) && (cc + 32 > dlo);
              const bool any_special = __any_sync(0xffffffffu, special);
#pragma unroll
              for (int i4 = 0; i4 < 8; ++i4) {
                const float4 l4 = ls4[i4];
                const float ls[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const int i = i4 * 4 + q;
                  const float dot = __uint_as_float(v[i]);
                  float pr = ex2(fmaf(dot, w2, b2) - ls[q]);                     // lse = +inf past the end
                  if (any_special && cc + i >= dlo && cc + i < dhi) pr = 0.f;    // own speaker's rows
                  if (RG && ((neg >> i) & 1u)) pr = -pr;                          // g_r p_rk
                  dw_seg = fmaf(pr, dot + eps, dw_seg);
                  gq[i] = __float_as_uint(round_tf32(wg * pr));
                }
              }
            }
            tmem_st32(t_addr + ch * 32, gq);
          }
        }
        tr.mark();   // tile consumed
        if (!kBwd) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) arrive_leader(s_empty0 + 8u * buf);
        } else {
          if (is_dc && half == 0 && i + 1 < s1 - s0 && !deferred) stage_row(buf ^ 1, nvalid, nraw, ncd, ngr);
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) arrive_leader(g_full0 + 8u * buf);
        }
      }

      // ------------------------------------------------------------ segment flush
      const bool full = (s0 == 0 && s1 == p.ST[kind]);
      if (!kBwd) {
        // fold the two column halves of every row (upper half hands its state over through smem)
        float2 mine;
        if (VARIANT == GE2E_SOFTMAX) mine = make_float2(m2r, lsum);
        else mine = make_float2(best, __int_as_float(bestk));
        if (half == 1) tail->xch[trow] = mine;
        named_bar_sync(1, kEpiThreads);
        const float2 theirs = tail->xch[trow];
        named_bar_sync(1, kEpiThreads);    // xch may be rewritten by the next segment from here on
        if (half == 0 && tile_valid) {     // tile_valid is CTA-uniform: barrier 2 below stays consistent
          auto fold = [&](float2 q) {
            if (VARIANT == GE2E_SOFTMAX) {
              const float mn = fmaxf(m2r, q.x);
              lsum = lsum * ex2(m2r - mn) + q.y * ex2(q.x - mn);
              m2r = mn;
            } else {
              const int qk = __float_as_int(q.y);
              if (q.x > best || (q.x == best && qk < bestk)) { best = q.x; bestk = qk; }
            }
          };
          fold(theirs);
          // publish the partial row state, last finisher of this owner tile merges
          const int st = p.ST[SEG_DE];
          const int first_cl = cluster_of_pair(static_cast<long long>(og) * st, p.GP, NC);
          bool last = full;
          if (!full) {
            float2 part;
            if (VARIANT == GE2E_SOFTMAX) part = make_float2(m2r, lsum);
            else part = make_float2(best, __int_as_float(bestk));
            p.seg_part[(static_cast<size_t>(ot) * p.maxseg + (cl - first_cl)) * kTile + trow] = part;
            __threadfence();
            named_bar_sync(2, kTile);
            if (trow == 0) {
              const int done = atomicAdd(p.seg_done + ot, s1 - s0) + (s1 - s0);
              tail->flag = (done == st);
              if (done == st) p.seg_done[ot] = 0;      // leave the workspace zeroed for the next call
            }
            named_bar_sync(2, kTile);
            last = tail->flag != 0;
            if (last) {
              __threadfence();
              const int last_cl = cluster_of_pair(static_cast<long long>(og) * st + st - 1, p.GP, NC);
              const int nseg = last_cl - first_cl + 1;
              m2r = xd2; lsum = 0.f; best = -INFINITY; bestk = INT_MAX;
              for (int sgi = 0; sgi < nseg; ++sgi)
                fold(__ldcg(&p.seg_part[(static_cast<size_t>(ot) * p.maxseg + sgi) * kTile + trow]));
            }
          }
          if (last && ovalid) {
            const float Sd = fmaf(w, cd + eps, b);
            float per, stat, aux = 0.f;
            int ks = -1;
            if (VARIANT == GE2E_SOFTMAX) {
              const RowClose rc = close_softmax_row_log2(m2r, lsum, xd2, Sd, eps);   // s3:120-121
              stat = rc.stat; aux = rc.q; per = rc.per;
            } else {
              per = 1.f - 1.f / (1.f + expf(-Sd));
              stat = best;
              if (bestk != INT_MAX) { ks = bestk; per += 1.f / (1.f + expf(-best)); }
            }
            p.row_stat_out[orow] = stat;
            if (p.row_aux_out != nullptr) p.row_aux_out[orow] = aux;
            if (VARIANT == GE2E_CONTRAST && p.kstar_out != nullptr) p.kstar_out[orow] = ks;
            if (p.per_row_out != nullptr) p.per_row_out[orow] = per;
            loss_acc += per;
          }
        }
      } else {
        // pass 1: the row sums are final once the last tile has been consumed -- they do not wait for the
        // accumulator; the segment counts its units into the tile's counter and the CTA that completes the tile
        // closes its rows, all while the last MMA2 of the segment runs
        if (!is_dc && !close_here) {
          // SPLIT (or a lone pass 1 never happens without close_here in TF32): nothing to publish
        } else if (!is_dc) {
          if (et == 0) wait_zero_fill();
          named_bar_sync(1, kEpiThreads);
          // value-returning atomics: when the old value is back the add has been performed at the L2, so
          // the barrier arrival below needs no device-wide fence behind 256 outstanding reductions
          if (ovalid) {
            const float old = atomicAdd(p.rowsum + orow, rs_acc);
            asm volatile("" ::"f"(old));
          }
          // value-returning atomics: when the old value is back the add has been performed at the L2, so the
          // release below needs one fence, not one per thread
          named_bar_sync(1, kEpiThreads);
          if (et == 0) {
            bool last = false;
            if (tile_valid) {
              __threadfence();
              last = atomicAdd(p.seg_done + ot, s1 - s0) + (s1 - s0) == p.ST[SEG_DE];
              if (last) { __threadfence(); atomicAdd(p.ctr + 2, 1); }
            }
            tail->flag = last;
          }
          named_bar_sync(1, kEpiThreads);
          if (tail->flag != 0) {      // CTA-uniform; tail->flag is rewritten after the flush's barrier only
            __threadfence();          // acquire: every other segment's row sums of this tile are visible
            if (et < kTile && ot * kTile + et < p.n_own[SEG_DE]) close_row(ot * kTile + et);
          }
          if (DBG && wk.kind == SEG_DE && wk.gp >= wk.end) tr.put(kTraceEvents - 3, globaltimer_ns());   // pass 1 out
        } else if (ovalid) {
          if (RG && kSplit) dw_acc += dw_seg * (exp2f(static_cast<float>(-lift2)) * gamma);
          else dw_acc += kSplit ? dw_seg * exp2f(static_cast<float>(-lift2)) : dw_seg;
        }
        // drain the accumulator [128 x D] of this segment (columns split between the two halves)
        mbar_wait(bar(BAR_ACC_FULL), sg & 1);
        tc_fence_after();
        tr.mark();   // accumulator complete
        // TMEM -> registers -> owner area of shared memory (free: every MMA1 of the segment has
        // completed) in the 128B-swizzled slab layout -> one TMA store per 32-column slab.  A range
        // that covers the whole owner group stores, a partial range adds into the zeroed output
        // (cp.reduce.async.bulk: the fp32 add happens at the L2).  Rows past n_own are clipped.
        fence_proxy_async_smem();
        const int ch0 = half ? kslabs / 2 : 0, ch1 = half ? kslabs : kslabs / 2;
        for (int ch = ch0; ch < ch1; ++ch) {
          uint32_t v[32];
          tmem_ld32(tmem + lane_addr + 2 * kUnit + ch * 32, v);
          tmem_ld_wait();
          if (kSplit && is_dc) {       // the G planes carried p * 2^lift2: dC_hat = w g 2^-lift2 (.)  (RG: w gamma)
            const float fs = (RG ? wg * gamma : wg) * exp2f(static_cast<float>(-lift2));
#pragma unroll
            for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * fs);
          }
          const uint32_t row_smem = a_smem + ch * kSlabBytes + trow * 128;
#pragma unroll
          for (int c = 0; c < 8; ++c)
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row_smem + ((c ^ (trow & 7)) << 4)),
                         "r"(v[4 * c]), "r"(v[4 * c + 1]), "r"(v[4 * c + 2]), "r"(v[4 * c + 3])
                         : "memory");
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) arrive_leader(acc_empty);
        tr.mark();   // accumulator drained into shared memory
        fence_proxy_async_smem();
        named_bar_sync(1, kEpiThreads);
        if (et == 0) {
          // one bulk group per slab: slab k goes back to the TMA warp (next owner tile) as soon as ITS store
          // has read it, so the reload of the owner area interleaves with the flush instead of following it
          if (tile_valid) {
            const CUtensorMap* tm_out = &tms.out[kind];
            int row0 = ot * kTile;
            bool store = full;
            if (is_dc && p.peer_rows > 0) {
              // the owner rank zero-filled its rows before the cross-rank barrier in front of this kernel;
              // every rank adds (fp32 add at the owner's L2 -- over NVLink for the other ranks)
              const int r = row0 / p.peer_rows;
              tm_out = &tms.out_peer[r];
              row0 -= r * p.peer_rows;
              store = false;
            } else if (!full) {
              wait_zero_fill();
            }
            for (int ks = 0; ks < kslabs; ++ks) {
              if (store) tma_store_2d(tm_out, ks * kSlabCols, row0, a_smem + ks * kSlabBytes);
              else tma_reduce_add_2d(tm_out, ks * kSlabCols, row0, a_smem + ks * kSlabBytes);
              tma_store_commit();
            }
          }
          for (int ks = 0; ks < kslabs; ++ks) {
            if (tile_valid) tma_store_wait_read_pending(kslabs - 1 - ks);
            mbar_arrive(bar(BAR_A_FREE + ks));
          }
        }
      }
      tr.mark();   // segment flushed
    }
    if (kBwd && !close_here && !closed) close_rows();     // no pass-2 segment in this cluster (or pass 1 alone)
    if (DBG && kBwd) tr.put(kTraceEvents - 1, ready_wait_ns);

    // ------------------------------------------------------------ scalar reductions (once per CTA)
    if (!kBwd) {
      loss_acc = warp_sum(loss_acc);
      if (lane == 0) tail->red[ew] = loss_acc;
      named_bar_sync(1, kEpiThreads);
      if (ew == 0 && lane == 0) {
        float t = 0.f;
        for (int i = 0; i < kEpiWarps; ++i) t += tail->red[i];
        atomicAdd(p.loss_accum, t);
      }
    } else {
      loss_acc = warp_sum(loss_acc);
      dw_acc = warp_sum(dw_acc) * g;
      db_acc = warp_sum(db_acc) * g;
      if (lane == 0) { tail->red3[ew] = loss_acc; tail->red3[kEpiWarps + ew] = dw_acc; tail->red3[2 * kEpiWarps + ew] = db_acc; }
      named_bar_sync(1, kEpiThreads);
      if (et == 0) {
        float tl = 0.f, tw = 0.f, tb = 0.f;
        for (int i = 0; i < kEpiWarps; ++i) {
          tl += tail->red3[i]; tw += tail->red3[kEpiWarps + i]; tb += tail->red3[2 * kEpiWarps + i];
        }
        if (close_here) atomicAdd(p.loss_accum, tl);
        if (p.phases & PASS_CENTROIDS) { atomicAdd(p.dwdb + 0, tw); atomicAdd(p.dwdb + 1, tb); }
        if (p.stamps != nullptr) p.stamps[2 * blockIdx.x + 1] = globaltimer_ns();
        // last CTA out restores the counters: every other CTA has counted its pass-1 units and read the tile
        // counters for the last time before its own arrival here
        const bool last_out = atomicAdd(p.ctr + 1, 1) == static_cast<int>(gridDim.x) - 1;
        if (last_out) { atomicExch(p.ctr, 0); atomicExch(p.ctr + 1, 0); atomicExch(p.ctr + 2, 0); }
        tail->flag = last_out;
      }
      named_bar_sync(1, kEpiThreads);
      if (close_here && tail->flag != 0)
        for (int t = et; t < p.OT[SEG_DE]; t += kEpiThreads) p.seg_done[t] = 0;
    }
  }

  // ------------------------------------------------------------------------- teardown
  tc_fence_before();
  __syncthreads();
  if (CG > 1) cluster_sync_all();     // no CTA leaves while its peer may still arrive on it / read its smem
  if (warp == 2) {
    if (CG == 1) tmem_dealloc<512>(tmem); else tmem_dealloc_2cta<512>(tmem);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (fn == nullptr) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(ptr);
  }
  return fn;
}

// Encoding a tensor map is a driver call (~2 us); a step needs ten of them and training loops come
// back with the same buffers (caching allocators), so the last few encodings are kept per thread.
struct MapKey {
  const void* base; int rows, D, box, dims;
  bool operator==(const MapKey& o) const {
    return base == o.base && rows == o.rows && D == o.D && box == o.box && dims == o.dims;
  }
};
constexpr int kMapCache = 32;
struct MapCache { MapKey key[kMapCache]; CUtensorMap map[kMapCache]; int next = 0, used = 0; };
thread_local MapCache g_maps;

bool map_lookup(const MapKey& k, CUtensorMap* m) {
  for (int i = 0; i < g_maps.used; ++i)
    if (g_maps.key[i] == k) { *m = g_maps.map[i]; return true; }
  return false;
}
void map_store(const MapKey& k, const CUtensorMap& m) {
  g_maps.key[g_maps.next] = k;
  g_maps.map[g_maps.next] = m;
  g_maps.next = (g_maps.next + 1) % kMapCache;
  g_maps.used = std::min(g_maps.used + 1, kMapCache);
}

// 2-D map over X[rows, D] fp32: box = [box_rows][32 cols], 128-byte swizzle (K-major slabs).
int make_map_2d(CUtensorMap* m, const float* base, int rows, int D, int box_rows) {
  const MapKey key{base, rows, D, box_rows, 2};
  if (map_lookup(key, m)) return GE2E_OK;
  auto enc = get_encode();
  if (enc == nullptr) return GE2E_ERR_LAUNCH;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(D) * 4};
  cuuint32_t box[2] = {kSlabCols, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_SUCCESS) map_store(key, *m);
  return r == CUDA_SUCCESS ? GE2E_OK : GE2E_ERR_LAUNCH;
}

// 3-D map over the same X viewed as [D/32][rows][32]: box = [box_slabs][32 rows][32 cols]
// (MN-major operand chunks for MMA2: 32 k-rows x D columns per ring stage).  32-bit MN-major
// operands must use the 32-byte-atom flavour of the 128B swizzle (UMMA SWIZZLE_128B_BASE32B).
int make_map_3d(CUtensorMap* m, const float* base, int rows, int D, int box_slabs) {
  const MapKey key{base, rows, D, box_slabs, 3};
  if (map_lookup(key, m)) return GE2E_OK;
  auto enc = get_encode();
  if (enc == nullptr) return GE2E_ERR_LAUNCH;
  cuuint64_t dims[3] = {kSlabCols, static_cast<cuuint64_t>(rows), static_cast<cuuint64_t>(D / kSlabCols)};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(D) * 4, kSlabCols * 4};
  cuuint32_t box[3] = {kSlabCols, kMma2Rows, static_cast<cuuint32_t>(box_slabs)};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_SUCCESS) map_store(key, *m);
  return r == CUDA_SUCCESS ? GE2E_OK : GE2E_ERR_LAUNCH;
}

// SPLIT operands: X as fp16 planes [rows][2][D] (a row's hi plane, then its lo plane, in the bytes of the fp32 row).
// 3-D map {D, rows, plane}: box = [1][box_rows][64 cols] = one K-major slab of one plane, 128-byte swizzle.
int make_map_h3(CUtensorMap* m, const void* base, int rows, int D, int box_rows) {
  const MapKey key{base, rows, D, box_rows, 15};
  if (map_lookup(key, m)) return GE2E_OK;
  auto enc = get_encode();
  if (enc == nullptr) return GE2E_ERR_LAUNCH;
  cuuint64_t dims[3] = {static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(rows), 2};
  cuuint64_t strides[2] = {static_cast<cuuint64_t>(D) * 4, static_cast<cuuint64_t>(D) * 2};
  cuuint32_t box[3] = {64, static_cast<cuuint32_t>(box_rows), 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_SUCCESS) map_store(key, *m);
  return r == CUDA_SUCCESS ? GE2E_OK : GE2E_ERR_LAUNCH;
}
// 4-D map {64, rows, D/64, plane}: box = [2 planes][box_chunks][32 rows][64 cols] (MN-major operand of MMA2:
// 32 k-rows x this CTA's columns, both planes, per ring stage); fp16 MN-major takes the plain 128B swizzle.
int make_map_h4(CUtensorMap* m, const void* base, int rows, int D, int box_chunks, int planes) {
  const int box_rows = planes == 1 ? 64 : kMma2Rows;      // see kM2 in the kernel
  const MapKey key{base, rows, D, box_chunks, 12 + planes};
  if (map_lookup(key, m)) return GE2E_OK;
  auto enc = get_encode();
  if (enc == nullptr) return GE2E_ERR_LAUNCH;
  cuuint64_t dims[4] = {64, static_cast<cuuint64_t>(rows), static_cast<cuuint64_t>(D / 64), 2};
  cuuint64_t strides[3] = {static_cast<cuuint64_t>(D) * 4, 128, static_cast<cuuint64_t>(D) * 2};
  cuuint32_t box[4] = {64, static_cast<cuuint32_t>(box_rows), static_cast<cuuint32_t>(box_chunks),
                       static_cast<cuuint32_t>(planes)};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_SUCCESS) map_store(key, *m);
  return r == CUDA_SUCCESS ? GE2E_OK : GE2E_ERR_LAUNCH;
}

// HYB operand copies: X as ONE compact fp16 matrix [rows][D]; box = [box_rows][64 cols], 128-byte swizzle.
int make_map_h2(CUtensorMap* m, const void* base, int rows, int D, int box_rows) {
  const MapKey key{base, rows, D, box_rows, 16};
  if (map_lookup(key, m)) return GE2E_OK;
  auto enc = get_encode();
  if (enc == nullptr) return GE2E_ERR_LAUNCH;
  cuuint64_t dims[2] = {static_cast<cuuint64_t>(D), static_cast<cuuint64_t>(rows)};
  cuuint64_t strides[1] = {static_cast<cuuint64_t>(D) * 2};
  cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r == CUDA_SUCCESS) map_store(key, *m);
  return r == CUDA_SUCCESS ? GE2E_OK : GE2E_ERR_LAUNCH;
}

// fp32 -> fp16 copies of the two operand matrices (HYB), one launch between prep / the exchange and the step kernel
__global__ void __launch_bounds__(256)
to_f16_kernel(const float4* __restrict__ a, uint2* __restrict__ a16, long long na4, const float4* __restrict__ b,
              uint2* __restrict__ b16, long long nb4) {
  pdl_wait();
  pdl_trigger();
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < na4 + nb4; i += stride) {
    const float4 v = (i < na4) ? __ldcg(a + i) : __ldcg(b + (i - na4));
    const __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
    uint2 o;
    o.x = *reinterpret_cast<const uint32_t*>(&h0); o.y = *reinterpret_cast<const uint32_t*>(&h1);
    if (i < na4) a16[i] = o; else b16[i - na4] = o;
  }
}

int g_hybrid_mode = 0;                   // 0 = where it was measured faster, 1 = every supported shape, -1 = never

unsigned long long* g_trace = nullptr;   // set through tc_set_trace (debug only)
int g_trace_mode = -1;                   // -1: every kernel, else only TC_FWD / TC_STEP
int g_trace_fine = 0;                    // 8: per-stage marks in the MMA warp's trace
unsigned long long* g_stamps = nullptr;  // set through tc_set_stamps: per-CTA {start, end} of the step kernel

// SM count and co-resident cluster count are properties of the CURRENT device: cached per device
constexpr int kMaxDevices = 64;
int current_device() {
  int dev = 0;
  cudaGetDevice(&dev);
  return dev;
}

int sm_count() {
  static int n[kMaxDevices] = {0};
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices) return 148;
  if (n[dev] == 0) {
    cudaDeviceGetAttribute(&n[dev], cudaDevAttrMultiProcessorCount, dev);
    if (n[dev] <= 0) n[dev] = 148;
  }
  return n[dev];
}

// CTA-pair mode (cta_group::2) needs an even number of 32-column chunks of D so that an MMA2 stage
// splits evenly between the two CTAs.
int pick_cg(int D) { return ((D / kSlabCols) % 2 != 0) ? 1 : 2; }

// How many clusters of size CG can be co-resident (1 CTA per SM: the kernel needs ~225 KB smem).
// The step kernel's readiness polls rely on this number: every CTA of its grid must be resident.
template <int MODE, int VARIANT, int CG>
int max_clusters() {
  constexpr bool DBG = false;
  static int cache[kMaxDevices] = {0};
  const int dev = current_device();
  const bool cacheable = dev >= 0 && dev < kMaxDevices;
  if (cacheable && cache[dev] != 0) return cache[dev];
  int n = 0;
  {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(sm_count() / CG * CG);
    cfg.blockDim = dim3(kThreadsTc);
    cfg.dynamicSmemBytes = kSmemBytes;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = CG; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    // same block size, shared memory and cluster shape in every precision: the TF32 instantiation answers for all
    cudaFuncSetAttribute(tc_strip_kernel<MODE, VARIANT, CG, PREC_TF32, DBG>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         (int)kSmemBytes);
    if (cudaOccupancyMaxActiveClusters(&n, tc_strip_kernel<MODE, VARIANT, CG, PREC_TF32, DBG>, &cfg) != cudaSuccess) n = 0;
    (void)cudaGetLastError();
  }
  if (n <= 0) return 0;        // not cached: the caller reports GE2E_ERR_LAUNCH
  n = std::min(n, kMaxClusters);
  if (cacheable) cache[dev] = n;
  return n;
}

struct Layout {
  int OT, ST, CG, OG, NC, maxseg;
  long long GP;
  size_t done_bytes, part_bytes;
  bool whole;       // every cluster's range is a whole number of owner groups: no partial flushes
};

Layout make_layout(int n_own, int n_str, int cg, int max_cl) {
  Layout L{};
  L.OT = (n_own + kTile - 1) / kTile;
  L.ST = (n_str + kUnit - 1) / kUnit;
  L.CG = cg;
  L.OG = (L.OT + L.CG - 1) / L.CG;
  L.GP = static_cast<long long>(L.OG) * L.ST;
  L.NC = static_cast<int>(std::min<long long>(std::max(max_cl, 1), L.GP));
  const long long per = L.GP / L.NC;                 // >= 1
  L.maxseg = static_cast<int>(std::min<long long>(L.ST, L.ST / per + 2));
  L.done_bytes = (static_cast<size_t>(L.OT) * sizeof(int) + 255) & ~static_cast<size_t>(255);
  L.part_bytes = static_cast<size_t>(L.OT) * L.maxseg * kTile * sizeof(float2);
  L.whole = (L.GP % L.NC == 0) && (per % L.ST == 0);
  return L;
}

// Schedule of the step kernel (see the header comment).  A pass is `OG` owner groups of `ST` stream units;
// cluster c works on the contiguous pair range [out[c], out[c + 1]).  Changing owner group inside a range
// (a "straddle") costs an accumulator flush, an owner-tile load and a pipeline refill -- about kStraddle
// units of work (measured: 8-9 us against 2.7 us per unit at config 3) -- so three cuts compete on the load
// of the busiest cluster:
//   whole     whole groups per cluster (plain stores, nothing to zero-fill)
//   assigned  OG <= clusters: every cluster belongs to ONE group, whose units are split over its clusters
//   flat      equal contiguous ranges of the flat pair list; ranges straddle groups
// `delay[c]` (units, nullable) is how much later than the others cluster c can start this pass (pass 2: a
// cluster that finishes pass 1 last flushes AFTER the grid barrier instead of under it); the assigned and
// flat cuts hand such a cluster correspondingly fewer units.  Returns true when some group is cut.
constexpr int kStraddle = 3;
bool cut_pass(long long GP, int OG, int ST, int NC, const double* delay, int* out) {
  if (GP == 0) { for (int c = 0; c <= NC; ++c) out[c] = 0; return false; }
  const long long level = (GP + NC - 1) / NC;
  const long long cost_whole = static_cast<long long>((OG + NC - 1) / NC) * ST;
  const long long cost_flat = level + ((GP % NC == 0 && level % ST == 0) ? 0 : kStraddle);
  long long cost_assigned = LLONG_MAX;
  if (OG <= NC) {
    const int n_min = NC / OG;                          // clusters of the least served group
    cost_assigned = (ST + n_min - 1) / n_min;
  }
  // split `units` pairs starting at pair `base` over clusters [c0, c1) in proportion to K - delay[c]
  auto split = [&](int c0, int c1, long long base, long long units) {
    const int n = c1 - c0;
    double dsum = 0;
    for (int c = c0; c < c1; ++c) dsum += delay ? delay[c] : 0.0;
    const double K = (static_cast<double>(units) + dsum) / n;
    double wsum = 0, cum = 0;
    for (int c = c0; c < c1; ++c) wsum += std::max(0.25, K - (delay ? delay[c] : 0.0));
    for (int c = c0; c < c1; ++c) {
      out[c] = static_cast<int>(base + static_cast<long long>(units * (cum / wsum) + 0.5));
      cum += std::max(0.25, K - (delay ? delay[c] : 0.0));
    }
  };
  if (cost_assigned <= cost_whole && cost_assigned <= cost_flat && OG < NC) {
    for (int g = 0; g < OG; ++g) {
      const int c0 = static_cast<int>(static_cast<long long>(g) * NC / OG);
      const int c1 = static_cast<int>(static_cast<long long>(g + 1) * NC / OG);
      split(c0, c1, static_cast<long long>(g) * ST, ST);
    }
    out[NC] = static_cast<int>(GP);
    return NC > OG;
  }
  if (cost_whole <= cost_flat) {
    for (int c = 0; c <= NC; ++c) out[c] = static_cast<int>((static_cast<long long>(c) * OG / NC) * ST);
    return false;
  }
  split(0, NC, 0, GP);
  out[NC] = static_cast<int>(GP);
  return true;
}

// Model of one step-kernel launch whose pass 1 closes the rows (TF32 / HYB, both passes), in units of one stream
// unit's work.  Cluster c runs its pass-1 range first; a pass-1 segment ends `len` units (plus kStraddle when it is
// not the cluster's first) after the previous one, and the utterance tiles of its owner group are complete when
// the last segment touching them ends.  Pass 2 starts at load1[c] + kPassSwitch (accumulator drain, pass-2 owner
// tile load: what the MMA warp waits for before the first pass-2 tile) and a pass-2 unit cannot be consumed before
// its utterance tile is complete.  kPassSwitch: 6.7 us from "row sums out" to the first pass-2 tile against 2.66 us
// per stream unit at cfg3 (instrumented trace, B200 at 1000 W, profiles/r5_step_dataflow).
constexpr double kPassSwitch = 2.5;

struct StepModel {
  int NC = 0;
  double start2[kMaxClusters];    // pass-2 start of every cluster
  std::vector<double> ready;      // [STc] time utterance tile t is complete
};

void model_pass1(const int* de, int NC, int STe, int cg, int STc, StepModel* m) {
  m->NC = NC;
  m->ready.assign(STc, 0.0);
  for (int c = 0; c < NC; ++c) {
    double t = 0;
    for (long long gp = de[c]; gp < de[c + 1];) {
      const long long og = gp / STe, end = std::min<long long>(de[c + 1], (og + 1) * STe);
      t += static_cast<double>(end - gp) + (gp > de[c] ? kStraddle : 0);
      for (int k = 0; k < cg; ++k) {
        const long long tile = og * cg + k;
        if (tile < STc) m->ready[tile] = std::max(m->ready[tile], t);
      }
      gp = end;
    }
    m->start2[c] = de[c + 1] > de[c] ? t + kPassSwitch : 0.0;
  }
}

// finish time of cluster c walking pass-2 pairs [a, b) (units visited from a + rot on, wrapping in one group)
double model_finish(const StepModel& m, int c, long long a, long long b, int STc, int rot) {
  double t = m.start2[c];
  const long long n = b - a;
  for (long long i = 0; i < n; ++i) {
    long long gp = a + i + rot;
    if (gp >= b) gp -= n;
    if (i > 0 && gp / STc != (gp - 1) / STc && rot == 0) t += kStraddle;
    t = std::max(t, m.ready[gp % STc]) + 1.0;
  }
  return t;
}

// rotation that visits the last-completed tile of a one-group range last (0 when the range spans groups)
int best_rotation(const StepModel& m, long long a, long long b, int STc) {
  if (b - a < 2 || a / STc != (b - 1) / STc) return 0;
  long long late = a;
  for (long long gp = a; gp < b; ++gp)
    if (m.ready[gp % STc] >= m.ready[late % STc]) late = gp;
  return static_cast<int>((late + 1 - a) % (b - a));
}

// Pass-2 cut for a makespan target T: clusters in order take pairs while their predicted finish stays within T --
// in order for a range that spans groups, else with the last-completed tiles visited last (best_rotation).  A range
// touches at most two owner groups when a group is no shorter than the level share.
bool greedy_pass2(const StepModel& m, long long GP, int STc, double T, int* out) {
  const int NC = m.NC;
  const long long level = (GP + NC - 1) / NC;
  long long gp = 0;
  for (int c = 0; c < NC; ++c) {
    out[c] = static_cast<int>(gp);
    double late = -1, t_in = m.start2[c];
    long long n = 0, nlate = 0;
    bool crossed = false;
    while (gp < GP) {
      const bool cross = n > 0 && gp % STc == 0;
      if (cross && STc >= level && crossed) break;    // a third group
      const double r = m.ready[gp % STc];
      const double t1 = std::max(t_in + (cross ? kStraddle : 0), r) + 1.0;
      const double l = std::max(late, r);
      const long long nl = (r > late) ? 1 : nlate + (r == late ? 1 : 0);
      const double est = (crossed || cross) ? t1 : std::max(m.start2[c] + static_cast<double>(n + 1), l + nl);
      if (est > T) break;
      crossed = crossed || cross; t_in = t1; late = l; nlate = nl; ++n; ++gp;
    }
  }
  out[NC] = static_cast<int>(GP);
  return gp == GP;
}

double model_makespan(const StepModel& m, const int* dc, int STc, const unsigned char* rot, double* finish) {
  double worst = 0;
  for (int c = 0; c < m.NC; ++c) {
    const double f = std::max(m.start2[c], model_finish(m, c, dc[c], dc[c + 1], STc, rot[c]));
    if (finish != nullptr) finish[c] = f;
    worst = std::max(worst, f);
  }
  return worst;
}

// the barrier version's schedule: pass 2 cut with `delay` for the clusters that finish pass 1 within kStraddle
// units of the busiest one (they flushed after the barrier instead of under it)
bool cut_pass2_barrier(const int* de, int NC, long long GPe, long long GPc, int OGc, int STc, int* dc) {
  double delay[kMaxClusters];
  long long busiest = 0;
  for (int c = 0; c < NC; ++c) busiest = std::max<long long>(busiest, de[c + 1] - de[c]);
  for (int c = 0; c < NC; ++c) {
    const long long load = de[c + 1] - de[c];
    delay[c] = (GPe > 0 && load > 0) ? std::max<double>(0.0, kStraddle - static_cast<double>(busiest - load)) : 0.0;
  }
  return cut_pass(GPc, OGc, STc, NC, GPe > 0 ? delay : nullptr, dc);
}

struct SchedKey {
  int OGe, STe, OGc, STc, phases, max_cl, cg, rows_closed;
  bool operator==(const SchedKey& o) const {
    return OGe == o.OGe && STe == o.STe && OGc == o.OGc && STc == o.STc && phases == o.phases &&
           max_cl == o.max_cl && cg == o.cg && rows_closed == o.rows_closed;
  }
};
struct SchedEntry { SchedKey key; StepSched S; int NC; bool dep, dcp; };
thread_local SchedEntry g_sched[4];
thread_local int g_sched_used = 0, g_sched_next = 0;

// rows_closed: pass 1 closes the rows in the launch (TF32 / HYB) -- pass 2 waits per utterance tile, and the
// pass-2 cut follows the model above; otherwise (SPLIT, rows closed by the forward kernel) the cut of the
// barrier version is kept.  model_finish (nullable): the model's per-cluster finish times of the result.
int make_step_sched(int OGe, int STe, int OGc, int STc, int phases, int max_cl, int cg, bool rows_closed,
                    StepSched* S, bool* de_partial, bool* dc_partial, double* model_out = nullptr,
                    double* barrier_makespan = nullptr) {
  const SchedKey key{OGe, STe, OGc, STc, phases, max_cl, cg, rows_closed ? 1 : 0};
  if (model_out == nullptr && barrier_makespan == nullptr)
    for (int i = 0; i < g_sched_used; ++i)
      if (g_sched[i].key == key) {
        *S = g_sched[i].S; *de_partial = g_sched[i].dep; *dc_partial = g_sched[i].dcp;
        return g_sched[i].NC;
      }
  const long long GPe = (phases & PASS_ROWS) ? static_cast<long long>(OGe) * STe : 0;
  const long long GPc = (phases & PASS_CENTROIDS) ? static_cast<long long>(OGc) * STc : 0;
  const int NC = static_cast<int>(std::max<long long>(1, std::min<long long>(max_cl, std::max(GPe, GPc))));
  std::memset(S->dc_rot, 0, sizeof(S->dc_rot));
  *de_partial = cut_pass(GPe, OGe, STe, NC, nullptr, S->de);
  const bool both = phases == (PASS_ROWS | PASS_CENTROIDS);
  *dc_partial = cut_pass2_barrier(S->de, NC, both ? GPe : 0, GPc, OGc, STc, S->dc);
  // The model cut costs ~24 greedy passes over the pair list (46 us of host time at cfg3, 4 ms at cfg4 when every
  // cluster carries ~443 units a pass); past 64 units per cluster the transition and the readiness waits are a few
  // percent of a pass at most, and the barrier version's cut is walked without the barrier.
  if (both && rows_closed) {
    StepModel m;
    model_pass1(S->de, NC, STe, cg, STc, &m);
    if (barrier_makespan != nullptr) {
      // the barrier version: pass 2 of cluster c started at max(busiest pass 1, its own + kPassSwitch)
      StepModel mb = m;
      double p1 = 0;
      for (int c = 0; c < NC; ++c) p1 = std::max(p1, mb.start2[c] - kPassSwitch);
      for (int c = 0; c < NC; ++c) mb.start2[c] = std::max(p1, mb.start2[c]);
      std::fill(mb.ready.begin(), mb.ready.end(), 0.0);
      *barrier_makespan = model_makespan(mb, S->dc, STc, S->dc_rot, nullptr);
    }
    // candidate 1: the barrier version's cut, walked in order without the barrier
    double best = model_makespan(m, S->dc, STc, S->dc_rot, nullptr);
    // candidate 2: the smallest makespan target the greedy cut meets (bisection)
    int cand[kMaxClusters + 1];
    unsigned char rot[kMaxClusters];
    double lo = 0, hi = best;
    for (int c = 0; c < NC; ++c) lo = std::max(lo, std::min(m.start2[c], hi));
    lo = std::max(lo, static_cast<double>(GPc) / NC);
    const bool small = GPc <= 64LL * NC;
    for (int iter = 0; small && iter < 24 && hi - lo > 0.02; ++iter) {
      const double mid = 0.5 * (lo + hi);
      if (greedy_pass2(m, GPc, STc, mid, cand)) hi = mid; else lo = mid;
    }
    if (small && greedy_pass2(m, GPc, STc, hi, cand)) {
      for (int c = 0; c < NC; ++c) rot[c] = static_cast<unsigned char>(std::min(255, best_rotation(m, cand[c], cand[c + 1], STc)));
      for (int c = 0; c < NC; ++c)
        if (cand[c + 1] - cand[c] > 255) rot[c] = 0;
      const double got = model_makespan(m, cand, STc, rot, nullptr);
      if (got < best) {
        best = got;
        std::memcpy(S->dc, cand, sizeof(int) * (NC + 1));
        std::memcpy(S->dc_rot, rot, sizeof(rot[0]) * NC);
        *dc_partial = false;
        for (int c = 0; c <= NC; ++c) *dc_partial |= (S->dc[c] % STc) != 0;
      }
    }
    if (model_out != nullptr) model_makespan(m, S->dc, STc, S->dc_rot, model_out);
  }
  SchedEntry& e = g_sched[g_sched_next];
  e.key = key; e.S = *S; e.NC = NC; e.dep = *de_partial; e.dcp = *dc_partial;
  g_sched_next = (g_sched_next + 1) % 4;
  g_sched_used = std::min(g_sched_used + 1, 4);
  return NC;
}

template <int MODE, int VARIANT, int CG, int PREC, bool DBG, bool RG = false>
int launch_tc_impl(const TmSet& tms, const StepSched& sched, const TcParams& p, int NC, bool pdl, cudaStream_t st) {
  auto kern = tc_strip_kernel<MODE, VARIANT, CG, PREC, DBG, RG>;
  static bool attr_set[kMaxDevices] = {false};    // per instantiation and device
  const int dev = current_device();
  if (dev < 0 || dev >= kMaxDevices || !attr_set[dev]) {
    GE2E_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytesT<RG>));
    if (dev >= 0 && dev < kMaxDevices) attr_set[dev] = true;
  }
  TcParams q = p;
  q.trace = (g_trace_mode < 0 || g_trace_mode == MODE) ? g_trace : nullptr;
  q.dbg = g_trace_fine;
  q.stamps = (MODE == TC_STEP) ? g_stamps : nullptr;
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(NC * CG);
  cfg.blockDim = dim3(kThreadsTc);
  cfg.dynamicSmemBytes = kSmemBytesT<RG>;
  cfg.stream = st;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = CG; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at; cfg.numAttrs = pdl ? 2 : 1;
  GE2E_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, tms, sched, q));
  GE2E_LAUNCHED();
  return GE2E_OK;
}

// the instrumented instantiation runs only while a trace buffer is set (ge2e_b200_debug_trace)
template <int MODE, int VARIANT, int CG>
int launch_tc(const TmSet& tms, const StepSched& sched, const TcParams& p, int NC, bool pdl, cudaStream_t st) {
  if (g_trace != nullptr) return launch_tc_impl<MODE, VARIANT, CG, PREC_TF32, true>(tms, sched, p, NC, pdl, st);
  return launch_tc_impl<MODE, VARIANT, CG, PREC_TF32, false>(tms, sched, p, NC, pdl, st);
}
// fp16 operand planes (prec = PREC_SPLIT / PREC_F16): softmax, CTA pairs (D = 128 or 256), no instrumented twin
template <int MODE>
int launch_tc_split(int prec, const TmSet& tms, const StepSched& sched, const TcParams& p, int NC, bool pdl, cudaStream_t st) {
  if (prec == PREC_F16) {
    if (MODE == TC_STEP && g_trace != nullptr)      // instrumented twin of the step kernel (ge2e_b200_debug_trace)
      return launch_tc_impl<MODE, GE2E_SOFTMAX, 2, PREC_F16, true>(tms, sched, p, NC, pdl, st);
    return launch_tc_impl<MODE, GE2E_SOFTMAX, 2, PREC_F16, false>(tms, sched, p, NC, pdl, st);
  }
  return launch_tc_impl<MODE, GE2E_SOFTMAX, 2, PREC_SPLIT, false>(tms, sched, p, NC, pdl, st);
}

template <int MODE, int VARIANT>
int max_clusters_cg(int cg) {
  return cg == 2 ? max_clusters<MODE, VARIANT, 2>() : max_clusters<MODE, VARIANT, 1>();
}
template <int MODE, int VARIANT>
int launch_tc_cg(int cg, const TmSet& tms, const StepSched& sched, const TcParams& p, int NC, bool pdl,
                 cudaStream_t st) {
  return cg == 2 ? launch_tc<MODE, VARIANT, 2>(tms, sched, p, NC, pdl, st)
                 : launch_tc<MODE, VARIANT, 1>(tms, sched, p, NC, pdl, st);
}

void fill_common(TcParams& p, const RowsArgs& a) {
  p.D = a.D; p.kslabs = a.D / kSlabCols; p.oslabs = p.kslabs; p.M = a.M; p.spk_offset = a.spk_offset;
  p.cos_diag = a.cos_diag; p.w = a.w; p.b = a.b; p.eps = a.eps;
}

Layout fwd_layout(int U, int n_total, int D, int variant) {
  const int cg = pick_cg(D);
  const int mc = (variant == GE2E_SOFTMAX) ? max_clusters_cg<TC_FWD, GE2E_SOFTMAX>(cg)
                                           : max_clusters_cg<TC_FWD, GE2E_CONTRAST>(cg);
  return make_layout(U, n_total, cg, mc > 0 ? mc : sm_count() / cg);
}

size_t rowsum_bytes(int U) { return (static_cast<size_t>((U + 3) & ~3) * sizeof(float) + 255) & ~static_cast<size_t>(255); }

}  // namespace

void tc_set_trace(unsigned long long* device_buf, int mode) {
  g_trace = device_buf;
  g_trace_fine = (mode >= 0 && (mode & 0x100)) ? 8 : 0;
  g_trace_mode = mode < 0 ? -1 : (mode & 0xff);
}
void tc_set_stamps(unsigned long long* device_buf) { g_stamps = device_buf; }

// Host-only view of the step schedule for tests: same arithmetic as tc_step, the number of
// co-resident clusters is an argument instead of an occupancy query.
int tc_debug_step_schedule(int u_local, int n_total, int cg, int max_clusters, int* de_begin, int* dc_begin,
                           int* partial, int* units) {
  if (u_local <= 0 || n_total <= 0 || (cg != 1 && cg != 2) || max_clusters <= 0 || max_clusters > kMaxClusters)
    return GE2E_ERR_ARGUMENT;
  const int OTe = (u_local + kTile - 1) / kTile, STe = (n_total + kUnit - 1) / kUnit;
  const int OTc = (n_total + kTile - 1) / kTile, STc = (u_local + kUnit - 1) / kUnit;
  StepSched S{};
  bool dep = false, dcp = false;
  const int NC = make_step_sched((OTe + cg - 1) / cg, STe, (OTc + cg - 1) / cg, STc, PASS_ROWS | PASS_CENTROIDS,
                                 max_clusters, cg, true, &S, &dep, &dcp);
  for (int c = 0; c <= NC; ++c) { de_begin[c] = S.de[c]; dc_begin[c] = S.dc[c]; }
  partial[0] = dep ? 1 : 0; partial[1] = dcp ? 1 : 0;
  units[0] = (OTe + cg - 1) / cg; units[1] = STe; units[2] = (OTc + cg - 1) / cg; units[3] = STc;
  return NC;
}

int tc_debug_step_model(int u_local, int n_total, int cg, int max_clusters, int* dc_rot, double* finish,
                        double* model) {
  if (u_local <= 0 || n_total <= 0 || (cg != 1 && cg != 2) || max_clusters <= 0 || max_clusters > kMaxClusters)
    return GE2E_ERR_ARGUMENT;
  const int OTe = (u_local + kTile - 1) / kTile, STe = (n_total + kUnit - 1) / kUnit;
  const int OTc = (n_total + kTile - 1) / kTile, STc = (u_local + kUnit - 1) / kUnit;
  StepSched S{};
  bool dep = false, dcp = false;
  const int NC = make_step_sched((OTe + cg - 1) / cg, STe, (OTc + cg - 1) / cg, STc, PASS_ROWS | PASS_CENTROIDS,
                                 max_clusters, cg, true, &S, &dep, &dcp, finish, &model[1]);
  for (int c = 0; c < NC; ++c) dc_rot[c] = S.dc_rot[c];
  model[0] = kPassSwitch;
  return NC;
}

bool tc_supported(int n_local, int n_total, int M, int D, int variant) {
  (void)variant;
  if (D % kSlabCols != 0 || D < kSlabCols || D > kMaxSlabs * kSlabCols) return false;
  // up to 128 speakers the single-kernel SIMT step is faster (32 us at N = 128, M = 10 against 57 / 40 us here);
  // from 129 on these kernels win (N = 129..255: 57 us split / 40 us TF32 against 94..152 us on the SIMT pipeline)
  if (n_total < 129 || static_cast<long long>(n_local) * M < 256) return false;
  return get_encode() != nullptr;
}

bool tc_split_supported(int n_local, int n_total, int M, int D, int variant) {
  // softmax only (the contrast backward is a SIMT gather over fp32 operands); D = 128 / 256: prep's warp
  // kernels write the planes, and the MMA2 stage must split evenly over the CTA pair
  return variant == GE2E_SOFTMAX && (D == 128 || D == 256) && tc_supported(n_local, n_total, M, D, variant);
}

void tc_set_hybrid(int mode) { g_hybrid_mode = mode < -1 || mode > 1 ? 0 : mode; }

// GE2E_TF32, softmax step: MMA1 on fp16 copies of the operands (PREC_HYB) where the step is long enough to pay for
// the conversion launch -- from 2^26 (local utterance, speaker) pairs: config 4 and its shards, not config 3
bool tc_hybrid_selected(int n_local, int n_total, int M, int D, int variant) {
  if (g_hybrid_mode < 0 || variant != GE2E_SOFTMAX || D % 64 != 0 || !tc_supported(n_local, n_total, M, D, variant))
    return false;
  return g_hybrid_mode > 0 || static_cast<long long>(n_local) * M * n_total >= (1LL << 26);
}
size_t f16_copy_bytes(int rows, int D) { return (static_cast<size_t>(rows) * D * 2 + 255) & ~static_cast<size_t>(255); }

// workspace: [header 256 B: step counters][FWD seg_done][FWD seg_part][STEP row sums][HYB: e_hat, c_hat as fp16]
size_t tc_workspace_bytes(int n_local, int n_total, int M, int D, int variant) {
  const Layout L = fwd_layout(n_local * M, n_total, D, variant);
  size_t n = kWsHeaderBytes + L.done_bytes + L.part_bytes + rowsum_bytes(n_local * M);
  if (tc_hybrid_selected(n_local, n_total, M, D, variant)) n += f16_copy_bytes(n_local * M, D) + f16_copy_bytes(n_total, D);
  return n;
}

namespace {

// The forward kernel: loss and row statistics of either variant.
int tc_fwd_rows(const RowsArgs& a, const TcRowsBufs& b, void* ws, cudaStream_t st, int prec) {
  const int U = a.n_local * a.M;
  const bool split = prec != PREC_TF32;         // fp16 operand planes
  const Layout L = fwd_layout(U, a.n_total, a.D, a.variant);
  TmSet tms{};
  int rc;
  if (split) {
    if ((rc = make_map_h3(&tms.own[0], a.e_hat, U, a.D, kTile)) != GE2E_OK) return rc;
    if ((rc = make_map_h3(&tms.strk[0], a.c_hat_all, a.n_total, a.D, kBoxRows)) != GE2E_OK) return rc;
  } else {
    if ((rc = make_map_2d(&tms.own[0], a.e_hat, U, a.D, kTile)) != GE2E_OK) return rc;
    if ((rc = make_map_2d(&tms.strk[0], a.c_hat_all, a.n_total, a.D, kBoxRows)) != GE2E_OK) return rc;
  }
  TcParams p{};
  fill_common(p, a);
  if (split) p.oslabs = (prec == PREC_SPLIT ? 2 : 1) * (a.D / 64);
  p.n_own[0] = U; p.n_str[0] = a.n_total; p.OT[0] = L.OT; p.ST[0] = L.ST; p.GP = L.GP;
  p.row_stat_out = b.row_stat; p.kstar_out = b.row_kstar; p.row_aux_out = b.row_aux; p.loss_accum = b.loss_accum;
  p.per_row_out = b.per_row;
  // the workspace is zero on entry (caller's contract) and the kernel leaves it zeroed
  p.seg_done = reinterpret_cast<int*>(static_cast<uint8_t*>(ws) + kWsHeaderBytes);
  p.seg_part = reinterpret_cast<float2*>(static_cast<uint8_t*>(ws) + kWsHeaderBytes + L.done_bytes);
  p.maxseg = L.maxseg;
  // programmatic dependent launch: barrier init / TMEM allocation / tensormap prefetch run under the
  // tail of whatever kernel precedes this one in the stream; the kernel waits before touching memory
  static const StepSched no_sched{};
  if (split) return launch_tc_split<TC_FWD>(prec, tms, no_sched, p, L.NC, true, st);
  if (a.variant == GE2E_SOFTMAX)
    return launch_tc_cg<TC_FWD, GE2E_SOFTMAX>(L.CG, tms, no_sched, p, L.NC, true, st);
  return launch_tc_cg<TC_FWD, GE2E_CONTRAST>(L.CG, tms, no_sched, p, L.NC, true, st);
}

// The softmax step kernel.  phases = PASS_ROWS: forward rows + un-normalised dE_hat (+ row_scale);
// PASS_CENTROIDS: dC_hat_partial, {dw, db} from the row statistics of an earlier rows pass; both: one launch, in
// which pass 2 waits for the row sums of each utterance tile before it reads them.  TF32 / HYB: pass 1 closes the
// rows (row statistics, loss); SPLIT / F16: the forward kernel closed them, and both passes read them.
int tc_step(const RowsArgs& a, int phases, const TcRowsBufs& b, void* ws, cudaStream_t st, int prec) {
  const int U = a.n_local * a.M;
  const bool peers = b.dC_owner != nullptr && b.n_ranks > 1;
  const bool split = prec != PREC_TF32;         // fp16 operand planes
  const bool hyb = !split && tc_hybrid_selected(a.n_local, a.n_total, a.M, a.D, a.variant);
  const bool closes_rows = !split && (phases & PASS_ROWS);
  const int cg = pick_cg(a.D);
  const int slabs = a.D / kSlabCols;
  const int max_cl = max_clusters_cg<TC_STEP, GE2E_SOFTMAX>(cg);
  // pass 2 polls for row sums that other CTAs' pass 1 produces: every CTA of the grid must be co-resident
  if (max_cl <= 0) return GE2E_ERR_LAUNCH;
  // segment kind DE: owner = utterance tiles, stream = centroids; DC: owner = centroid tiles, stream = utterances
  TcParams p{};
  fill_common(p, a);
  if (split) p.oslabs = (prec == PREC_SPLIT ? 2 : 1) * (a.D / 64);
  if (hyb) p.oslabs = a.D / 64;
  p.phases = phases;
  p.grad_out = b.grad_out; p.grad_rows = b.grad_rows; p.dwdb = b.dwdb;
  if (closes_rows) {
    p.row_stat_out = b.row_stat; p.row_aux_out = b.row_aux; p.loss_accum = b.loss_accum; p.per_row_out = b.per_row;
  } else {
    p.row_stat = b.row_stat; p.row_aux = b.row_aux;
  }
  p.row_scale_out = b.row_scale;
  p.n_own[SEG_DE] = U; p.n_str[SEG_DE] = a.n_total;
  p.n_own[SEG_DC] = a.n_total; p.n_str[SEG_DC] = U;
  for (int k = 0; k < 2; ++k) {
    p.OT[k] = (p.n_own[k] + kTile - 1) / kTile;
    p.ST[k] = (p.n_str[k] + kUnit - 1) / kUnit;
  }
  StepSched sched{};
  bool de_partial = false, dc_partial = false;
  const int NC = make_step_sched((p.OT[SEG_DE] + cg - 1) / cg, p.ST[SEG_DE], (p.OT[SEG_DC] + cg - 1) / cg, p.ST[SEG_DC],
                                 phases, max_cl, cg, !split, &sched, &de_partial, &dc_partial);
  // outputs assembled from partial accumulators (TMA reduce-add) are zero-filled by the kernel itself;
  // D % 32 == 0 makes every row a whole number of float4
  if ((phases & PASS_CENTROIDS) && dc_partial && !peers) {
    p.zero_base = reinterpret_cast<float4*>(b.dC_hat_partial);
    p.zero_n4 = static_cast<long long>(a.n_total) * a.D / 4;
  }
  if ((phases & PASS_ROWS) && de_partial) {
    p.zero2_base = reinterpret_cast<float4*>(b.dE_hat);
    p.zero2_n4 = static_cast<long long>(U) * a.D / 4;
  }
  p.ctr = static_cast<int*>(ws);
  const Layout L = fwd_layout(U, a.n_total, a.D, a.variant);
  p.rowsum = reinterpret_cast<float*>(static_cast<uint8_t*>(ws) + kWsHeaderBytes + L.done_bytes + L.part_bytes);
  // per-utterance-tile pass-1 counters: the forward kernel's stream-K counters (OT = the same U rows), zero on
  // entry and exit of either kernel
  p.seg_done = reinterpret_cast<int*>(static_cast<uint8_t*>(ws) + kWsHeaderBytes);
  // {dw, db} accumulate: zeroed by prep when the passes run in one step; a lone backward clears them here
  if (phases == PASS_CENTROIDS) GE2E_CUDA_TRY(cudaMemsetAsync(b.dwdb, 0, 2 * sizeof(float), st));

  // the operands: [SEG_DE] utterances, [SEG_DC] centroids; segment k owns op[k] and streams op[1 - k]
  const float* op[2] = {a.e_hat, a.c_hat_all};
  const int op_rows[2] = {U, a.n_total};
  const void* op_k[2] = {op[0], op[1]};         // what MMA1 reads K-major
  if (hyb) {
    // fp16 copies behind the row sums in the workspace; MMA1 reads them (K-major), MMA2 the fp32 originals (MN-major)
    uint8_t* e16 = reinterpret_cast<uint8_t*>(p.rowsum) + rowsum_bytes(U);
    uint8_t* c16 = e16 + f16_copy_bytes(U, a.D);
    const long long na4 = static_cast<long long>(U) * a.D / 4, nb4 = static_cast<long long>(a.n_total) * a.D / 4;
    const long long want = (na4 + nb4 + 255) / 256;
    const unsigned blocks = static_cast<unsigned>(std::min<long long>(want, static_cast<long long>(sm_count()) * 8));
    GE2E_CUDA_TRY(launch_pdl(to_f16_kernel, dim3(blocks), dim3(256), 0, st, phases != PASS_CENTROIDS,
                             reinterpret_cast<const float4*>(a.e_hat), reinterpret_cast<uint2*>(e16), na4,
                             reinterpret_cast<const float4*>(a.c_hat_all), reinterpret_cast<uint2*>(c16), nb4));
    GE2E_LAUNCHED();
    op_k[0] = e16; op_k[1] = c16;
  }
  // only the map makers differ between the operand encodings (split planes / HYB copies / TF32)
  auto map_k = [&](CUtensorMap* m, const void* base, int rows, int box_rows) {
    if (split) return make_map_h3(m, base, rows, a.D, box_rows);
    if (hyb) return make_map_h2(m, base, rows, a.D, box_rows);
    return make_map_2d(m, static_cast<const float*>(base), rows, a.D, box_rows);
  };
  auto map_mn = [&](CUtensorMap* m, const float* base, int rows) {
    if (split) return make_map_h4(m, base, rows, a.D, a.D / 64 / cg, prec == PREC_SPLIT ? 2 : 1);
    return make_map_3d(m, base, rows, a.D, slabs / cg);
  };
  TmSet tms{};
  int rc;
  for (int k = 0; k < 2; ++k) {
    if ((rc = map_k(&tms.own[k], op_k[k], op_rows[k], kTile)) != GE2E_OK) return rc;
    if ((rc = map_k(&tms.strk[k], op_k[1 - k], op_rows[1 - k], kBoxRows)) != GE2E_OK) return rc;
    if ((rc = map_mn(&tms.strmn[k], op[1 - k], op_rows[1 - k])) != GE2E_OK) return rc;
  }
  if ((rc = make_map_2d(&tms.out[SEG_DE], b.dE_hat, U, a.D, kTile)) != GE2E_OK) return rc;
  if ((rc = make_map_2d(&tms.out[SEG_DC], b.dC_hat_partial != nullptr ? b.dC_hat_partial : b.dE_hat, a.n_total, a.D,
                        kTile)) != GE2E_OK)
    return rc;
  if (peers) {
    p.peer_rows = a.n_total / b.n_ranks;
    for (int r = 0; r < b.n_ranks; ++r) {
      if (b.dC_owner[r] == nullptr || (reinterpret_cast<uintptr_t>(b.dC_owner[r]) & 15) != 0) return GE2E_ERR_ARGUMENT;
      if ((rc = make_map_2d(&tms.out_peer[r], b.dC_owner[r], p.peer_rows, a.D, kTile)) != GE2E_OK) return rc;
    }
  }
  if (b.grad_rows != nullptr) {     // row-gradient instantiations (no instrumented twins); phases == PASS_CENTROIDS
    if (split)
      return prec == PREC_F16 ? launch_tc_impl<TC_STEP, GE2E_SOFTMAX, 2, PREC_F16, false, true>(tms, sched, p, NC, false, st)
                              : launch_tc_impl<TC_STEP, GE2E_SOFTMAX, 2, PREC_SPLIT, false, true>(tms, sched, p, NC, false, st);
    if (hyb) return launch_tc_impl<TC_STEP, GE2E_SOFTMAX, 2, PREC_HYB, false, true>(tms, sched, p, NC, true, st);
    return cg == 2 ? launch_tc_impl<TC_STEP, GE2E_SOFTMAX, 2, PREC_TF32, false, true>(tms, sched, p, NC, false, st)
                   : launch_tc_impl<TC_STEP, GE2E_SOFTMAX, 1, PREC_TF32, false, true>(tms, sched, p, NC, false, st);
  }
  if (split) return launch_tc_split<TC_STEP>(prec, tms, sched, p, NC, phases != PASS_CENTROIDS, st);
  if (hyb) {
    if (g_trace != nullptr) return launch_tc_impl<TC_STEP, GE2E_SOFTMAX, 2, PREC_HYB, true>(tms, sched, p, NC, true, st);
    return launch_tc_impl<TC_STEP, GE2E_SOFTMAX, 2, PREC_HYB, false>(tms, sched, p, NC, true, st);
  }
  return launch_tc_cg<TC_STEP, GE2E_SOFTMAX>(cg, tms, sched, p, NC, phases != PASS_CENTROIDS, st);
}

}  // namespace

int tc_rows(const RowsArgs& a, int prec, int phases, const TcRowsBufs& b, void* ws, size_t ws_bytes,
            cudaStream_t st) {
  const bool split = prec != PREC_TF32;         // fp16 operand planes
  const bool peers = b.dC_owner != nullptr && b.n_ranks > 1;
  if (split && !tc_split_supported(a.n_local, a.n_total, a.M, a.D, a.variant)) return GE2E_ERR_UNSUPPORTED;
  if (peers && (b.n_ranks > kMaxPeers || a.n_total % b.n_ranks != 0 || (a.n_total / b.n_ranks) % kTile != 0 ||
                !(phases & PASS_CENTROIDS)))
    return GE2E_ERR_UNSUPPORTED;
  // a per-row upstream gradient is known only after the forward: the centroid pass alone, on one device
  if (b.grad_rows != nullptr && (phases != PASS_CENTROIDS || peers)) return GE2E_ERR_UNSUPPORTED;
  if (ws == nullptr || ws_bytes < tc_workspace_bytes(a.n_local, a.n_total, a.M, a.D, a.variant))
    return GE2E_ERR_WORKSPACE;
  if (phases != 0 && (reinterpret_cast<uintptr_t>(ws) & 15) != 0) return GE2E_ERR_WORKSPACE;
  // the forward kernel closes the rows: alone, or on fp16 planes ahead of a step that has the rows pass (whose
  // pass 1 then forms dE_hat from probabilities that are already normalised)
  if (phases == 0 || (split && (phases & PASS_ROWS))) {
    const int rc = tc_fwd_rows(a, b, ws, st, prec);
    if (rc != GE2E_OK || phases == 0) return rc;
  }
  return tc_step(a, phases, b, ws, st, prec);
}

}  // namespace ge2e
