// K2/K3: pair scorer as a tcgen05 GEMM with a fused per-query top-k candidate filter.
//
// Reference arithmetic (models/match_head.py:160-162, evaluate_movingfashion.py:263-268):
//   x5 = last((q - g)^2),  score = softmax(x5)[1] = sigmoid(l1 - l0).
// Ranking needs only d_ij = l1 - l0 = dw.(q_i - g_j)^2 + db with dw = w1 - w0, which expands to
//   d_ij = rq_i + [ a_i . g_j + cg_j ] + db,   a_i = -2 dw (.) q_i,  rq_i = dw.q_i^2,  cg_j = dw.g_j^2.
// The bracket v_ij is what this kernel evaluates: a_i . g_j on the tensor cores (fp16 operands,
// fp32 accumulation in TMEM), + cg_j in the epilogue.  The (Q,G) matrix never leaves the SM.
//
// Candidate filter (branch-free).  Every query row keeps a lower bound thr on its 32nd best v:
// each of the row's 4 epilogue threads keeps 16 running group maxima (a group = 4 adjacent columns
// of every tile; groups are pairwise disjoint); at least 8 distinct gallery items sit at or above the
// 8th largest of a thread's 16 maxima, so the smallest of the four threads' values is such a bound --
// with about 60 items above it.  Candidates are appended to the row's lists in global memory by QUADS
// of adjacent columns: iff max(w0..w3) > thr, one predicated 16-byte store of the four values, whose
// 6 low mantissa bits carry the quad's position and the gallery tile index (see "Candidate records"
// below).  Nothing is ever pruned or re-ordered on the SM; the re-score kernel (score_exact.cuh)
// selects the best 32 of a row's lists and certifies the result.  Bounds are shared between the 4
// threads of a row through shared memory every other tile and between CTAs working on the same rows
// through global memory (atomicMax on an order-preserving integer image of the float).  To warm the
// bound before anything is appended, the segment holding a row's first gallery tile -- and whatever
// segment a CTA sweeps first -- previews a few sample tiles of its range in threshold-only mode.
//
// Work decomposition: the (query tile, gallery tile) grid is linearised query-major and cut
// into one contiguous range per CTA, balanced on the host by cost (tiles + sample tiles + segment
// starts); a range is processed as at most a few "segments" (one query tile x a run of gallery
// tiles), last segment first (segment_before).
//
// Roles (608 threads): warp 0 = TMA producer, warp 1 = MMA issuer (one lane), warp 2 = TMEM
// allocator, then stages cg tiles, warps 3..18 = epilogue (warp%4 selects the TMEM lane quarter =
// 32 query rows, (warp-3)/4 the 64-column quarter of the tile).
// Tile: 128 queries x 256 gallery rows, K = 256 as 4 k-blocks of 64 fp16 (128-byte swizzle).
// The A (query) tile stays resident in shared memory for a whole segment; B (gallery)
// k-blocks stream through a 4-stage ring; two 256-column TMEM accumulators alternate, and an
// epilogue warp hands its accumulator back as soon as its last 16-column load has landed (half-way
// through its work on the tile).
#pragma once
#include <cstdint>
#include <utility>
#include <cuda.h>
#include "sm100_ptx.cuh"

namespace seam {
namespace score {

constexpr int BM = 128, BN = 256, BK = 64, NKB = 4, NSTAGE = 4;
constexpr int CTRL_WARPS = 3, EPI_WARPS = 16;   // 608 threads, 96 registers each (warps are allocated in fours)
constexpr int THREADS = (CTRL_WARPS + EPI_WARPS) * 32;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int NQ = 4;                  // column quarters = sub-lists per (row, piece)
constexpr int QCOLS = BN / NQ;         // 64 accumulator columns per thread per tile
constexpr int HALF = 32;               // columns per tcgen05.ld
constexpr int CMD_SEED = 1, CMD_SEG_START = 2, CMD_SEG_END = 4, CMD_SEED_END = 8;
constexpr int GROUPS = 16;             // running group maxima per thread; its bound is their 8th largest
                                       // (4 threads x 8 guaranteed items = 32 per row)
constexpr uint32_t A_KB_BYTES = BM * BK * 2;
constexpr uint32_t B_ST_BYTES = BN * BK * 2;

constexpr uint32_t OFF_A = 0;
constexpr uint32_t OFF_B = OFF_A + NKB * A_KB_BYTES;
constexpr uint32_t OFF_CG = OFF_B + NSTAGE * B_ST_BYTES;
constexpr uint32_t OFF_THRX = OFF_CG + 2 * BN * 4;
constexpr uint32_t OFF_CMD = OFF_THRX + BM * NQ * 4;   // 2 x int4 tile commands
constexpr uint32_t OFF_BAR = OFF_CMD + 2 * 16;
constexpr uint32_t NUM_BARS = 2 * NSTAGE + 2 + 8;
constexpr uint32_t OFF_TMEM = OFF_BAR + NUM_BARS * 8;
constexpr uint32_t SMEM_BYTES = OFF_TMEM + 16 + 1024;   // + slack for manual 1024-byte alignment
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB per-CTA shared memory limit");
static_assert(OFF_CG % 16 == 0 && OFF_THRX % 16 == 0 && OFF_CMD % 16 == 0 && OFF_BAR % 8 == 0, "alignment");

constexpr int MAX_GRID = 160;          // one persistent CTA per SM
constexpr int VAR_RANK = 6;            // kernel variant: rank of one designated gallery item per query

// The work decomposition, cost-balanced on the host: CTA b of nb sweeps the linearised tiles [tb[b], tb[b+1]).
// A query tile's sweep is shared by consecutive CTAs, its rows' "pieces", each of which writes 4 sub-lists
// per row (count + group maxima, every call).  Slots beyond a row's pieces hold stale data from other problem
// shapes and are never looked at -- so nothing has to be reset between calls.
struct TilePlan {
  int ntiles_n, nb;
  int tb[MAX_GRID + 1];
};

// the CTA whose (non-empty) range contains tile t: the largest b with tb[b] <= t
__device__ __forceinline__ int cta_of_tile(const TilePlan& pl, long long t) {
  int lo = 0, hi = pl.nb - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if ((long long)pl.tb[mid] <= t) lo = mid;
    else hi = mid - 1;
  }
  return lo;
}
// the number of CTAs that swept query row qi's gallery tiles
__device__ __forceinline__ int pieces_of_row(const TilePlan& pl, int qi) {
  const long long r0 = (long long)(qi / BM) * pl.ntiles_n;
  return cta_of_tile(pl, r0 + pl.ntiles_n - 1) - cta_of_tile(pl, r0) + 1;
}

struct Params {
  int Q, G;
  int P;                      // sub-list slots per row: max CTAs sharing one query tile's sweep
  int CAP;                    // entries per sub-list
  int nseed;                  // threshold-only sample tiles at the start of a segment
  const float* cg;            // (G)
  uint32_t* thr_global;       // (Q) ordered-uint image of the per-row lower bound
  uint32_t* rowcnt;           // (Q, P, 4) quad records in each sub-list
  uint32_t* rowflag;          // (Q) nonzero: the row lost candidates, must be ranked exhaustively
  uint2* rowbuf;              // (Q, P, 4, CAP x 8 bytes) = CAP/2 quad records {w0,w1,w2,w3} per sub-list
  float* gmax;                // (Q, P, 4, 16) final group maxima of each thread (disjoint column groups)
  TilePlan plan;
  // rank-of-target variant (VAR_RANK): per-row band (lo, hi] around the target's value and, per sub-list,
  // the number of elements certainly above it
  const float* rank_lo;       // (Q)
  const float* rank_hi;       // (Q)
  int32_t* rank_above;        // (Q, P, 4)
};

// One segment = query tile m, gallery tiles [nt0, nt0 + n_main), preceded by n_seed sample tiles
// (threshold-only previews of tiles spread over the same range).
struct Segment {
  int m, nt0, n_main, n_seed, ntiles_n;
  __device__ __forceinline__ int count() const { return n_seed + n_main; }
  __device__ __forceinline__ int tile(int i) const {
    // sample tiles are taken from the segment's own range, so that every group maximum a thread
    // ever records belongs to a column of its own piece (pieces of a row are disjoint)
    return i < n_seed ? nt0 + (int)((unsigned)((2 * i + 1) * n_main) / (unsigned)(2 * n_seed)) : nt0 + (i - n_seed);
  }
};
// Sweep order and sampling.  The whole grid starts cold at the same moment, so a row's bound has to be
// warmed by somebody: the segment that contains the row's first gallery tile (its "head") previews
// min(nseed, n_main) sample tiles, and so does whatever segment a CTA sweeps first.  A CTA sweeps the
// segments of its range LAST FIRST: the last one is normally a head, the first one the tail of a row
// whose head is the first thing the previous CTA sweeps -- by the time this CTA gets to the tail the
// row's bound has long been published in thr_global (after the sample sweep, then every 8 tiles), and
// the tail starts warm without samples.  Every row is thus sampled once, not once per piece.
constexpr int NSEED = 4;               // sample tiles of a sampled segment (the rank variant takes none)
__device__ __forceinline__ Segment segment_before(const Params& p, long long t_begin, long long t_hi, long long t_end,
                                                  long long& next_hi) {
  Segment s;
  s.m = (int)((t_hi - 1) / p.plan.ntiles_n);
  const long long row0 = (long long)s.m * p.plan.ntiles_n;
  const long long start = max(t_begin, row0);
  s.nt0 = (int)(start - row0);
  s.n_main = (int)(t_hi - start);
  s.n_seed = (t_hi == t_end || start == row0) ? min(p.nseed, s.n_main) : 0;
  s.ntiles_n = p.plan.ntiles_n;
  next_hi = start;
  return s;
}

__device__ __forceinline__ float max3(float a, float b, float c) {
  float r;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}
__device__ __forceinline__ float min3(float a, float b, float c) {
  float r;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c));
  return r;
}

// ---- the 8th largest of 16 values -------------------------------------------------------
#define SEAM_CE_DESC(a, b)          \
  {                                 \
    const float hi_ = fmaxf(a, b);  \
    const float lo_ = fminf(a, b);  \
    a = hi_;                        \
    b = lo_;                        \
  }
// 19-comparator sorting network, descending
__device__ __forceinline__ void sort8_desc(float (&s)[8]) {
  SEAM_CE_DESC(s[0], s[1]) SEAM_CE_DESC(s[2], s[3]) SEAM_CE_DESC(s[4], s[5]) SEAM_CE_DESC(s[6], s[7])
  SEAM_CE_DESC(s[0], s[2]) SEAM_CE_DESC(s[1], s[3]) SEAM_CE_DESC(s[4], s[6]) SEAM_CE_DESC(s[5], s[7])
  SEAM_CE_DESC(s[1], s[2]) SEAM_CE_DESC(s[5], s[6]) SEAM_CE_DESC(s[0], s[4]) SEAM_CE_DESC(s[3], s[7])
  SEAM_CE_DESC(s[1], s[5]) SEAM_CE_DESC(s[2], s[6])
  SEAM_CE_DESC(s[1], s[4]) SEAM_CE_DESC(s[3], s[6])
  SEAM_CE_DESC(s[2], s[4]) SEAM_CE_DESC(s[3], s[5])
  SEAM_CE_DESC(s[3], s[4])
}
// At least 8 of the 16 values are >= the result (each is the maximum of a distinct column group,
// so 8 distinct gallery items are).  With the halves sorted descending, the k-th largest of the
// union is max over i+j=k of min(a_i, b_j) (1-based, a_0 = b_0 = +inf).
__device__ __forceinline__ float eighth_largest_of_16(const float (&gm)[16]) {
  float a[8], b[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    a[i] = gm[i];
    b[i] = gm[8 + i];
  }
  sort8_desc(a);
  sort8_desc(b);
  float r = fmaxf(a[7], b[7]);
#pragma unroll
  for (int i = 1; i <= 7; ++i) r = fmaxf(r, fminf(a[i - 1], b[7 - i]));
  return r;
}

// Candidate records.  Memory instructions are the expensive part of this epilogue (a store occupies
// its scheduler's dispatch for several cycles even when every lane is predicated off), so candidates
// are appended by QUADS of adjacent columns: one predicated 16-byte store per four accumulator elements,
//   if (max(w0..w3) > cmp) { *wp = {w0,w1,w2,w3}; wp += 16; }            (no branch)
// where w_e = (acc_e + cg_e) with the 6 low mantissa bits replaced by a tag: w0 carries the quad's
// position q (0..15) inside the thread's 64-column quarter, w1..w3 carry 18 bits of the gallery tile
// index, so a record names its four gallery rows by itself.  |w - v| <= 2^-17 |v| -- far inside the
// fp16 operand error the re-score kernel allows for (it adds the term to its eps).  w is what is
// compared and recorded as group maximum too: the whole filter is consistent in "w space".
constexpr uint32_t TAG_MASK = 63u;
constexpr int TAG_BITS = 6;
constexpr int TAG_TILES = 1 << (3 * TAG_BITS);   // gallery tiles a record can name
// The gallery column of w0 of a record read from sub-list l of its row; w1..w3 are the next three.  The
// inverse of the tagging in filter16 / filter16_rank: the sub-list gives the column quarter.
__device__ __forceinline__ uint32_t quad_first_col(const uint4& rec, int l) {
  const uint32_t tile =
      (rec.y & TAG_MASK) | ((rec.z & TAG_MASK) << TAG_BITS) | ((rec.w & TAG_MASK) << (2 * TAG_BITS));
  return tile * BN + ((uint32_t)l % NQ) * QCOLS + (rec.x & TAG_MASK) * 4u;
}
template <int Q4>
__device__ __forceinline__ float tagged_imm(uint32_t acc, float cg, uint32_t keep) {
  float w;
  asm("{\n"
      ".reg .f32 v;\n"
      "add.f32 v, %1, %2;\n"
      "lop3.b32 %0, v, %3, %4, 0xEA;\n"      // (v & keep) | Q4
      "}\n"
      : "=f"(w)
      : "f"(__uint_as_float(acc)), "f"(cg), "r"(keep), "n"(Q4));
  return w;
}
__device__ __forceinline__ float tagged_reg(uint32_t acc, float cg, uint32_t keep, uint32_t tag) {
  float w;
  asm("{\n"
      ".reg .f32 v;\n"
      "add.f32 v, %1, %2;\n"
      "lop3.b32 %0, v, %3, %4, 0xEA;\n"
      "}\n"
      : "=f"(w)
      : "f"(__uint_as_float(acc)), "f"(cg), "r"(keep), "r"(tag));
  return w;
}
// Only the low address word advances: a sub-list never straddles a 4 GiB boundary (power-of-two size,
// aligned to it).
__device__ __forceinline__ void append_quad(uint64_t& wp, float m, float cmp, float w0, float w1, float w2, float w3) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b32 lo, hi;\n"
      "setp.gt.f32 p, %1, %2;\n"
      "@p st.global.v4.f32 [%0], {%3, %4, %5, %6};\n"
      "mov.b64 {lo, hi}, %0;\n"
      "@p add.u32 lo, lo, 16;\n"
      "mov.b64 %0, {lo, hi};\n"
      "}\n"
      : "+l"(wp)
      : "f"(m), "f"(cmp), "f"(w0), "f"(w1), "f"(w2), "f"(w3)
      : "memory");
}

// ties the destination registers of an in-flight tcgen05.ld to the wait so the compiler
// cannot read them before the data has landed
__device__ __forceinline__ void tmem_ld_wait_x32(uint32_t (&a)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                 "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]),
                 "+r"(a[15]), "+r"(a[16]), "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]),
                 "+r"(a[22]), "+r"(a[23]), "+r"(a[24]), "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]),
                 "+r"(a[29]), "+r"(a[30]), "+r"(a[31])
               :
               : "memory");
}

// 16 accumulator columns of one row: + cg, tag, append the quads that beat cmp, fold the quad maxima
// into 4 of the 16 group maxima (chunk c of a tile feeds groups 4c..4c+3: a group is 4 adjacent
// columns of every tile, groups are pairwise disjoint)
struct TileTags {
  uint32_t t1, t2, t3;   // bits [0,6), [6,12), [12,18) of the gallery tile index
};
template <int GOFF, int Q0>
__device__ __forceinline__ void filter16(const uint32_t (&r)[16], const float* cgp, float (&gm)[GROUPS], uint64_t& wp,
                                         float cmp, uint32_t keep, const TileTags& tg) {
  float cgv[16];
#pragma unroll
  for (int c4 = 0; c4 < 4; ++c4) {
    const float4 g4 = *reinterpret_cast<const float4*>(cgp + c4 * 4);
    cgv[c4 * 4 + 0] = g4.x;
    cgv[c4 * 4 + 1] = g4.y;
    cgv[c4 * 4 + 2] = g4.z;
    cgv[c4 * 4 + 3] = g4.w;
  }
  // acc + cg two columns per instruction (add.rn.f32x2: the same IEEE sums, half the issue slots), then the tags
  float v[16];
#pragma unroll
  for (int e = 0; e < 16; e += 2) {
    unsigned long long s2;
    asm("{\n"
        ".reg .b64 a, b;\n"
        "mov.b64 a, {%1, %2};\n"
        "mov.b64 b, {%3, %4};\n"
        "add.rn.f32x2 %0, a, b;\n"
        "}\n"
        : "=l"(s2)
        : "r"(r[e]), "r"(r[e + 1]), "f"(cgv[e]), "f"(cgv[e + 1]));
    asm("mov.b64 {%0, %1}, %2;" : "=f"(v[e]), "=f"(v[e + 1]) : "l"(s2));
  }
  float w[16];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=f"(w[4 * q]) : "f"(v[4 * q]), "r"(keep), "r"((uint32_t)(Q0 + q)));
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=f"(w[4 * q + 1]) : "f"(v[4 * q + 1]), "r"(keep), "r"(tg.t1));
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=f"(w[4 * q + 2]) : "f"(v[4 * q + 2]), "r"(keep), "r"(tg.t2));
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=f"(w[4 * q + 3]) : "f"(v[4 * q + 3]), "r"(keep), "r"(tg.t3));
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const float m = fmaxf(max3(w[4 * q], w[4 * q + 1], w[4 * q + 2]), w[4 * q + 3]);
    gm[GOFF + q] = fmaxf(gm[GOFF + q], m);
    append_quad(wp, m, cmp, w[4 * q], w[4 * q + 1], w[4 * q + 2], w[4 * q + 3]);
  }
}

// Rank-of-target variant of the filter.  The row's band (lo, hi] brackets the target item's value by the
// error bound of this pass: an element above hi certainly ranks before the target (counted here, one
// compare + one predicated add), an element at or below lo certainly does not, and quads holding an
// element inside the band are appended for the resolve kernel to decide in exact fp32.
__device__ __forceinline__ void filter16_rank(const uint32_t (&r)[16], const float* cgp, uint64_t& wp, uint32_t& above,
                                              float lo_or_inf, float hi, uint32_t keep, const TileTags& tg,
                                              int q0) {
  float cgv[16];
#pragma unroll
  for (int c4 = 0; c4 < 4; ++c4) {
    const float4 g4 = *reinterpret_cast<const float4*>(cgp + c4 * 4);
    cgv[c4 * 4 + 0] = g4.x;
    cgv[c4 * 4 + 1] = g4.y;
    cgv[c4 * 4 + 2] = g4.z;
    cgv[c4 * 4 + 3] = g4.w;
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    float w[4], t[4];
    w[0] = tagged_reg(r[4 * q + 0], cgv[4 * q + 0], keep, (uint32_t)(q0 + q));
    w[1] = tagged_reg(r[4 * q + 1], cgv[4 * q + 1], keep, tg.t1);
    w[2] = tagged_reg(r[4 * q + 2], cgv[4 * q + 2], keep, tg.t2);
    w[3] = tagged_reg(r[4 * q + 3], cgv[4 * q + 3], keep, tg.t3);
#pragma unroll
    for (int e = 0; e < 4; ++e)
      asm("{\n"
          ".reg .pred p;\n"
          "setp.gt.f32 p, %2, %3;\n"
          "@p add.u32 %0, %0, 1;\n"
          "selp.f32 %1, 0fFF800000, %2, p;\n"      // elements above the band do not make a quad uncertain
          "}\n"
          : "+r"(above), "=f"(t[e])
          : "f"(w[e]), "f"(hi));
    const float m = fmaxf(max3(t[0], t[1], t[2]), t[3]);
    append_quad(wp, m, lo_or_inf, w[0], w[1], w[2], w[3]);
  }
}

template <int VAR>   // 0 = top-k candidate filter; VAR_RANK = rank of one designated gallery item per query
__global__ void __launch_bounds__(THREADS, 1)
score_topk_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const Params p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);

  uint8_t* sA = smem + OFF_A;
  uint8_t* sB = smem + OFF_B;
  float* cg_s = reinterpret_cast<float*>(smem + OFF_CG);        // [2][BN]
  float* thr_x = reinterpret_cast<float*>(smem + OFF_THRX);     // [BM][NQ] group-minimum of each thread
  int* cmd_s = reinterpret_cast<int*>(smem + OFF_CMD);           // [2][4] tile command of each accumulator slot
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* full = bars;                    // [NSTAGE]  TMA -> MMA
  uint64_t* empty = bars + NSTAGE;          // [NSTAGE]  MMA -> TMA
  uint64_t* a_full = bars + 2 * NSTAGE;     // A tile landed
  uint64_t* a_empty = a_full + 1;           // all MMAs of the segment retired
  uint64_t* t_full = a_empty + 1;           // [2] accumulator ready            (MMA -> epilogue)
  uint64_t* t_empty = t_full + 2;           // [2] accumulator read out         (epilogue -> MMA)
  uint64_t* cg_full = t_empty + 2;          // [2] cg tile staged               (warp 3 -> epilogue)
  uint64_t* cg_empty = cg_full + 2;         // [2] cg tile consumed             (epilogue -> warp 3)
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem + OFF_TMEM);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(ptx::FULL_MASK, tid >> 5, 0);   // provably warp-uniform role dispatch

  if (tid == 0) {
    ptx::prefetch_tensormap(&tmA);
    ptx::prefetch_tensormap(&tmB);
    for (int i = 0; i < NSTAGE; ++i) {
      ptx::mbar_init(&full[i], 1);
      ptx::mbar_init(&empty[i], 1);
    }
    ptx::mbar_init(a_full, 1);
    ptx::mbar_init(a_empty, 1);
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&t_full[i], 1);
      ptx::mbar_init(&t_empty[i], EPI_WARPS);
      ptx::mbar_init(&cg_full[i], 1);
      ptx::mbar_init(&cg_empty[i], EPI_WARPS);
    }
    ptx::fence_mbar_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc(tmem_ptr_s, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;

  long long t_begin, t_end;
  t_begin = p.plan.tb[blockIdx.x];
  t_end = p.plan.tb[blockIdx.x + 1];

  if (warp == 0) {
    // ================================================================= TMA producer
    // The whole warp walks the loop (converged), one elected lane issues: uniform-datapath instructions
    // (UTMALDG, UTCHMMA, SYNCS) inside a divergent `lane == 0` region are expanded by the compiler into
    // a per-active-lane loop of ~14 instructions each.
    {
      uint32_t stage = 0, sphase = 0, iphase = 0;
      long long t = t_end, next;
      while (t > t_begin) {
        const Segment sg = segment_before(p, t_begin, t, t_end, next);
        ptx::mbar_wait(a_empty, iphase ^ 1);
        if (ptx::elect_one()) {
          ptx::mbar_arrive_expect_tx(a_full, NKB * A_KB_BYTES);
          for (int kb = 0; kb < NKB; ++kb) ptx::tma_load_2d(sA + kb * A_KB_BYTES, &tmA, a_full, kb * BK, sg.m * BM);
        }
        __syncwarp();
        const int n = sg.count();
        for (int i = 0; i < n; ++i) {
          const int nt = sg.tile(i);
          for (int kb = 0; kb < NKB; ++kb) {
            ptx::mbar_wait(&empty[stage], sphase ^ 1);
            if (ptx::elect_one()) {
              ptx::mbar_arrive_expect_tx(&full[stage], B_ST_BYTES);
              ptx::tma_load_2d(sB + stage * B_ST_BYTES, &tmB, &full[stage], kb * BK, nt * BN);
            }
            __syncwarp();
            if (++stage == NSTAGE) {
              stage = 0;
              sphase ^= 1;
            }
          }
        }
        iphase ^= 1;
        t = next;
      }
    }
  } else if (warp == 1) {
    // ================================================================= MMA issuer (converged warp, one elected lane)
    {
      constexpr uint32_t idesc = ptx::umma_idesc(0 /*fp16*/, BM, BN);
      const uint32_t a_addr = ptx::smem_u32(sA), b_addr = ptx::smem_u32(sB);
      uint32_t stage = 0, sphase = 0, iphase = 0, acc = 0, aphase = 0;
      long long t = t_end, next;
      while (t > t_begin) {
        const Segment sg = segment_before(p, t_begin, t, t_end, next);
        const int n = sg.count();
        ptx::mbar_wait(a_full, iphase);
        for (int i = 0; i < n; ++i) {
          ptx::mbar_wait(&t_empty[acc], aphase ^ 1);
          ptx::tc_fence_after();
          const uint32_t d_tmem = tmem_base + acc * BN;
          for (int kb = 0; kb < NKB; ++kb) {
            ptx::mbar_wait(&full[stage], sphase);
            ptx::tc_fence_after();
            if (ptx::elect_one()) {
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) {
                const uint64_t ad = ptx::umma_desc_k_sw128(a_addr + kb * A_KB_BYTES + k * 32);
                const uint64_t bd = ptx::umma_desc_k_sw128(b_addr + stage * B_ST_BYTES + k * 32);
                ptx::umma_f16(d_tmem, ad, bd, idesc, (kb | k) != 0 ? 1u : 0u);
              }
              ptx::umma_commit(&empty[stage]);
              if (kb == NKB - 1) ptx::umma_commit(&t_full[acc]);
            }
            __syncwarp();
            if (++stage == NSTAGE) {
              stage = 0;
              sphase ^= 1;
            }
          }
          if (++acc == 2) {
            acc = 0;
            aphase ^= 1;
          }
        }
        if (ptx::elect_one()) ptx::umma_commit(a_empty);
        __syncwarp();
        iphase ^= 1;
        t = next;
      }
    }
  } else if (warp == 2) {
    // ================================================================= tile director (after the TMEM allocation)
    // Walks the CTA's tile sequence and, per tile, stages the cg values and a 16-byte command
    // {gallery tile | -1 = done, flags, query tile, piece} for the epilogue warps, which therefore
    // carry no segment bookkeeping of their own.
    uint32_t acc = 0, aphase = 0;
    long long t = t_end, next;
    while (t > t_begin) {
      const Segment sg = segment_before(p, t_begin, t, t_end, next);
      const int n = sg.count();
      const int piece = blockIdx.x - cta_of_tile(p.plan, (long long)sg.m * p.plan.ntiles_n);
      for (int i = 0; i < n; ++i) {
        const int nt = sg.tile(i);
        const int j0 = nt * BN + lane * 8;
        float c[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) c[e] = (j0 + e < p.G) ? __ldg(p.cg + j0 + e) : -INFINITY;   // padded columns never qualify
        ptx::mbar_wait(&cg_empty[acc], aphase ^ 1);
        float* dst = cg_s + acc * BN + lane * 8;
        *reinterpret_cast<float4*>(dst) = make_float4(c[0], c[1], c[2], c[3]);
        *reinterpret_cast<float4*>(dst + 4) = make_float4(c[4], c[5], c[6], c[7]);
        if (lane == 0) {
          const int flags = (i < sg.n_seed ? CMD_SEED : 0) | (i == 0 ? CMD_SEG_START : 0) |
                            (i == n - 1 ? CMD_SEG_END : 0) | (i + 1 == sg.n_seed ? CMD_SEED_END : 0);
          *reinterpret_cast<int4*>(cmd_s + acc * 4) = make_int4(nt, flags, sg.m, piece);
        }
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&cg_full[acc]);
        if (++acc == 2) {
          acc = 0;
          aphase ^= 1;
        }
      }
      t = next;
    }
    ptx::mbar_wait(&cg_empty[acc], aphase ^ 1);
    if (lane == 0) {
      *reinterpret_cast<int4*>(cmd_s + acc * 4) = make_int4(-1, 0, 0, 0);
      ptx::mbar_arrive(&cg_full[acc]);
    }
  } else if (warp >= CTRL_WARPS) {
    // ================================================================= epilogue
    const int ew = warp - CTRL_WARPS;
    const int lq = warp & 3;                 // TMEM lane quarter: hardware ties it to warp % 4
    const int cq = ew >> 2;                  // column quarter of the tile
    const int R = lq * 32 + lane;            // row within the CTA tile
    uint32_t acc = 0, aphase = 0;
    // per-segment state, kept small: the tile prologue below is a serial chain that all four warps
    // of a scheduler run at the same moment (they wake on the same barrier), so nothing hides it
    constexpr uint32_t ST_ROW = 1, ST_SLOT = 2, ST_CLOSED = 4, ST_LOSSY = 8;
    uint32_t st = ST_CLOSED;                 // flags | piece << 8
    int grow = 0, itile = 0;
    uint64_t wp = 0;
    uint32_t wlo_begin = 0;
    // a sub-list closes when another tile's worst case (16 quads) might not fit
    const uint32_t room = (uint32_t)p.CAP * 8u - (uint32_t)(QCOLS / 4) * 16u;
    // kept in a register (opaque to ptxas) so that the quad tag can be the LOP3's immediate operand
    const uint32_t keep = ~TAG_MASK | (uint32_t)(p.Q >> 31);
    float thr = INFINITY;                    // VAR_RANK: the band's lower edge
    float gm[GROUPS];
    float rank_hi = INFINITY;                // VAR_RANK only
    uint32_t above = 0;
    for (;;) {
      ptx::mbar_wait(&cg_full[acc], aphase);
      const int4 cmd = *reinterpret_cast<const int4*>(cmd_s + acc * 4);
      if (cmd.x < 0) break;
      if (cmd.y & CMD_SEG_START) {
        grow = cmd.z * BM + R;
        const bool row_ok = grow < p.Q;
        const bool slot_ok = row_ok && cmd.w >= 0 && cmd.w < p.P;
        const size_t li = slot_ok ? ((size_t)grow * p.P + cmd.w) * NQ + cq : 0;   // this thread's sub-list
        wp = reinterpret_cast<uint64_t>(p.rowbuf + li * (size_t)p.CAP);
        wlo_begin = (uint32_t)wp;            // only the low address word ever changes (no 4 GiB straddle)
        if constexpr (VAR == VAR_RANK) {
          thr = row_ok ? p.rank_lo[grow] : INFINITY;
          rank_hi = row_ok ? p.rank_hi[grow] : INFINITY;
          above = 0;
        } else {
          thr = row_ok ? ptx::ordered_to_float(__ldcg(p.thr_global + grow)) : INFINITY;
        }
        st = (row_ok ? ST_ROW : 0u) | (slot_ok ? ST_SLOT : (ST_CLOSED | ST_LOSSY)) | ((uint32_t)(cmd.w & 0xffff) << 8);
        itile = 0;
#pragma unroll
        for (int g = 0; g < GROUPS; ++g) gm[g] = -INFINITY;
        thr_x[R * NQ + cq] = -INFINITY;
        ptx::named_bar_sync(1, EPI_THREADS); // previous segment's bounds are gone before anyone reads
      }
      ptx::mbar_wait(&t_full[acc], aphase);
      ptx::tc_fence_after();
      // four chunks of 16 columns; the first load is issued before anything else is derived
      const uint32_t taddr = tmem_base + (uint32_t(lq * 32) << 16) + acc * BN + cq * QCOLS;
      uint32_t ra[16], rb[16];
      ptx::tmem_ld_x16(taddr, ra);
      const bool seed = (cmd.y & CMD_SEED) != 0;
      if (!seed && !(st & ST_CLOSED) && (uint32_t)wp - wlo_begin > room)   // no room for another tile:
        st |= ST_CLOSED | ST_LOSSY;                                         // the row goes to the exhaustive path
      const float cmp = (seed || (st & ST_CLOSED)) ? INFINITY : thr;
      const float* cgp = cg_s + acc * BN + cq * QCOLS;
      TileTags tg;
      tg.t1 = (uint32_t)cmd.x & TAG_MASK;
      tg.t2 = ((uint32_t)cmd.x >> TAG_BITS) & TAG_MASK;
      tg.t3 = ((uint32_t)cmd.x >> (2 * TAG_BITS)) & TAG_MASK;
      ptx::tmem_ld_wait_x16(ra);
      ptx::tmem_ld_x16(taddr + 16, rb);
      if constexpr (VAR == VAR_RANK) filter16_rank(ra, cgp, wp, above, cmp, rank_hi, keep, tg, 0);
      else filter16<0, 0>(ra, cgp, gm, wp, cmp, keep, tg);
      ptx::tmem_ld_wait_x16(rb);
      ptx::tmem_ld_x16(taddr + 32, ra);
      if constexpr (VAR == VAR_RANK) filter16_rank(rb, cgp + 16, wp, above, cmp, rank_hi, keep, tg, 4);
      else filter16<4, 4>(rb, cgp + 16, gm, wp, cmp, keep, tg);
      ptx::tmem_ld_wait_x16(ra);
      ptx::tmem_ld_x16(taddr + 48, rb);
      // The MMA of the tile after next cannot start before the slowest of the 16 warps has read its
      // columns, so the last load is waited for right away (half-way through the tile's work, the
      // scheduler's other warps fill the gap) and the slot handed back before the remaining two chunks.
      ptx::tmem_ld_wait_x16(rb);
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&t_empty[acc]);
      if constexpr (VAR == VAR_RANK) {
        filter16_rank(ra, cgp + 32, wp, above, cmp, rank_hi, keep, tg, 8);
        filter16_rank(rb, cgp + 48, wp, above, cmp, rank_hi, keep, tg, 12);
      } else {
        filter16<8, 8>(ra, cgp + 32, gm, wp, cmp, keep, tg);
        filter16<12, 12>(rb, cgp + 48, gm, wp, cmp, keep, tg);
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&cg_empty[acc]);
      // share the bound: each of the row's 4 threads vouches for 8 distinct items at or above the
      // 8th largest of its 16 group maxima (re-derived every other tile), the smallest of the four
      // values therefore for 32
      const bool seed_end = (cmd.y & CMD_SEED_END) != 0;
      if constexpr (VAR != VAR_RANK) {
        if ((itile & 1) || seed_end) {
          thr_x[R * NQ + cq] = eighth_largest_of_16(gm);
          // After the sample sweep the four warps of a row meet once, so that the first appended
          // tile already sees all four bounds; later reads may be stale (still valid bounds).
          if (seed_end) ptx::named_bar_sync(2 + lq, 4 * 32);
          const float4 o = *reinterpret_cast<const float4*>(thr_x + R * NQ);
          thr = fmaxf(thr, fminf(fminf(o.x, o.y), fminf(o.z, o.w)));
        }
        if (((itile & 7) == 7 || seed_end) && (st & ST_ROW)) {   // exchange with the other CTAs sweeping these rows
          const uint32_t old = atomicMax(p.thr_global + grow, ptx::float_to_ordered(thr));
          thr = fmaxf(thr, ptx::ordered_to_float(old));
        }
      }
      ++itile;
      // ---- segment end: publish the list length, the bound and the loss flag
      if ((cmd.y & CMD_SEG_END) && (st & ST_ROW)) {
        if (st & ST_SLOT) {
          const size_t li = ((size_t)grow * p.P + (st >> 8)) * NQ + cq;
          p.rowcnt[li] = ((uint32_t)wp - wlo_begin) >> 4;   // quads
          if constexpr (VAR == VAR_RANK) {
            p.rank_above[li] = (int32_t)above;
          } else {
            float4* gd = reinterpret_cast<float4*>(p.gmax + li * GROUPS);
            gd[0] = make_float4(gm[0], gm[1], gm[2], gm[3]);
            gd[1] = make_float4(gm[4], gm[5], gm[6], gm[7]);
            gd[2] = make_float4(gm[8], gm[9], gm[10], gm[11]);
            gd[3] = make_float4(gm[12], gm[13], gm[14], gm[15]);
          }
        }
        if (st & ST_LOSSY) atomicOr(p.rowflag + grow, 1u);
        if constexpr (VAR != VAR_RANK) atomicMax(p.thr_global + grow, ptx::float_to_ordered(thr));
      }
      if (++acc == 2) {
        acc = 0;
        aphase ^= 1;
      }
    }
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 2) ptx::tmem_dealloc(tmem_base, 512);
}

}  // namespace score
}  // namespace seam
