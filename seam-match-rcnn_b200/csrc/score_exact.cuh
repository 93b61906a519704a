// Scorer support kernels: operand preparation for the tensor-core pass, fp32 direct-form
// re-scoring + certification of the nominated candidates, the exhaustive fp32 ranking used
// for rows that cannot be certified, dense logits, rank-of-target and the shard merge.
//
// "Direct form" below always means the reference's own arithmetic, in fp32:
//   l_c = sum_k W[c][k] * (q_k - g_k)^2 + b_c   (models/match_head.py:161-162,
//   evaluate_movingfashion.py:263-264), score = softmax(l)[1] (:265-267).
#pragma once
#include <type_traits>
#include <climits>
#include <cstdint>
#include <cuda_fp16.h>
#include "exchange.cuh"
#include "fold.cuh"
#include "score_tc.cuh"
#include "sm100_ptx.cuh"
#include "warp_sort.cuh"

namespace seam {
namespace exact {

constexpr float FP16_MAX = 65504.f;
// bound on |fp16 tensor-core value - exact value| relative to ||a_i|| * max_j ||g_j||:
// two operand roundings (2^-11 each) + fp32 accumulation slack.
constexpr float EPS_COEFF = 9.9e-4f;   // 2^-10 = 9.77e-4, plus accumulation slack
constexpr float TAG_REL_ERR = 8e-6f;   // > 2^-17 = 7.63e-6: 6 mantissa bits replaced by a column tag

__device__ __forceinline__ float softmax1(float l0, float l1) {
  const float m = fmaxf(l0, l1);
  const float e0 = expf(l0 - m), e1 = expf(l1 - m);
  return e1 / (e0 + e1);
}

// this lane's slice of a 256-vector: elements [4l,4l+4) and [128+4l,128+4l+4)
struct Slice {
  float4 lo, hi;
};
__device__ __forceinline__ Slice load_slice(const float* row, int lane) {
  Slice s;
  s.lo = *reinterpret_cast<const float4*>(row + 4 * lane);
  s.hi = *reinterpret_cast<const float4*>(row + 128 + 4 * lane);
  return s;
}
// the same slice of an fp16 row: two 8-byte loads, widened exactly (every later instruction is the fp32 path's)
__device__ __forceinline__ float4 widen4(uint2 v) {
  const float2 a = __half22float2(*reinterpret_cast<const __half2*>(&v.x));
  const float2 b = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ Slice load_slice(const __half* row, int lane) {
  Slice s;
  s.lo = widen4(*reinterpret_cast<const uint2*>(row + 4 * lane));
  s.hi = widen4(*reinterpret_cast<const uint2*>(row + 128 + 4 * lane));
  return s;
}
// Packed fp32 pairs (sub/mul/fma .f32x2 = one issue slot for two IEEE fp32 operations: every kernel
// here is bound by instruction issue).  Each lane forms two partial sums per logit (even / odd
// channels of its slice) and adds them at the end.
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk2(float lo, float hi) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ float sum2(u64 v) {
  float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
  return lo + hi;
}
__device__ __forceinline__ void sqdiff_dot2(const Slice& q, const Slice& g, const Slice& w0, const Slice& w1,
                                            float& p0, float& p1) {
  u64 a0, a1, d, s;
#define SEAM_TERM2(F, X, Y, FIRST)                                                                   \
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pk2(q.F.X, q.F.Y)), "l"(pk2(g.F.X, g.F.Y)));      \
  asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(s) : "l"(d));                                               \
  if (FIRST) {                                                                                       \
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(a0) : "l"(pk2(w0.F.X, w0.F.Y)), "l"(s));                  \
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(a1) : "l"(pk2(w1.F.X, w1.F.Y)), "l"(s));                  \
  } else {                                                                                           \
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a0) : "l"(pk2(w0.F.X, w0.F.Y)), "l"(s));              \
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(a1) : "l"(pk2(w1.F.X, w1.F.Y)), "l"(s));              \
  }
  SEAM_TERM2(lo, x, y, true) SEAM_TERM2(lo, z, w, false) SEAM_TERM2(hi, x, y, false) SEAM_TERM2(hi, z, w, false)
#undef SEAM_TERM2
  p0 = sum2(a0);
  p1 = sum2(a1);
}
// both logits of one pair, all lanes get the result; Row: float or __half gallery rows
template <typename Row>
__device__ __forceinline__ void pair_logits(const Slice& q, const Row* grow, const Slice& w0, const Slice& w1,
                                            float b0, float b1, int lane, float& l0, float& l1) {
  const Slice g = load_slice(grow, lane);
  float p0, p1;
  sqdiff_dot2(q, g, w0, w1, p0, p1);
  l0 = ptx::warp_sum_b(p0) + b0;   // same association as the butterfly in rescore_kernel
  l1 = ptx::warp_sum_b(p1) + b1;
}

// ---------------------------------------------------------------- gallery preparation
// warp per gallery row: fp16 copy, cg_j = dw . g_j^2, max_j ||g_j|| (gstat[0]), overflow flag (gstat[1]).
// Row = __half: the caller's rows are the fp16 operand already -- cg and gstat only (g16 is not written).
template <typename Row>
__global__ void __launch_bounds__(256) prep_gallery_kernel(const Row* __restrict__ g, int G,
                                                           const float* __restrict__ fold, __half* __restrict__ g16,
                                                           float* __restrict__ cg, float* __restrict__ gstat) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int j = blockIdx.x * 8 + warp;
  if (j >= G) return;
  const Slice x = load_slice(g + (size_t)j * 256, lane);
  const Slice dw = load_slice(fold + Fold::DW, lane);
  const float xs[8] = {x.lo.x, x.lo.y, x.lo.z, x.lo.w, x.hi.x, x.hi.y, x.hi.z, x.hi.w};
  const float ds[8] = {dw.lo.x, dw.lo.y, dw.lo.z, dw.lo.w, dw.hi.x, dw.hi.y, dw.hi.z, dw.hi.w};
  float c = 0.f, n2 = 0.f, amax = 0.f;
  __half h[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    c = fmaf(ds[e], xs[e] * xs[e], c);
    n2 = fmaf(xs[e], xs[e], n2);
    amax = fmaxf(amax, fabsf(xs[e]));
    h[e] = __float2half_rn(xs[e]);
  }
  if constexpr (std::is_same<Row, float>::value) {
    __half* dst = g16 + (size_t)j * 256;
    *reinterpret_cast<uint2*>(dst + 4 * lane) = *reinterpret_cast<const uint2*>(&h[0]);
    *reinterpret_cast<uint2*>(dst + 128 + 4 * lane) = *reinterpret_cast<const uint2*>(&h[4]);
  }
  c = ptx::warp_sum(c);
  n2 = ptx::warp_sum(n2);
  amax = ptx::warp_max(amax);
  if (lane == 0) {
    cg[j] = c;
    atomicMax(reinterpret_cast<unsigned int*>(gstat), __float_as_uint(sqrtf(n2)));   // non-negative floats
    if (!(amax < FP16_MAX)) atomicMax(reinterpret_cast<unsigned int*>(gstat + 1), __float_as_uint(1.f));
  }
}

// ---------------------------------------------------------------- query preparation
// warp per query: a = -2 dw (.) q as fp16, rq = dw . q^2, ||a||, threshold reset
__global__ void __launch_bounds__(256) prep_queries_kernel(const float* q, int Q,
                                                           const float* __restrict__ fold, __half* __restrict__ a16,
                                                           float* __restrict__ rq, float* __restrict__ anorm,
                                                           uint32_t* __restrict__ thr_global,
                                                           uint32_t* __restrict__ rowflag,
                                                           int32_t* __restrict__ counters,
                                                           int32_t* __restrict__ xdone, const int x_on,
                                                           const xchg::Exchange xc) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + warp;
  if (x_on) {   // sharded search: the queries are the descriptors every rank has written into this rank's q_all
    const uint32_t step = xchg::current_step(xc);
    xchg::wait_all(xc, xchg::KIND_Q, step);
    q = xc.q_all[xc.rank] + (size_t)(step & 1u) * xc.Q * 256;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    counters[0] = 0;   // rows needing the exhaustive pass
    counters[1] = 0;   // fp16 overflow among the queries
  }
  if (i >= Q) return;
  const Slice x = load_slice(q + (size_t)i * 256, lane);
  const Slice dw = load_slice(fold + Fold::DW, lane);
  const float xs[8] = {x.lo.x, x.lo.y, x.lo.z, x.lo.w, x.hi.x, x.hi.y, x.hi.z, x.hi.w};
  const float ds[8] = {dw.lo.x, dw.lo.y, dw.lo.z, dw.lo.w, dw.hi.x, dw.hi.y, dw.hi.z, dw.hi.w};
  float r = 0.f, n2 = 0.f, amax = 0.f;
  __half h[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float a = -2.f * ds[e] * xs[e];
    r = fmaf(ds[e], xs[e] * xs[e], r);
    n2 = fmaf(a, a, n2);
    amax = fmaxf(amax, fabsf(a));
    h[e] = __float2half_rn(a);
  }
  __half* dst = a16 + (size_t)i * 256;
  *reinterpret_cast<uint2*>(dst + 4 * lane) = *reinterpret_cast<const uint2*>(&h[0]);
  *reinterpret_cast<uint2*>(dst + 128 + 4 * lane) = *reinterpret_cast<const uint2*>(&h[4]);
  r = ptx::warp_sum(r);
  n2 = ptx::warp_sum(n2);
  amax = ptx::warp_max(amax);
  if (lane == 0) {
    rq[i] = r;
    anorm[i] = sqrtf(n2);
    thr_global[i] = ptx::float_to_ordered(-INFINITY);
    rowflag[i] = 0;
    if (xdone) xdone[i] = 0;            // exhaustive kernel: slices finished per uncertified row
    if (!(amax < FP16_MAX)) atomicExch(counters + 1, 1);
  }
}

// ---------------------------------------------------------------- re-score + certify
struct RescoreParams {
  const float* q;        // (Q,256)
  const void* g;         // (G,256) rows of the kernel's Row type (float or __half)
  const float* fold;
  const uint2* rowbuf;         // (Q,nlists,CAP x 8 bytes): CAP/2 quad records {w0,w1,w2,w3} per sub-list
  const uint32_t* rowcnt;      // (Q,nlists) quad records in each sub-list
  const uint32_t* rowflag;     // (Q)
  const uint32_t* thr_global;  // (Q)
  const float* gmax;           // (Q,nlists,16) final group maxima (disjoint column groups)
  const float* rq;
  const float* anorm;
  const float* gstat;
  int Q, G, nlists, CAP, k, index_offset;
  float* out_score;
  float* out_margin;
  int32_t* out_idx;
  int32_t* counters;      // [0] number of uncertified rows, [1] query overflow flag
  int32_t* fallback_rows; // (Q)
  int x_on;               // sharded search: queries from the exchange's q_all, lists to the queries' owners
  xchg::Exchange x;
  score::TilePlan plan;   // which of the row's nlists slots the tensor-core pass wrote
};

// Where a query's top-k row goes.  Single GPU: row qi of the caller's (Q,k) outputs.  Sharded search: slot
// `rank` of the list buffer of the rank that owns the query (it merges the shards' lists); the score is a
// function of the margin and is not exchanged.
struct TopkDest {
  float* score;
  float* margin;
  int32_t* idx;
};
__device__ __forceinline__ TopkDest topk_dest(int x_on, const xchg::Exchange& x, uint32_t step, int qi, int k,
                                              float* out_score, float* out_margin, int32_t* out_idx) {
  TopkDest d;
  if (!x_on) {
    const size_t o = (size_t)qi * k;
    d.score = out_score + o;
    d.margin = out_margin + o;
    d.idx = out_idx + o;
  } else {
    const int ow = xchg::owner_of(x, qi);
    const size_t o = ((((size_t)(step & 1u) * x.world + x.rank) * x.own_max) + (size_t)(qi - x.q_lo[ow])) * k;
    d.score = nullptr;
    d.margin = x.list_margin[ow] + o;
    d.idx = x.list_idx[ow] + o;
  }
  return d;
}

// warp per query.
//  1. streams the row's candidate sub-lists (everything the tensor-core pass saw above the
//     bound the row had at the time), compacts the entries at or above the row's final bound
//     tau into shared memory and keeps the best 32 by approximate value, sorted;
//  2. S = candidates whose approximate value is within 2*eps of the k-th best approximate
//     value (eps bounds |approximate - exact|): the exact top-k is a subset of S as long as S
//     does not fill all 32 lanes (every item outside the 32 is <= the 32nd approximate value);
//  3. re-scores S in the fp32 direct form, orders it (margin desc, index asc), writes k entries.
// Rows that cannot be certified (S fills the window, candidates were dropped, fp16 overflow,
// or an observed |approximate - exact| above eps) go to the exhaustive kernel.
constexpr int RS_SUBL = 4;          // sub-lists swept per round (one 16-byte load per lane each)
constexpr int RESCORE_WBUF = 160;   // compaction buffer entries per warp (128 new + < 32 kept)

// merge the entries wb[begin, begin+32) (fewer at the tail) into the running sorted best-32
__device__ __forceinline__ void rescore_merge32(const uint2* wb, int begin, int end, float& cv, uint32_t& cidx,
                                                int lane) {
  float v = -INFINITY;
  uint32_t id = 0xffffffffu;
  if (begin + lane < end) {
    const uint2 e = wb[begin + lane];
    v = __uint_as_float(e.x);
    id = e.y;
  }
  const float worst = __shfl_sync(ptx::FULL_MASK, cv, 31);
  if (!(v > worst)) {
    v = -INFINITY;
    id = 0xffffffffu;
  }
  if (!__any_sync(ptx::FULL_MASK, v > -INFINITY)) return;
  wsort::sort32<false>(v, id, lane);           // ascending: cv (descending) || v is bitonic
  if (v > cv) {
    cv = v;
    cidx = id;
  }
  wsort::merge32<true>(cv, cidx, lane);
}

// (other occupancies were measured: 5 CTAs per SM = 48 registers, 168 bytes of spills: 70 -> 83 us; 3 CTAs = 80 registers: 78 us)
template <typename Row>
__global__ void __launch_bounds__(256) rescore_kernel(const RescoreParams p) {
  __shared__ uint2 wbuf[8][RESCORE_WBUF];
  __shared__ uint4 qbuf[8][64];
  __shared__ uint32_t qcol[8][64];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qi = blockIdx.x * 8 + warp;
  if (qi >= p.Q) return;
  const uint32_t xstep = p.x_on ? xchg::current_step(p.x) : 0u;
  const float* qbase = p.x_on ? p.x.q_all[p.x.rank] + (size_t)(xstep & 1u) * p.x.Q * 256 : p.q;
  const bool overflow = p.counters[1] != 0 || p.gstat[1] != 0.f;
  bool certified = !overflow && p.rowflag[qi] == 0;
  const float tau = ptx::ordered_to_float(p.thr_global[qi]);
  const int nl_valid = min(p.nlists, 4 * score::pieces_of_row(p.plan, qi));   // the sub-lists written for this row
  float cv = -INFINITY;
  uint32_t cidx = 0xffffffffu;
  uint2* wb = wbuf[warp];
  int fill = 0;
  // Streaming top-32 with a running cut: an entry is compacted into shared memory only if it
  // beats both the row's final bound tau and the 32nd best seen so far, and the buffer is merged
  // into the sorted best-32 (one bitonic sort + merge) whenever 32 such entries have gathered --
  // about 32 (1 + ln(n/32)) entries ever get that far.  Sub-lists are short (tens of entries):
  // they are swept four at a time with eight loads per lane in flight.
  float cut = tau;                                 // max(tau, 32nd best so far); entries equal to tau pass
  bool cut_strict = false;
  // one compare per value: v passes iff v > cut_lo, cut_lo = cut (strict) or the next float below it
  float cut_lo = tau > -INFINITY ? nextafterf(tau, -INFINITY) : -INFINITY;
  {
    // A tighter start: the row's group maxima belong to pairwise distinct gallery items, so the
    // 32nd largest of them (here: its ordered-integer image to 8 significant bits, found MSB
    // first) also bounds the 32nd best -- with ~40 instead of ~300 items above it.
    const int nval = nl_valid * 16;
    const float* gmp = p.gmax + (size_t)qi * p.nlists * 16;
    // NK keys per lane: 4 when the row's sweep was shared by at most two CTAs (128 maxima: the eval sizes), else 8
    auto start_cut = [&](auto nk_tag) {
      constexpr int NK = decltype(nk_tag)::value;
      uint32_t key[NK];
#pragma unroll
      for (int u = 0; u < NK; ++u) {
        const int i = lane + 32 * u;
        key[u] = i < nval ? ptx::float_to_ordered(gmp[i]) : 0u;
      }
      // The answer lies between lo = the smallest lane maximum (32 distinct maxima are >= it) and
      // hi = the largest maximum: only the bits below their common prefix need deciding.
      uint32_t lmax = key[0];
#pragma unroll
      for (int j = 1; j < NK; ++j) lmax = max(lmax, key[j]);
      const uint32_t hi = __reduce_max_sync(ptx::FULL_MASK, lmax);
      const uint32_t lo = __reduce_min_sync(ptx::FULL_MASK, lmax);
      uint32_t K = lo;
      if (hi != lo) {
        const int b0 = 31 - __clz(hi ^ lo);
        K = hi & ~((2u << b0) - 1u);                  // common prefix; at least 32 keys are >= it
        for (int b = b0; b >= 0 && b > b0 - 8; --b) {
          const uint32_t T = K | (1u << b);
          uint32_t c = 0;
#pragma unroll
          for (int j = 0; j < NK; ++j)
            asm("{\n.reg .pred p;\nsetp.ge.u32 p, %1, %2;\n@p add.u32 %0, %0, 1;\n}\n" : "+r"(c) : "r"(key[j]), "r"(T));
          if (__reduce_add_sync(ptx::FULL_MASK, c) >= 32u) K = T;
        }
      }
      const float tt = ptx::ordered_to_float(K);
      if (K != 0 && tt > cut) {                      // K == 0: fewer than 32 finite maxima
        cut = tt;
        cut_lo = nextafterf(tt, -INFINITY);
      }
    };
    if (nval <= 128) start_cut(std::integral_constant<int, 4>{});
    else if (nval <= 256) start_cut(std::integral_constant<int, 8>{});
  }
  // A record is a quad {w0,w1,w2,w3} of adjacent gallery rows whose tags name them (score_tc.cuh,
  // quad_first_col).  Two levels: quads whose maximum passes the cut are compacted into qb (one ballot
  // per 32 quads); every 32 of those are expanded into elements, which are compacted into wb and merged
  // into the best 32 as before.
  const int capq = p.CAP / 2;
  const uint4* rowq = reinterpret_cast<const uint4*>(p.rowbuf) + (size_t)qi * p.nlists * capq;
  uint4* qb = qbuf[warp];
  uint32_t* qc = qcol[warp];
  int qfill = 0;
  auto expand = [&](int start, int count) {
    uint4 rec = make_uint4(0u, 0u, 0u, 0u);
    uint32_t col = 0;
    const bool have = lane < count;
    if (have) {
      rec = qb[start + lane];
      col = qc[start + lane];
    }
    const uint32_t wv[4] = {rec.x, rec.y, rec.z, rec.w};
#pragma unroll
    for (int el = 0; el < 4; ++el) {
      const float ev = __uint_as_float(wv[el]);
      const bool pass = have && ev > cut_lo;
      const uint32_t mask = __ballot_sync(ptx::FULL_MASK, pass);
      if (mask == 0u) continue;                      // warp-uniform
      if (pass) wb[fill + __popc(mask & ((1u << lane) - 1u))] = make_uint2(wv[el], col + el);
      fill += __popc(mask);
    }
    if (fill >= 32) {                                // at most 128 new entries since the last check
      __syncwarp();
      while (fill >= 32) {                           // newest first: the tail of the buffer
        rescore_merge32(wb, fill - 32, fill, cv, cidx, lane);
        fill -= 32;
      }
      const float worst = __shfl_sync(ptx::FULL_MASK, cv, 31);
      if (worst > cut || (worst == cut && worst > -INFINITY)) {
        cut = worst;
        cut_strict = true;                           // ties with the 32nd best cannot displace it
        cut_lo = worst;
      }
    }
    __syncwarp();
  };
  for (int l0 = 0; l0 < nl_valid && certified; l0 += 32) {
    const int my_l = l0 + lane;
    uint32_t my_n = my_l < nl_valid ? p.rowcnt[(size_t)qi * p.nlists + my_l] : 0u;
    if (__any_sync(ptx::FULL_MASK, my_n > (uint32_t)capq)) {
      certified = false;
      break;
    }
    const int nl = min(32, nl_valid - l0);            // a multiple of RS_SUBL = 4 (4 sub-lists per piece)
    for (int j0 = 0; j0 < nl; j0 += RS_SUBL) {       // RS_SUBL sub-lists per round, 32 quads of each
      int n4[RS_SUBL];
      int nmax = 0;
#pragma unroll
      for (int u = 0; u < RS_SUBL; ++u) {
        n4[u] = (int)__shfl_sync(ptx::FULL_MASK, my_n, j0 + u);
        nmax = max(nmax, n4[u]);
      }
      const uint4* lp = rowq + (size_t)(l0 + j0) * capq + lane;
      for (int base = 0; base < nmax; base += 32) {
        uint4 e[RS_SUBL];
#pragma unroll
        for (int u = 0; u < RS_SUBL; ++u)             // slots past a list's end read as -inf: never pass
          e[u] = base + lane < n4[u] ? __ldcs(lp + (size_t)u * capq + base)
                                     : make_uint4(0xff800000u, 0xff800000u, 0xff800000u, 0xff800000u);
#pragma unroll
        for (int u = 0; u < RS_SUBL; ++u) {
          const float m = fmaxf(fmaxf(__uint_as_float(e[u].x), __uint_as_float(e[u].y)),
                                fmaxf(__uint_as_float(e[u].z), __uint_as_float(e[u].w)));
          const bool pass = m > cut_lo;
          const uint32_t mask = __ballot_sync(ptx::FULL_MASK, pass);
          if (mask == 0u) continue;                  // warp-uniform
          if (pass) {
            const int pos = qfill + __popc(mask & ((1u << lane) - 1u));
            qb[pos] = e[u];
            qc[pos] = score::quad_first_col(e[u], l0 + j0 + u);
          }
          qfill += __popc(mask);
          if (qfill >= 32) {
            __syncwarp();
            expand(qfill - 32, 32);
            qfill -= 32;
          }
        }
      }
    }
  }
  __syncwarp();
  if (certified && qfill > 0) expand(0, qfill);
  __syncwarp();
  if (certified && fill > 0) rescore_merge32(wb, 0, fill, cv, cidx, lane);
  const bool valid = (int)cidx >= 0;
  const int n_valid = __popc(__ballot_sync(ptx::FULL_MASK, valid));
  if (n_valid < min(32, p.G)) certified = false;          // candidates are missing
  const float a_k = __shfl_sync(ptx::FULL_MASK, cv, min(p.k, 32) - 1);
  // the tensor-core pass tags the 6 low mantissa bits of a value with its column (score_tc.cuh):
  // |tagged - untagged| <= 2^-17 |value|, bounded here by the largest magnitude in the window
  const float amax = ptx::warp_max(valid ? fabsf(cv) : 0.f);
  const float eps = EPS_COEFF * p.anorm[qi] * p.gstat[0] + 1e-5f + TAG_REL_ERR * amax;
  const float cutoff = a_k - 2.f * eps;                   // a_k = -inf when fewer than k candidates
  const bool in_S = valid && cv >= cutoff;
  const uint32_t smask = __ballot_sync(ptx::FULL_MASK, in_S);
  if (p.G > 32 && (smask >> 31)) certified = false;       // S fills the window
  const int ns = __popc(smask);                           // S is a prefix of the sorted lanes

  const Slice qs = load_slice(qbase + (size_t)qi * 256, lane);
  const Slice w0 = load_slice(p.fold + Fold::LAST_W, lane);
  const Slice w1 = load_slice(p.fold + Fold::LAST_W + 256, lane);
  const float b0 = p.fold[Fold::CONSTS + 5], b1 = p.fold[Fold::CONSTS + 6];
  float my_l0 = 0.f, my_l1 = 0.f;
  if (certified) {
    // four candidates per step: their 1 KB gallery rows are fetched together
    for (int c0 = 0; c0 < ns; c0 += 4) {
      Slice gs[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = __shfl_sync(ptx::FULL_MASK, (int)cidx, min(c0 + u, ns - 1));
        gs[u] = load_slice(static_cast<const Row*>(p.g) + (size_t)idx * 256, lane);
      }
      float part[8];
#pragma unroll
      for (int u = 0; u < 4; ++u) sqdiff_dot2(qs, gs[u], w0, w1, part[2 * u], part[2 * u + 1]);
      const float tot = ptx::treduce<8>(part, lane);   // lane l: total of part[l % 8]
      // candidate c0+u keeps its own pair: l0 from lane 2u, l1 from lane 2u+1
      const int u_mine = lane - c0;
      const float l0 = __shfl_sync(ptx::FULL_MASK, tot, (2 * u_mine) & 7) + b0;
      const float l1 = __shfl_sync(ptx::FULL_MASK, tot, (2 * u_mine + 1) & 7) + b1;
      if (u_mine >= 0 && u_mine < 4) {
        my_l0 = l0;
        my_l1 = l1;
      }
    }
  }
  float d = in_S ? my_l1 - my_l0 : -INFINITY;
  int id = in_S ? (int)cidx : INT_MAX;
  // observed error of the tensor-core value against the bound it was trusted with
  const float approx_d = cv + p.rq[qi] + p.fold[Fold::CONSTS + 4];
  const bool violated = in_S && !(fabsf(d - approx_d) <= eps + 2e-5f * (1.f + fabsf(d)));
  if (__any_sync(ptx::FULL_MASK, violated)) certified = false;
  wsort::sort32_rank2(d, id, lane);
  if (lane < p.k) {
    const TopkDest dst = topk_dest(p.x_on, p.x, xstep, qi, p.k, p.out_score, p.out_margin, p.out_idx);
    const bool ok = id != INT_MAX;
    // softmax(l0, l1)[1] depends on the logits only through d = l1 - l0 (the larger logit is
    // subtracted exactly), so it is formed after the sort: bit-identical to softmax1(l0, l1)
    if (dst.score) dst.score[lane] = ok ? softmax1(0.f, d) : 0.f;
    dst.margin[lane] = d;
    dst.idx[lane] = ok ? id + p.index_offset : -1;
  }
  if (!certified && lane == 0) {
    const int slot = atomicAdd(p.counters, 1);
    p.fallback_rows[slot] = qi;
  }
}

// ---------------------------------------------------------------- exhaustive fp32 ranking
struct ExactParams {
  const float* q;
  const void* g;          // rows of the kernel's Row type
  const float* fold;
  int Q, G, k, index_offset;
  const int32_t* count;   // number of rows to process (device), or null: all Q rows
  const int32_t* rows;    // row list when count != null
  float* out_score;
  float* out_margin;
  int32_t* out_idx;
  float* part_d;          // (max(grid, Q), 32) per-slice lists of a row split over several CTAs (null: never split)
  int32_t* part_i;
  int32_t* done;          // (Q) slices finished per listed row; zero on entry (prep_queries_kernel), zero again on exit
  int x_on;               // sharded search: see RescoreParams; this is the step's last list-writing kernel: it signals
  xchg::Exchange x;
};

constexpr int EXACT_MIN_SLICE = 128;   // gallery rows per slice at least (16 per warp: 4 rounds of 4)

// CTA (8 warps) per (row, gallery slice): each warp scans its share of the slice four items at a time (eight 16-byte
// loads per lane in flight, one transposing butterfly for the eight partial sums) keeping a sorted best-32 in its
// lanes; the eight lists are merged through shared memory.  A handful of uncertified rows must not cost a gallery
// sweep by ONE CTA each (15,000 items: 0.87 ms for a single row, four times the whole step): with fewer rows than CTAs
// a row's gallery is cut into S = grid / rows slices, every slice's list goes to global memory and the CTA that
// finishes a row's last slice merges them.  The result is independent of S: (margin desc, index asc) is a total order.
template <typename Row>
__global__ void __launch_bounds__(256) exact_topk_kernel(const ExactParams p) {
  __shared__ float sd[8][32];
  __shared__ int si[8][32];
  __shared__ int s_last;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nrows = p.count ? *p.count : p.Q;
  const uint32_t xstep = p.x_on ? xchg::current_step(p.x) : 0u;
  const float* qbase = p.x_on ? p.x.q_all[p.x.rank] + (size_t)(xstep & 1u) * p.x.Q * 256 : p.q;
  int S = 1;
  if (p.part_d && nrows > 0 && nrows < (int)gridDim.x) S = max(1, min((int)gridDim.x / nrows, p.G / EXACT_MIN_SLICE));
  const long long units = (long long)nrows * S;
  if (units == 0) {        // the usual case (every row certified): leave before anything is loaded
    if (p.x_on) xchg::signal_all(p.x, xchg::KIND_L, xstep, false);
    return;
  }
  const Slice w0 = load_slice(p.fold + Fold::LAST_W, lane);
  const Slice w1 = load_slice(p.fold + Fold::LAST_W + 256, lane);
  const float b0 = p.fold[Fold::CONSTS + 5], b1 = p.fold[Fold::CONSTS + 6];
  float cd;
  int cidx;
  // the eight warps' sorted lists -> one sorted best-32 in warp 0
  auto cta_merge = [&]() {
    sd[warp][lane] = cd;
    si[warp][lane] = cidx;
    __syncthreads();
    if (warp == 0) {
      float dummy = 0.f;
      for (int w = 1; w < 8; ++w) {
        const float od = sd[w][31 - lane];
        const int oi = si[w][31 - lane];
        if (wsort::ranks_before(od, oi, cd, cidx)) {
          cd = od;
          cidx = oi;
        }
        wsort::merge32_rank(cd, cidx, dummy, lane);
      }
    }
  };
  auto write_row = [&](int qi) {                 // warp 0
    if (lane < p.k) {
      const TopkDest dst = topk_dest(p.x_on, p.x, xstep, qi, p.k, p.out_score, p.out_margin, p.out_idx);
      const bool ok = cidx != INT_MAX;
      // softmax(l0, l1)[1] as a function of d = l1 - l0: bit-identical to softmax1(l0, l1) (rescore_kernel)
      if (dst.score) dst.score[lane] = ok ? softmax1(0.f, cd) : 0.f;
      dst.margin[lane] = cd;
      dst.idx[lane] = ok ? cidx + p.index_offset : -1;
    }
  };
  for (long long e = blockIdx.x; e < units; e += gridDim.x) {
    const int r = (int)(e / S), sl = (int)(e - (long long)r * S);
    const int qi = p.count ? p.rows[r] : r;
    const int j_lo = (int)((long long)p.G * sl / S), j_hi = (int)((long long)p.G * (sl + 1) / S);
    const Slice qs = load_slice(qbase + (size_t)qi * 256, lane);
    cd = -INFINITY;
    cidx = INT_MAX;
    for (int j0 = j_lo + 4 * warp; j0 < j_hi; j0 += 32) {
      Slice gs[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) gs[u] = load_slice(static_cast<const Row*>(p.g) + (size_t)min(j0 + u, j_hi - 1) * 256, lane);
      float part[8];
#pragma unroll
      for (int u = 0; u < 4; ++u) sqdiff_dot2(qs, gs[u], w0, w1, part[2 * u], part[2 * u + 1]);
      const float tot = ptx::treduce<8>(part, lane);   // lane l: total of part[l % 8] -- the association of warp_sum_b
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float l0 = __shfl_sync(ptx::FULL_MASK, tot, 2 * u) + b0;
        const float l1 = __shfl_sync(ptx::FULL_MASK, tot, 2 * u + 1) + b1;
        const float d = l1 - l0;
        const int j = j0 + u;
        const float wd = __shfl_sync(ptx::FULL_MASK, cd, 31);
        const int wi = __shfl_sync(ptx::FULL_MASK, cidx, 31);
        if (j < j_hi && wsort::ranks_before(d, j, wd, wi)) {   // warp-uniform
          const int pos = __popc(__ballot_sync(ptx::FULL_MASK, wsort::ranks_before(cd, cidx, d, j)));
          const float ud = __shfl_up_sync(ptx::FULL_MASK, cd, 1);
          const int ui = __shfl_up_sync(ptx::FULL_MASK, cidx, 1);
          if (lane > pos) {
            cd = ud;
            cidx = ui;
          } else if (lane == pos) {
            cd = d;
            cidx = j;
          }
        }
      }
    }
    cta_merge();
    if (S == 1) {
      if (warp == 0) write_row(qi);
      __syncthreads();
      continue;
    }
    // this slice's list -> global; the CTA that completes the row merges the S lists
    if (warp == 0) {
      __stcg(p.part_d + (size_t)e * 32 + lane, cd);
      __stcg(p.part_i + (size_t)e * 32 + lane, cidx);
      __threadfence();
      __syncwarp();
      if (lane == 0) s_last = atomicAdd(p.done + r, 1) == S - 1;
    }
    __syncthreads();
    if (s_last) {
      __threadfence();
      cd = -INFINITY;
      cidx = INT_MAX;
      float dummy = 0.f;
      for (int s2 = warp; s2 < S; s2 += 8) {
        const size_t o = ((size_t)r * S + s2) * 32 + (31 - lane);
        const float od = __ldcg(p.part_d + o);
        const int oi = __ldcg(p.part_i + o);
        if (wsort::ranks_before(od, oi, cd, cidx)) {
          cd = od;
          cidx = oi;
        }
        wsort::merge32_rank(cd, cidx, dummy, lane);
      }
      __syncthreads();                       // sd / si of the slice merge are free again
      cta_merge();
      if (warp == 0) {
        write_row(qi);
        if (lane == 0) p.done[r] = 0;        // as found: the next call may use any number of slices
      }
    }
    __syncthreads();
  }
  if (p.x_on) {          // every list row of this step (re-score kernel before: complete at its end; this one now) is on its way
    __syncthreads();
    xchg::signal_all(p.x, xchg::KIND_L, xstep, (long long)blockIdx.x < units);
  }
}

// ---------------------------------------------------------------- dense logits
// x5 (Q,G,2).  32 queries x 32 gallery rows per CTA, operands staged in shared memory.
template <bool PROB>     // false: x5 (Q,G,2) logits; true: (Q,G) class-1 probabilities softmax(x5)[...,1]
__global__ void __launch_bounds__(256) dense_logits_kernel(const float* __restrict__ q, int Q,
                                                           const float* __restrict__ g, int G,
                                                           const float* __restrict__ fold, float* __restrict__ x5) {
  __shared__ float qs[32][129];
  __shared__ float gs[32][129];
  __shared__ float ws[2][256];
  const int t = threadIdx.x;
  const int i0 = blockIdx.y * 32, j0 = blockIdx.x * 32;
  ws[0][t] = fold[Fold::LAST_W + t];
  ws[1][t] = fold[Fold::LAST_W + 256 + t];
  const int tx = t & 31, ty = t >> 5;   // gallery row, query group (4 queries each)
  float l0[4] = {}, l1[4] = {};
  for (int kh = 0; kh < 256; kh += 128) {   // K staged in two halves (static smem <= 48 KB)
    __syncthreads();
    for (int e = t; e < 32 * 128; e += 256) {
      const int r = e >> 7, c = e & 127;
      qs[r][c] = (i0 + r < Q) ? q[(size_t)(i0 + r) * 256 + kh + c] : 0.f;
      gs[r][c] = (j0 + r < G) ? g[(size_t)(j0 + r) * 256 + kh + c] : 0.f;
    }
    __syncthreads();
    for (int k = 0; k < 128; ++k) {
      const float gv = gs[tx][k];
      const float wa = ws[0][kh + k], wb = ws[1][kh + k];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float d = qs[ty * 4 + u][k] - gv;
        const float s = d * d;
        l0[u] = fmaf(wa, s, l0[u]);
        l1[u] = fmaf(wb, s, l1[u]);
      }
    }
  }
  const float b0 = fold[Fold::CONSTS + 5], b1 = fold[Fold::CONSTS + 6];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int i = i0 + ty * 4 + u, j = j0 + tx;
    if (i < Q && j < G) {
      if constexpr (PROB) {
        x5[(size_t)i * G + j] = softmax1(l0[u] + b0, l1[u] + b1);
      } else {
        float2 o = make_float2(l0[u] + b0, l1[u] + b1);
        *reinterpret_cast<float2*>(x5 + ((size_t)i * G + j) * 2) = o;
      }
    }
  }
}

// ---------------------------------------------------------------- per-product distance fusions
// evaluate_movingfashion.py:294-316 ("AVG & MAX DISTANCE"): per product, the class-1 probabilities of its tracked
// frames against every shop item (compute_distances, :101-106) are averaged / maximised over the frames and the
// true shop item's position in the descending order is read off.  Here, for all products at once and without
// ever materialising the (frames x gallery) matrix: a CTA takes one product x 1024 shop items, keeps the
// product's frames (16 at a time) in shared memory, each warp scores shop rows in the fp32 direct form against
// 4 frames per butterfly, and the per-item running sum / maximum live in shared memory; the target item's fused
// values are computed by the same code path, then every item is compared with them and counted.
//   frames (N,256) sorted by product, start (P+1) CSR offsets, target (P) shop row, ranks (P) zero-initialised.
// Products without frames get rank G (as the eval script never ranks them).
struct FusedDistParams {
  const float* frames;
  const int32_t* start;
  const float* g;
  const int32_t* target;
  const float* fold;
  int P, G;
  int32_t* rank_avg;
  int32_t* rank_max;
};
constexpr int FD_ROWS = 1024, FD_FRAMES = 16;

__global__ void __launch_bounds__(256) fused_dist_rank_kernel(const FusedDistParams p) {
  __shared__ __align__(16) float fs[FD_FRAMES][256];
  __shared__ float acc_sum[FD_ROWS + 1], acc_max[FD_ROWS + 1];     // last slot: the target item
  __shared__ int cnt_s[2];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int prod = blockIdx.x, j0 = blockIdx.y * FD_ROWS;
  const int f0 = p.start[prod], nf = p.start[prod + 1] - f0;
  if (nf <= 0) {
    if (blockIdx.y == 0 && threadIdx.x == 0) {
      p.rank_avg[prod] = p.G;
      p.rank_max[prod] = p.G;
    }
    return;
  }
  const int rows = min(FD_ROWS, p.G - j0);
  const int tj = p.target[prod];
  for (int i = threadIdx.x; i <= FD_ROWS; i += 256) {
    acc_sum[i] = 0.f;
    acc_max[i] = -INFINITY;
  }
  if (threadIdx.x < 2) cnt_s[threadIdx.x] = 0;
  const Slice w0 = load_slice(p.fold + Fold::LAST_W, lane);
  const Slice w1 = load_slice(p.fold + Fold::LAST_W + 256, lane);
  const float b0 = p.fold[Fold::CONSTS + 5], b1 = p.fold[Fold::CONSTS + 6];
  for (int c0 = 0; c0 < nf; c0 += FD_FRAMES) {
    const int nc = min(FD_FRAMES, nf - c0);
    __syncthreads();                                   // previous chunk consumed (and the accumulators initialised)
    for (int e = threadIdx.x; e < nc * 64; e += 256)
      reinterpret_cast<float4*>(&fs[0][0])[e] = reinterpret_cast<const float4*>(p.frames + (size_t)(f0 + c0) * 256)[e];
    __syncthreads();
    for (int r = warp; r <= rows; r += 8) {            // r == rows: the target item
      const int j = r < rows ? j0 + r : tj;
      const int slot = r < rows ? r : FD_ROWS;
      const Slice gs = load_slice(p.g + (size_t)j * 256, lane);
      float sum = 0.f, mx = -INFINITY;
      for (int fb = 0; fb < nc; fb += 4) {
        float part[8];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const Slice fr = load_slice(&fs[min(fb + u, nc - 1)][0], lane);
          sqdiff_dot2(fr, gs, w0, w1, part[2 * u], part[2 * u + 1]);
        }
        const float tot = ptx::treduce<8>(part, lane);   // lane l: total of part[l % 8]
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float l0 = __shfl_sync(ptx::FULL_MASK, tot, 2 * u) + b0;
          const float l1 = __shfl_sync(ptx::FULL_MASK, tot, 2 * u + 1) + b1;
          if (fb + u < nc) {
            const float pr = softmax1(l0, l1);
            sum += pr;
            mx = fmaxf(mx, pr);
          }
        }
      }
      if (lane == 0) {                                 // this warp owns the slot in this pass
        acc_sum[slot] += sum;
        acc_max[slot] = fmaxf(acc_max[slot], mx);
      }
    }
  }
  __syncthreads();
  const float inv = 1.f / (float)nf;
  const float tavg = acc_sum[FD_ROWS] * inv, tmax = acc_max[FD_ROWS];
  int ca = 0, cm = 0;
  for (int i = threadIdx.x; i < rows; i += 256) {
    const int j = j0 + i;
    const float a = acc_sum[i] * inv, m = acc_max[i];
    ca += (a > tavg || (a == tavg && j < tj)) ? 1 : 0;
    cm += (m > tmax || (m == tmax && j < tj)) ? 1 : 0;
  }
  ca = __reduce_add_sync(ptx::FULL_MASK, ca);
  cm = __reduce_add_sync(ptx::FULL_MASK, cm);
  if (lane == 0) {
    atomicAdd(&cnt_s[0], ca);
    atomicAdd(&cnt_s[1], cm);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicAdd(p.rank_avg + prod, cnt_s[0]);
    atomicAdd(p.rank_max + prod, cnt_s[1]);
  }
}

// ---------------------------------------------------------------- rank of a target item
// CTA per query: margin of the target, then count items ranking before it -- exhaustive, fp32 direct
// form.  With a row list (count, rows) only those queries are processed (the rows the tensor-core
// path below could not certify).
// EXT (one shard of a sharded gallery): the target's margin is ext_margin[qi] (the row may live on another GPU),
// target[] holds global rows and row j of this shard is global row j + index_offset; out_rank is this shard's count.
template <typename Row, bool EXT>
__global__ void __launch_bounds__(256) rank_of_target_kernel(const float* __restrict__ q, int Q,
                                                             const Row* __restrict__ g, int G,
                                                             const int32_t* __restrict__ target,
                                                             const float* __restrict__ fold,
                                                             const int32_t* __restrict__ count,
                                                             const int32_t* __restrict__ rows,
                                                             int32_t* __restrict__ out_rank,
                                                             float* __restrict__ out_margin,
                                                             const float* __restrict__ ext_margin, int index_offset) {
  __shared__ int cnt_s[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Slice w0 = load_slice(fold + Fold::LAST_W, lane);
  const Slice w1 = load_slice(fold + Fold::LAST_W + 256, lane);
  const float b0 = fold[Fold::CONSTS + 5], b1 = fold[Fold::CONSTS + 6];
  const int nrows = count ? *count : Q;
  for (int e = blockIdx.x; e < nrows; e += gridDim.x) {
    const int qi = count ? rows[e] : e;
    const Slice qs = load_slice(q + (size_t)qi * 256, lane);
    // EXT: the target as a row of this shard (j + index_offset < target  <=>  j < target - index_offset)
    const int tj = EXT ? target[qi] - index_offset : target[qi];
    float l0, l1;
    float dt;
    if (EXT) {
      dt = ext_margin[qi];
    } else {
      pair_logits(qs, g + (size_t)tj * 256, w0, w1, b0, b1, lane, l0, l1);
      dt = l1 - l0;
    }
    int cnt = 0;
    for (int j = warp; j < G; j += 8) {
      pair_logits(qs, g + (size_t)j * 256, w0, w1, b0, b1, lane, l0, l1);
      if (wsort::ranks_before(l1 - l0, j, dt, tj)) ++cnt;
    }
    if (lane == 0) cnt_s[warp] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
      int tot = 0;
      for (int w = 0; w < 8; ++w) tot += cnt_s[w];
      out_rank[qi] = tot;
      if (out_margin) out_margin[qi] = dt;
    }
    __syncthreads();
  }
}

// warp per query: the target's margin l1 - l0 when global row target[qi] lies in this shard
// [index_offset, index_offset + G), else -inf (so that a MAX over the shards is exact).  The same pair_logits call and
// lane mapping as rank_prep_kernel: the bits are those of the unsharded path.
template <typename Row>
__global__ void __launch_bounds__(256) target_margin_kernel(const float* __restrict__ q, int Q,
                                                            const Row* __restrict__ g, int G, int index_offset,
                                                            const int32_t* __restrict__ target,
                                                            const float* __restrict__ fold,
                                                            float* __restrict__ out_margin) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qi = blockIdx.x * 8 + warp;
  if (qi >= Q) return;
  const long long t = (long long)target[qi] - index_offset;
  if (t < 0 || t >= G) {
    if (lane == 0) out_margin[qi] = -INFINITY;
    return;
  }
  const Slice w0 = load_slice(fold + Fold::LAST_W, lane);
  const Slice w1 = load_slice(fold + Fold::LAST_W + 256, lane);
  const float b0 = fold[Fold::CONSTS + 5], b1 = fold[Fold::CONSTS + 6];
  const Slice qs = load_slice(q + (size_t)qi * 256, lane);
  float l0, l1;
  pair_logits(qs, g + (size_t)t * 256, w0, w1, b0, b1, lane, l0, l1);
  if (lane == 0) out_margin[qi] = l1 - l0;
}

// ---------------------------------------------------------------- rank of a target item, tensor-core path
// rank_i = #{ j : (d_ij, j) ranks before (d_it, t) } without visiting every pair in fp32: the tcgen05 pass
// (score_tc.cuh, VAR_RANK) counts the elements whose value exceeds the target's by more than its error
// bound and appends the quads that hold an element inside the band; rank_resolve_kernel adds the exact
// fp32 verdict for those.
//
// warp per query: exact margin of the target, its image v* in the space of the tensor-core values
// (v = d - rq - db), and the band v* +- E with E >= |w - v| for every element near the band:
// EPS_COEFF ||a_i|| max_j ||g_j||  (fp16 operands)  +  TAG_REL_ERR (|v*| + that)  (column tag)  +  fp32 slack.
// EXT: the target's margin is ext_margin[qi] and no target row is read; the band is built from it in the same way,
// with this shard's max_j ||g_j||, so it bounds the error of every row of this shard.
template <typename Row, bool EXT>
__global__ void __launch_bounds__(256) rank_prep_kernel(const float* __restrict__ q, int Q, const Row* __restrict__ g,
                                                        const int32_t* __restrict__ target,
                                                        const float* __restrict__ fold, const float* __restrict__ rq,
                                                        const float* __restrict__ anorm,
                                                        const float* __restrict__ gstat, float* __restrict__ lo,
                                                        float* __restrict__ hi, float* __restrict__ dtarget,
                                                        int32_t* __restrict__ above, int nlists,
                                                        const float* __restrict__ ext_margin) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qi = blockIdx.x * 8 + warp;
  if (qi >= Q) return;
  float dt;
  if (EXT) {
    dt = ext_margin[qi];
  } else {
    const Slice w0 = load_slice(fold + Fold::LAST_W, lane);
    const Slice w1 = load_slice(fold + Fold::LAST_W + 256, lane);
    const float b0 = fold[Fold::CONSTS + 5], b1 = fold[Fold::CONSTS + 6];
    const Slice qs = load_slice(q + (size_t)qi * 256, lane);
    float l0, l1;
    pair_logits(qs, g + (size_t)target[qi] * 256, w0, w1, b0, b1, lane, l0, l1);
    dt = l1 - l0;
  }
  for (int l = lane; l < nlists; l += 32) above[(size_t)qi * nlists + l] = 0;
  if (lane == 0) {
    const float vstar = dt - rq[qi] - fold[Fold::CONSTS + 4];
    const float e0 = EPS_COEFF * anorm[qi] * gstat[0] + 1e-5f;
    const float E = e0 + TAG_REL_ERR * (fabsf(vstar) + e0) + 4e-6f * (1.f + fabsf(dt) + fabsf(vstar));
    lo[qi] = vstar - E;
    hi[qi] = vstar + E;
    dtarget[qi] = dt;
  }
}

struct RankResolveParams {
  const float* q;
  const void* g;             // rows of the kernel's Row type
  const float* fold;
  const uint2* rowbuf;
  const uint32_t* rowcnt;
  const uint32_t* rowflag;
  const int32_t* above;      // (Q,nlists)
  const float* lo;
  const float* hi;
  const float* dtarget;
  const float* rq;
  const float* gstat;
  const int32_t* target;
  int Q, G, nlists, CAP;
  score::TilePlan plan;
  int32_t* out_rank;
  float* out_margin;         // optional
  int32_t* counters;         // [0] rows for the exhaustive kernel, [1] query overflow flag
  int32_t* fallback_rows;
  int index_offset;          // EXT: global row of this shard's row 0 (target[] holds global rows)
};
constexpr int RANK_CAND = 96;    // in-band candidates gathered before they are decided (+ 128 of headroom per round)

// warp per query: certain count from the tensor-core pass + exact verdicts for the elements in the band
// (a target in the bulk of the ranking has about 1 % of the gallery inside its band; one near the top,
// the case the eval cares about, a handful)
// EXT: one shard of a sharded gallery -- ties with the target are broken by global row
template <typename Row, bool EXT>
__global__ void __launch_bounds__(256) rank_resolve_kernel(const RankResolveParams p) {
  __shared__ uint2 cand[8][RANK_CAND + 128];   // {approximate value, gallery row}
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qi = blockIdx.x * 8 + warp;
  if (qi >= p.Q) return;
  const bool overflow = p.counters[1] != 0 || p.gstat[1] != 0.f;
  bool ok = !overflow && p.rowflag[qi] == 0;
  const float lo = p.lo[qi], hi = p.hi[qi], dt = p.dtarget[qi];
  const int tj = EXT ? p.target[qi] - p.index_offset : p.target[qi];   // EXT: as a row of this shard
  const int capq = p.CAP / 2;
  const uint4* rowq = reinterpret_cast<const uint4*>(p.rowbuf) + (size_t)qi * p.nlists * capq;
  uint2* cb = cand[warp];
  const Slice qs = load_slice(p.q + (size_t)qi * 256, lane);
  const Slice w0 = load_slice(p.fold + Fold::LAST_W, lane);
  const Slice w1 = load_slice(p.fold + Fold::LAST_W + 256, lane);
  const float b0 = p.fold[Fold::CONSTS + 5], b1 = p.fold[Fold::CONSTS + 6];
  const float eps = 0.5f * (hi - lo);
  const float shift = p.rq[qi] + p.fold[Fold::CONSTS + 4];
  int total = 0, fill = 0, exact_before = 0;
  // decides the buffered candidates in exact fp32, four gallery rows per step
  auto decide = [&]() {
    __syncwarp();
    for (int c0 = 0; c0 < fill; c0 += 4) {
      Slice gs[4];
      uint2 ce[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        ce[u] = cb[min(c0 + u, fill - 1)];
        gs[u] = load_slice(static_cast<const Row*>(p.g) + (size_t)ce[u].y * 256, lane);
      }
      float part[8];
#pragma unroll
      for (int u = 0; u < 4; ++u) sqdiff_dot2(qs, gs[u], w0, w1, part[2 * u], part[2 * u + 1]);
      const float tot = ptx::treduce<8>(part, lane);   // lane l: total of part[l % 8]
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float l0v = __shfl_sync(ptx::FULL_MASK, tot, 2 * u) + b0;
        const float l1v = __shfl_sync(ptx::FULL_MASK, tot, 2 * u + 1) + b1;
        const float d = l1v - l0v;
        if (c0 + u < fill) {
          if (wsort::ranks_before(d, (int)ce[u].y, dt, tj)) ++exact_before;
          // observed error of the tensor-core value against the bound the band was built with
          if (!(fabsf(d - (__uint_as_float(ce[u].x) + shift)) <= eps)) ok = false;
        }
      }
    }
    fill = 0;
    __syncwarp();
  };
  const int nl_valid = min(p.nlists, 4 * score::pieces_of_row(p.plan, qi));
  for (int l0 = 0; l0 < nl_valid && ok; l0 += 32) {
    const int my_l = l0 + lane;
    const uint32_t my_n = my_l < nl_valid ? p.rowcnt[(size_t)qi * p.nlists + my_l] : 0u;
    total += my_l < nl_valid ? p.above[(size_t)qi * p.nlists + my_l] : 0;
    if (__any_sync(ptx::FULL_MASK, my_n > (uint32_t)capq)) ok = false;
    const int nl = min(32, nl_valid - l0);
    for (int j = 0; j < nl && ok; ++j) {
      const int n = (int)__shfl_sync(ptx::FULL_MASK, my_n, j);
      const uint4* lp = rowq + (size_t)(l0 + j) * capq;
      for (int base = 0; base < n && ok; base += 32) {
        const bool have = base + lane < n;
        const uint4 rec = have ? __ldcs(lp + base + lane) : make_uint4(0u, 0u, 0u, 0u);
        const uint32_t wv[4] = {rec.x, rec.y, rec.z, rec.w};
        const uint32_t col = score::quad_first_col(rec, l0 + j);
#pragma unroll
        for (int el = 0; el < 4; ++el) {
          const float ev = __uint_as_float(wv[el]);
          const bool in_band = have && ev > lo && !(ev > hi);
          const uint32_t mask = __ballot_sync(ptx::FULL_MASK, in_band);
          if (mask == 0u) continue;
          if (in_band) cb[fill + __popc(mask & ((1u << lane) - 1u))] = make_uint2(wv[el], col + el);
          fill += __popc(mask);
        }
        if (fill >= RANK_CAND) decide();
      }
    }
  }
  total = __reduce_add_sync(ptx::FULL_MASK, total);
  if (ok && fill > 0) decide();
  if (lane == 0) {
    if (ok) {
      p.out_rank[qi] = total + exact_before;
      if (p.out_margin) p.out_margin[qi] = dt;
    } else {
      const int slot = atomicAdd(p.counters, 1);
      p.fallback_rows[slot] = qi;
    }
  }
}

// ---------------------------------------------------------------- shard merge
// warp per query; each input list is sorted best first with idx < 0 marking padding.  scores may be
// null: the score is a function of the margin alone (softmax1(0, d), exactly what the re-score kernel
// writes), so shards need not exchange it.
__global__ void __launch_bounds__(256) merge_topk_kernel(const float* __restrict__ scores,
                                                         const float* __restrict__ margins,
                                                         const int32_t* __restrict__ idx, int N, int Q, int k,
                                                         float* __restrict__ out_score,
                                                         float* __restrict__ out_margin,
                                                         int32_t* __restrict__ out_idx) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int qi = blockIdx.x * 8 + warp;
  if (qi >= Q) return;
  float d = -INFINITY, s = 0.f;
  int id = INT_MAX;
  for (int n = 0; n < N; ++n) {
    const size_t base = ((size_t)n * Q + qi) * k;
    if (n == 0) {
      if (lane < k && idx[base + lane] >= 0) {
        d = margins[base + lane];
        s = scores ? scores[base + lane] : 0.f;
        id = idx[base + lane];
      }
    } else {
      const int e = 31 - lane;   // reversed: worst first
      float od = -INFINITY, os = 0.f;
      int oi = INT_MAX;
      if (e < k && idx[base + e] >= 0) {
        od = margins[base + e];
        os = scores ? scores[base + e] : 0.f;
        oi = idx[base + e];
      }
      if (wsort::ranks_before(od, oi, d, id)) {
        d = od;
        id = oi;
        s = os;
      }
      wsort::merge32_rank(d, id, s, lane);
    }
  }
  if (lane < k) {
    const size_t o = (size_t)qi * k + lane;
    const bool ok = id != INT_MAX;
    out_score[o] = ok ? (scores ? s : softmax1(0.f, d)) : 0.f;
    out_margin[o] = ok ? d : -INFINITY;
    out_idx[o] = ok ? id : -1;
  }
}

// Sharded merge: this rank merges the world per-shard lists of the queries it OWNS (they were written into its
// list buffer by every rank's re-score kernels), writes the merged rows into the final (Q,k) buffers of every
// rank when the exchange has them (else into the caller's (own,k) outputs), and -- as the last kernel of a step
// -- waits for every rank's merged rows to have landed here and advances the step.
__global__ void __launch_bounds__(256) merge_sharded_kernel(const xchg::Exchange x, float* __restrict__ out_score,
                                                            float* __restrict__ out_margin,
                                                            int32_t* __restrict__ out_idx) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t step = xchg::current_step(x);
  xchg::wait_all(x, xchg::KIND_L, step);
  const int own = x.q_lo[x.rank + 1] - x.q_lo[x.rank], k = x.k;
  const int qo = blockIdx.x * 8 + warp;
  if (qo < own) {
    const float* margins = x.list_margin[x.rank] + (size_t)(step & 1u) * x.world * x.own_max * k;
    const int32_t* idx = x.list_idx[x.rank] + (size_t)(step & 1u) * x.world * x.own_max * k;
    float d = -INFINITY, s = 0.f;
    int id = INT_MAX;
    for (int n = 0; n < x.world; ++n) {
      const size_t base = ((size_t)n * x.own_max + qo) * k;
      const int e = n == 0 ? lane : 31 - lane;   // later lists reversed: worst first
      float od = -INFINITY;
      int oi = INT_MAX;
      if (e < k) {
        const int32_t ii = __ldcg(idx + base + e);
        if (ii >= 0) {
          od = __ldcg(margins + base + e);
          oi = ii;
        }
      }
      if (n == 0) {
        d = od;
        id = oi;
      } else {
        if (wsort::ranks_before(od, oi, d, id)) {
          d = od;
          id = oi;
        }
        wsort::merge32_rank(d, id, s, lane);
      }
    }
    if (lane < k) {
      const bool ok = id != INT_MAX;
      const float sc = ok ? softmax1(0.f, d) : 0.f;
      const float dm = ok ? d : -INFINITY;
      const int ii = ok ? id : -1;
      if (x.final_score[0]) {
        const size_t o = (size_t)(x.q_lo[x.rank] + qo) * k + lane;
        if (x.final_score_mc) {               // NVSwitch multicast: one store reaches every rank's copy
          x.final_score_mc[o] = sc;
          x.final_margin_mc[o] = dm;
          x.final_idx_mc[o] = ii;
        } else {
          for (int r = 0; r < x.world; ++r) {
            x.final_score[r][o] = sc;
            x.final_margin[r][o] = dm;
            x.final_idx[r][o] = ii;
          }
        }
      } else {
        const size_t o = (size_t)qo * k + lane;
        out_score[o] = sc;
        out_margin[o] = dm;
        out_idx[o] = ii;
      }
    }
  }
  __syncthreads();
  if (xchg::signal_all(x, xchg::KIND_F, step)) {       // thread 0 of the grid's last CTA
    if (x.final_score[0]) {
      for (int r = 0; r < x.world; ++r) {
        const uint32_t* f = x.flags[x.rank] + xchg::KIND_F * xchg::MAX_WORLD + r;
        uint64_t t0 = 0;
        while ((int32_t)(xchg::ld_acquire_sys(f) - step) < 0) {
          __nanosleep(100);
          const uint64_t now = ptx::globaltimer_ns();
          if (t0 == 0) t0 = now;
          else if (now - t0 > 10000000000ull) ptx::watchdog_trap(210u, (uint32_t)r, step);
        }
      }
    }
    *reinterpret_cast<volatile uint32_t*>(x.step) = step + 1u;
  }
}

}  // namespace exact
}  // namespace seam
