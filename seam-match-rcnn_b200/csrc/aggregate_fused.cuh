// K1: temporal aggregation in ONE kernel -- streaming frame pass + the block's 256x256 map on the
// tensor cores, nothing but the descriptors ever written to global memory.
//
// Replaces the per-track Python loop of TemporalAggregationNLB.forward's seq-branch,
// models/match_head.py:133-154, and the block it calls, models/nlb.py:66-101, collapsed as in
// DESIGN.md "K1 algebra":
//   out = sum_t p_t x_t + M (sum_j q_j x_j) + (sum_j q_j) W_W b_g + b_W,   M = W_W W_g.
//
// Roles.  PRODUCER warps stream the tracks (bulk async copies into private shared-memory buffers,
// frames pulled into registers once, four dots per frame, T x T interaction + softmax, both weighted
// sums) exactly as a stand-alone streaming kernel would; instead of writing pooled' / r to global
// memory they PUBLISH them into a batch of NB = 16 tracks in shared memory: r as two fp16 terms
// (r * s = r1 + r2, s = a per-track power of two) in the 128-byte-swizzled K-major layout tcgen05 reads
// as its B operand, pooled' in fp32.  Four HELPER warps own the tensor core: M * S = M1 + M2 (fp16
// terms, fold.cuh) lives in TENSOR MEMORY for the whole kernel as the A operand (M1: 256 columns, the
// first 224 k's of M2: 224 columns, accumulator: 32 columns = all 512; the last 32 k's of M2 sit in
// 16 KB of shared memory), so a batch costs 96 small MMAs (D^T[256 ch x 16 tracks] = M1 r1 + M1 r2 +
// M2 r1, fp32 accumulation: 22-bit operands, the dropped M2 r2 term is 2^-22 relative) and NO operand
// traffic at all.  The helpers read the accumulator back (lane = channel, so every global store is a
// 128-byte line), add pooled' and write the descriptor.  Batches are double-buffered: producers run up
// to two batches ahead of the tensor core.
//
// Results do not depend on how tracks are grouped into batches (a column of D depends on its own track
// only; the accumulation order over k is fixed), nor on which slot a track lands in.
//
// Tracks are fp32 or fp16 (template parameter In): only the track buffers and the copies into them follow the element
// size; load_frame widens an fp16 frame to fp32 as it leaves shared memory (exact), so the fp16 instantiations give
// bit for bit what the fp32 ones give on the widened tracks.
//
// A producer's iteration is a LATENCY CHAIN (2-3 producer warps per scheduler: shuffle rounds, named barriers,
// shared-memory atomics, mbarrier polls and the hand-over of a copy to the copy engine all sit on one warp's
// critical path), so the code below trades instructions for fewer dependent steps: reductions are folded into
// loops that read the data anyway, warp maxima are one CREDUX, the softmax of a long track needs one barrier,
// butterflies run over 32 totals, a loader warp issues the short-track kernel's copies (DESIGN.md, K1).
#pragma once
#include <cstdint>
#include <type_traits>
#include <cuda.h>
#include <cuda_fp16.h>
#include "exchange.cuh"
#include "fold.cuh"
#include "sm100_ptx.cuh"

namespace seam {
namespace aggf {

constexpr int D = 256;
constexpr int NB = 16;                       // tracks per tensor-core batch (UMMA N)
constexpr int HELPER_WARPS = 4;
constexpr uint32_t IDLE_NS = 400;            // long tracks: sleep between polls of a helper warp waiting for the next batch
constexpr int KT = Fold::M2_KT;              // k's of M2 resident in tensor memory
constexpr int KS = 256 - KT;                 // k's of M2 in shared memory (64-byte rows, SWIZZLE_64B)
constexpr uint32_t COL_D = 0;                // accumulator: half h at COL_D + h*NB
constexpr uint32_t COL_M1 = 32;              // M1 half h at COL_M1 + h*128 (k pair c at + c)
constexpr uint32_t COL_M2 = COL_M1 + 256;    // M2 half h at COL_M2 + h*(KT/2)
static_assert(COL_M2 + KT == 512 && 2 * NB <= (int)COL_M1 && KS == 32, "tensor-memory column map");

constexpr uint32_t RT_TERM_BYTES = NB * 512;           // one fp16 term: 4 k-blocks x NB rows x 128 B
constexpr uint32_t RT_BYTES = 2 * RT_TERM_BYTES;       // r1 | r2
constexpr uint32_t TAIL_BYTES = 256 * KS * 2;          // 2 halves x 128 rows x 64 B
constexpr uint32_t POOL_BYTES = NB * D * 4;
constexpr uint32_t OFF_RT = 0;                         // [2] buffers
constexpr uint32_t OFF_TAIL = OFF_RT + 2 * RT_BYTES;
constexpr uint32_t OFF_META = OFF_TAIL + TAIL_BYTES;
struct Meta {
  int slot_track[2][NB];
  float fscale[2][NB];
  uint64_t tile_full[2];     // producers -> MMA      (NB x ARRIVALS arrivals)
  uint64_t buf_free[2];      // helpers  -> producers (HELPER_WARPS arrivals)
  uint64_t acc_full;         // MMA      -> helpers   (tcgen05.commit)
  uint64_t m_ready;          // all warps -> MMA      (their share of M sits in tensor memory)
  unsigned int next_slot;
  uint32_t tmem_base;
};
constexpr uint32_t OFF_POOL = OFF_META + 512;          // [2] buffers, only when pooled' is staged in shared memory
static_assert(sizeof(Meta) <= 512, "meta block");
template <bool POOL_SMEM>
__host__ __device__ constexpr uint32_t fused_bytes() {
  return (OFF_POOL + (POOL_SMEM ? 2 * POOL_BYTES : 0) + 1023u) & ~1023u;
}

struct Params {
  const void* seq;         // float or __half: the kernels' In
  const uint8_t* mask;     // (Q, 1+Tmax) or null
  const int32_t* lens;     // (Q) or null
  int Tmax, Q;
  long long frame_stride, track_stride;   // elements of seq
  const float* fold;
  float* out;      // (Q,256)
  float* att;      // (Q,Tmax) or null
  int use_tm;      // the warp kernel may fetch a full track with ONE 3-D tensor-map copy (tmSeq is valid)
  // gallery-sharded search (exchange.cuh): the descriptors of this rank's tracks go to row x_row0 + track of the
  // current-parity q_all buffer of EVERY rank; the launch that holds the rank's last tracks (x_last) signals
  int x_on, x_last, x_row0;
  xchg::Exchange x;
};
// where this rank's own copy of the descriptors lives
__device__ __forceinline__ float* local_out(const Params& p, uint32_t xstep) {
  return p.x_on ? p.x.q_all[p.x.rank] + ((size_t)(xstep & 1u) * p.x.Q + (size_t)p.x_row0) * D : p.out;
}

using ptx::treduce;

// ---- packed fp32 pairs (FFMA2 / FMUL2): the streaming pass is bound by instruction issue
typedef unsigned long long u64;
__device__ __forceinline__ u64 pk(float lo, float hi) {
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk(u64 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
  u64 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
  u64 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
  u64 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
struct Vec8 {   // this lane's channels [4l,4l+4) and [128+4l,128+4l+4) as four pairs
  u64 a, b, c, d;
};
__device__ __forceinline__ Vec8 load_vec8(const float* row, int lane) {
  const ulonglong2 lo = *reinterpret_cast<const ulonglong2*>(row + 4 * lane);
  const ulonglong2 hi = *reinterpret_cast<const ulonglong2*>(row + 128 + 4 * lane);
  return Vec8{lo.x, lo.y, hi.x, hi.y};
}
// a frame of the track buffer (In = float or __half) -> registers, with the lane -> channel mapping of load_vec8.
// fp16 frames are widened here (exact), so every instruction after this load is the fp32 path's.
__device__ __forceinline__ u64 widen2(uint32_t h2) {
  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h2));
  return pk(f.x, f.y);
}
template <typename In>
__device__ __forceinline__ Vec8 load_frame(const In* row, int lane) {
  if constexpr (std::is_same<In, float>::value) {
    return load_vec8(row, lane);
  } else {
    static_assert(std::is_same<In, __half>::value, "frames are float or __half");
    const uint2 lo = *reinterpret_cast<const uint2*>(row + 4 * lane);
    const uint2 hi = *reinterpret_cast<const uint2*>(row + 128 + 4 * lane);
    return Vec8{widen2(lo.x), widen2(lo.y), widen2(hi.x), widen2(hi.y)};
  }
}
__device__ __forceinline__ Vec8 zero_vec8() { return Vec8{0ull, 0ull, 0ull, 0ull}; }
__device__ __forceinline__ float dot8(const Vec8& x, const Vec8& u) {
  u64 acc = mul2(x.a, u.a);
  acc = fma2(x.b, u.b, acc);
  acc = fma2(x.c, u.c, acc);
  acc = fma2(x.d, u.d, acc);
  float lo, hi;
  upk(acc, lo, hi);
  return lo + hi;
}
__device__ __forceinline__ void fma8(Vec8& acc, u64 ss, const Vec8& x) {
  acc.a = fma2(ss, x.a, acc.a);
  acc.b = fma2(ss, x.b, acc.b);
  acc.c = fma2(ss, x.c, acc.c);
  acc.d = fma2(ss, x.d, acc.d);
}
__device__ __forceinline__ void unpack_vec8(const Vec8& v, float4& lo, float4& hi) {
  upk(v.a, lo.x, lo.y);
  upk(v.b, lo.z, lo.w);
  upk(v.c, hi.x, hi.y);
  upk(v.d, hi.z, hi.w);
}

// r * s = h1 + h2 in fp16 (h1 = round(r s), h2 = round(r s - h1): the residual is exact in fp32)
__device__ __forceinline__ void split16(float a, float b, float s, uint32_t& t1, uint32_t& t2) {
  const float as = a * s, bs = b * s;
  const __half2 h1 = __floats2half2_rn(as, bs);
  const float2 f1 = __half22float2(h1);
  const __half2 h2 = __floats2half2_rn(as - f1.x, bs - f1.y);
  t1 = *reinterpret_cast<const uint32_t*>(&h1);
  t2 = *reinterpret_cast<const uint32_t*>(&h2);
}
// power of two s with max * s in [1,2) (1 for max == 0); *inv = 1 / s
__device__ __forceinline__ float track_scale(float mx, float* inv) {
  unsigned eb = (__float_as_uint(mx) >> 23) & 0xffu;
  if (mx == 0.f) eb = 127u;
  eb = eb < 1u ? 1u : (eb > 253u ? 253u : eb);
  *inv = __uint_as_float(eb << 23);
  return __uint_as_float((254u - eb) << 23);
}

// ------------------------------------------------------------------------------------------------
// Publishing a finished track into the current batch.  slot = running count of the CTA's finished
// tracks; batch = slot / NB uses buffer batch & 1, which is free once the helpers are done with batch - 2.
struct Slot {
  int buf, pos;
};
__device__ __forceinline__ Slot wait_slot(Meta* meta, unsigned s) {   // s = the track's ticket (atomicAdd on next_slot)
  const unsigned batch = s / NB;
  Slot sl;
  sl.buf = (int)(batch & 1u);
  sl.pos = (int)(s % NB);
  ptx::mbar_wait(&meta->buf_free[sl.buf], ((batch >> 1) & 1u) ^ 1u, 101);
  return sl;
}
// 4 consecutive channels c..c+3 (c % 4 == 0) of both fp16 terms of row pos: one 8-byte store per term
__device__ __forceinline__ void store_r4(uint8_t* rt, int pos, int c, const float4& r, float s) {
  uint32_t a1, a2, b1, b2;
  split16(r.x, r.y, s, a1, a2);
  split16(r.z, r.w, s, b1, b2);
  const uint32_t off = (uint32_t)(c >> 6) * (NB * 128) + (uint32_t)pos * 128 +
                       ((((uint32_t)(c & 63) >> 3) ^ ((uint32_t)pos & 7u)) << 4) + ((uint32_t)(c & 7) << 1);
  *reinterpret_cast<uint2*>(rt + off) = make_uint2(a1, b1);
  *reinterpret_cast<uint2*>(rt + RT_TERM_BYTES + off) = make_uint2(a2, b2);
}
// 2 consecutive channels (c % 2 == 0)
__device__ __forceinline__ void store_r2(uint8_t* rt, int pos, int c, float r0, float r1, float s) {
  uint32_t a1, a2;
  split16(r0, r1, s, a1, a2);
  const uint32_t off = (uint32_t)(c >> 6) * (NB * 128) + (uint32_t)pos * 128 +
                       ((((uint32_t)(c & 63) >> 3) ^ ((uint32_t)pos & 7u)) << 4) + ((uint32_t)(c & 7) << 1);
  *reinterpret_cast<uint32_t*>(rt + off) = a1;
  *reinterpret_cast<uint32_t*>(rt + RT_TERM_BYTES + off) = a2;
}

// ------------------------------------------------------------------------------------------------
// M -> tensor memory, by ALL warps of the CTA (a warp can only write the 32 lanes of its own quarter,
// warp % 4): the 30 chunks of 16 columns (M1: 2 halves x 8, M2: 2 halves x 7) of a quarter are dealt out
// to the NWARPS / 4 warps that share it, two chunks (32 coalesced loads per thread) in flight at a time.
// A serial load by the four helper warps alone took 22 dependent round trips (~17 us, the floor of the
// kernel at small Q); producers do their share while their first frames are in flight.
template <int NWARPS, int INFLIGHT>
__device__ __forceinline__ void load_m_tmem(const Params& p, Meta* meta, int warp, int lane) {
  constexpr int NPART = NWARPS / 4, NCHUNK = 16 + 2 * (KT / 32);
  static_assert((KT / 2) % 4 == 0, "four columns per 16-byte load");
  const int part = warp >> 2, quarter = warp & 3;
  const uint32_t lane_base = meta->tmem_base + ((uint32_t)(quarter * 32) << 16);
  // the images are [column / 4][row][column % 4] words (fold.cuh): four columns of this lane's row per 16-byte load
  const uint4* f128 = reinterpret_cast<const uint4*>(p.fold) + quarter * 32 + lane;
  auto locate = [&](int c, const uint4*& src, uint32_t& col) {
    if (c < 16) {
      const int h = c >> 3, c0 = (c & 7) * 16;
      src = f128 + Fold::M1_IMG / 4 + ((h * 128 + c0) >> 2) * 128;
      col = COL_M1 + h * 128 + c0;
    } else {
      const int cc = c - 16, h = cc / (KT / 32), c0 = (cc % (KT / 32)) * 16;
      src = f128 + Fold::M2_IMG / 4 + ((h * (KT / 2) + c0) >> 2) * 128;
      col = COL_M2 + h * (KT / 2) + c0;
    }
  };
#pragma unroll 1
  for (int c = part; c < NCHUNK; c += INFLIGHT * NPART) {
    uint32_t v[INFLIGHT][16], col[INFLIGHT];
#pragma unroll
    for (int u = 0; u < INFLIGHT; ++u) {
      const uint4* src;
      const int cu = c + u * NPART;
      locate(cu < NCHUNK ? cu : c, src, col[u]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint4 w = __ldg(src + j * 128);
        v[u][4 * j + 0] = w.x;
        v[u][4 * j + 1] = w.y;
        v[u][4 * j + 2] = w.z;
        v[u][4 * j + 3] = w.w;
      }
    }
#pragma unroll
    for (int u = 0; u < INFLIGHT; ++u)
      if (c + u * NPART < NCHUNK) ptx::tmem_st_x16(lane_base + col[u], v[u]);
  }
  ptx::tmem_st_wait();
  ptx::tc_fence_before();
  __syncwarp();
  if (lane == 0) ptx::mbar_arrive(&meta->m_ready);
}

// ------------------------------------------------------------------------------------------------
// Helper warps: tensor-memory set-up, one MMA batch per NB published tracks, read-back + store.
//   units        producer units (warps or warp groups) of this CTA, unit u handles tracks
//                first0 + u, first0 + u + stride, ...
//   ARRIVALS     mbarrier arrivals per published track (warps per track)
template <int ARRIVALS, bool POOL_SMEM>
__device__ __forceinline__ void helper_role(const Params& p, uint8_t* fz, int hw, int lane, int units, long long first0,
                                            long long stride, float* out_local, uint32_t xstep) {
  Meta* meta = reinterpret_cast<Meta*>(fz + OFF_META);
  const uint32_t tmem = meta->tmem_base;
  const uint32_t lane_base = tmem + ((uint32_t)(hw * 32) << 16);
  const uint32_t* f32 = reinterpret_cast<const uint32_t*>(p.fold);

  // ---- M2's last k's -> shared memory (the tensor-memory part of M is loaded by all warps, load_m_tmem)
  {
    const uint4* tsrc = reinterpret_cast<const uint4*>(f32 + Fold::M2_TAIL);
    uint4* tdst = reinterpret_cast<uint4*>(fz + OFF_TAIL);
    for (int i = hw * 32 + lane; i < (int)(TAIL_BYTES / 16); i += HELPER_WARPS * 32) tdst[i] = __ldg(tsrc + i);
    ptx::fence_proxy_async_smem();
    ptx::named_bar_sync(1, HELPER_WARPS * 32);
  }

  // tracks this CTA handles (static strided assignment of the producers)
  long long n_cta = 0;
  for (int u = 0; u < units; ++u) {
    const long long f = first0 + u;
    if (f < p.Q) n_cta += (p.Q - f + stride - 1) / stride;
  }
  const int nbatch = (int)((n_cta + NB - 1) / NB);
  const float ms_inv = p.fold[Fold::CONSTS + 9];        // 1 / S
  const bool mc = p.x_on && p.x.world > 1 && p.x.q_all_mc != nullptr;
  const uint32_t rt_addr = ptx::smem_u32(fz + OFF_RT), tail_addr = ptx::smem_u32(fz + OFF_TAIL);
  constexpr uint32_t idesc = ptx::umma_idesc(0 /*fp16*/, 128, NB);

#pragma unroll 1
  for (int b = 0; b < nbatch; ++b) {
    const int buf = b & 1;
    const int cnt = (b == nbatch - 1) ? (int)(n_cta - (long long)b * NB) : NB;
    if (hw == 0) {
      // ------------------------------------------------ MMA issue (one elected lane of the converged warp)
      if (lane == 0)
        for (int i = 0; i < (NB - cnt) * ARRIVALS; ++i) ptx::mbar_arrive(&meta->tile_full[buf]);   // slots nobody fills
      if constexpr (POOL_SMEM) ptx::mbar_wait(&meta->tile_full[buf], (uint32_t)(b >> 1) & 1u, 102);   // short tracks: a batch every few us
      else ptx::mbar_wait_idle(&meta->tile_full[buf], (uint32_t)(b >> 1) & 1u, IDLE_NS, 102);          // long tracks: tens of us away
      if (b == 0) ptx::mbar_wait(&meta->m_ready, 0u, 108);
      ptx::tc_fence_after();
      if (ptx::elect_one()) {
        const uint32_t r1 = rt_addr + buf * RT_BYTES, r2 = r1 + RT_TERM_BYTES;
#pragma unroll 1
        for (int h = 0; h < 2; ++h) {
          const uint32_t d = tmem + COL_D + h * NB;
#pragma unroll
          for (int ks = 0; ks < 16; ++ks) {               // k-steps of 16
            const uint32_t boff = (uint32_t)(ks >> 2) * (NB * 128) + (uint32_t)(ks & 3) * 32;
            const uint64_t b1 = ptx::umma_desc_k_sw128(r1 + boff), b2 = ptx::umma_desc_k_sw128(r2 + boff);
            const uint32_t a1 = tmem + COL_M1 + h * 128 + ks * 8;
            ptx::umma_f16_ts(d, a1, b2, idesc, ks != 0 ? 1u : 0u);                                  // M1 r2 (small terms first)
            if (ks * 16 < KT) {
              ptx::umma_f16_ts(d, tmem + COL_M2 + h * (KT / 2) + ks * 8, b1, idesc, 1u);             // M2 r1
            } else {
              const uint64_t at = ptx::umma_desc_k_sw64(tail_addr + h * (128 * KS * 2) + (ks * 16 - KT) * 2);
              ptx::umma_f16(d, at, b1, idesc, 1u);
            }
            ptx::umma_f16_ts(d, a1, b1, idesc, 1u);                                                 // M1 r1
          }
        }
        ptx::umma_commit(&meta->acc_full);
      }
      __syncwarp();
    }
    // ---------------------------------------------------- read-back: thread = channel, register = track
    // Only warp 0 polls (the batch above, then its own MMAs: a few hundred ns); the other three helper warps wait at a
    // hardware barrier, which costs no issue slots (four polling warps executed ~10 % of the kernel's instructions).
    // The barrier also hands on what warp 0 acquired from the producers (slot_track, fscale, pooled').
    if (hw == 0) ptx::mbar_wait(&meta->acc_full, (uint32_t)b & 1u, 103);
    ptx::tc_fence_before();
    ptx::named_bar_sync(6, HELPER_WARPS * 32);
    ptx::tc_fence_after();
    uint32_t d0[16], d1[16];
    ptx::tmem_ld_x16(lane_base + COL_D, d0);
    ptx::tmem_ld_x16(lane_base + COL_D + NB, d1);
    ptx::tmem_ld_wait_x16(d0);
    ptx::tmem_ld_wait_x16(d1);
    ptx::tc_fence_before();
    ptx::named_bar_sync(1, HELPER_WARPS * 32);           // the accumulator may be overwritten by the next batch
    const int ch = hw * 32 + lane;
    const float* pool = reinterpret_cast<const float*>(fz + OFF_POOL + buf * POOL_BYTES);
#pragma unroll
    for (int t = 0; t < NB; ++t) {
      if (t < cnt) {                                      // warp-uniform
        const int track = meta->slot_track[buf][t];
        const float f = meta->fscale[buf][t] * ms_inv;
        float* o = out_local + (size_t)track * D + ch;
        float p0, p1;
        if constexpr (POOL_SMEM) {
          p0 = pool[t * D + ch];
          p1 = pool[t * D + 128 + ch];
        } else {
          p0 = __ldcg(o);
          p1 = __ldcg(o + 128);
        }
        const float v0 = fmaf(f, __uint_as_float(d0[t]), p0), v1 = fmaf(f, __uint_as_float(d1[t]), p1);
        o[0] = v0;
        o[128] = v1;
        if (p.x_on) {
          if (mc) {
            // NVSwitch multicast: ONE store (a 128-byte line per warp) lands in every rank's q_all -- the switch
            // replicates it, the descriptors leave this GPU once instead of world - 1 times
            float* mo = p.x.q_all_mc + ((size_t)(xstep & 1u) * p.x.Q + (size_t)p.x_row0 + (size_t)track) * D + ch;
            mo[0] = v0;
            mo[128] = v1;
          } else if constexpr (POOL_SMEM) {               // the finished row replaces pooled' in the staging tile (see below)
            float* pw = reinterpret_cast<float*>(fz + OFF_POOL + buf * POOL_BYTES);
            pw[t * D + ch] = v0;
            pw[t * D + 128 + ch] = v1;
          } else {                                        // long tracks: plain stores into every peer's buffer (NVLink)
            const size_t off = ((size_t)(xstep & 1u) * p.x.Q + (size_t)p.x_row0 + (size_t)track) * D + ch;
            for (int r = 0; r < p.x.world; ++r) {
              if (r == p.x.rank) continue;
              float* po = p.x.q_all[r] + off;
              po[0] = v0;
              po[128] = v1;
            }
          }
        }
      }
    }
    if constexpr (POOL_SMEM) {
      // Sharded search without multicast: the batch's finished rows go to the other ranks as 1 KB bulk async copies
      // shared -> peer global (NVLink), one (track, destination) pair per helper thread: the copy engine does the
      // remote writes, no warp waits on NVLink write credits (plain stores from the four helper warps took ~40 us
      // for 13 MB at 8 GPUs).
      if (p.x_on && p.x.world > 1 && !mc) {
        ptx::fence_proxy_async_smem();                   // generic writes of the rows -> visible to the copy engine
        ptx::named_bar_sync(1, HELPER_WARPS * 32);       // all four channel quarters of every row are in place
        const int h = hw * 32 + lane, t = h >> 3, r = h & 7;
        if (t < cnt && r < p.x.world && r != p.x.rank) {
          const int track = meta->slot_track[buf][t];
          float* dst = p.x.q_all[r] + ((size_t)(xstep & 1u) * p.x.Q + (size_t)p.x_row0 + (size_t)track) * D;
          ptx::bulk_store_1d(dst, fz + OFF_POOL + buf * POOL_BYTES + t * (D * 4), D * 4);
        }
        ptx::bulk_commit();
        ptx::bulk_wait_read();                           // the tile may be refilled once the engine has read it
      }
    }
    __syncwarp();
    if (lane == 0) ptx::mbar_arrive(&meta->buf_free[buf]);
  }
  if constexpr (POOL_SMEM) {
    if (p.x_on && p.x.world > 1 && !mc) {                // this thread's remote rows are written before the CTA is counted
      ptx::bulk_wait_all();
      ptx::fence_proxy_async_all();
    }
  }
}

// one-time CTA set-up shared by both kernels: barriers, slot counter, tensor-memory allocation
template <int ARRIVALS>
__device__ __forceinline__ void fused_setup(uint8_t* fz, int warp, int helper0, int m_warps) {
  Meta* meta = reinterpret_cast<Meta*>(fz + OFF_META);
  if (threadIdx.x == 0) {
    for (int i = 0; i < 2; ++i) {
      ptx::mbar_init(&meta->tile_full[i], NB * ARRIVALS);
      ptx::mbar_init(&meta->buf_free[i], HELPER_WARPS);
    }
    ptx::mbar_init(&meta->acc_full, 1);
    ptx::mbar_init(&meta->m_ready, m_warps);
    meta->next_slot = 0u;
    ptx::fence_mbar_init();
  }
  if (warp == helper0) {
    ptx::tmem_alloc(&meta->tmem_base, 512);
    ptx::tmem_relinquish();
  }
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
}
__device__ __forceinline__ void fused_teardown(uint8_t* fz, int warp, int helper0) {
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == helper0) ptx::tmem_dealloc(reinterpret_cast<Meta*>(fz + OFF_META)->tmem_base, 512);
}

// a rank that has no tracks in a step still tells the others that its (empty) share of the descriptors is complete
__global__ void signal_only_kernel(const xchg::Exchange x) {
  xchg::signal_all(x, xchg::KIND_Q, xchg::current_step(x));
}

// ================================================================================================
// Short tracks (up to TR = 4 / 10 / 16 frames): one producer WARP per track.
// ================================================================================================
template <int TR>
struct Cfg;
// LOADER (TR = 10): the sixteenth warp issues the copies of every producer's next track instead of a twelfth producer.
// Handing a box to the copy engine costs the issuing warp 400-900 cycles (it queues behind the other warps' boxes;
// 1,400-1,500 cycles as per-frame copies) -- 15 % of a producer's iteration when the producers issue their own.
// A seventeenth warp is not an option: the register file is four files of 16 K, one per scheduler, a fifth warp on one
// of them caps the launch count at 96 registers and the producers at 128 (they hold 80 of frames + 32 of weights).
template <>
struct Cfg<4> { static constexpr int NW = 16, SLOTS = 2, LOADER = 0, REGS_P = 104, REGS_H = 56; };   // the pool holds what the helpers release
template <>
struct Cfg<10> { static constexpr int NW = 11, SLOTS = 1, LOADER = 1, REGS_P = 152, REGS_H = 56; };
template <>
struct Cfg<16> { static constexpr int NW = 8, SLOTS = 1, LOADER = 0, REGS_P = 224, REGS_H = 56; };

// In: the element type of the tracks (float or __half); only the track buffers and the copies into them depend on it
template <int TR, typename In>
constexpr size_t warp_smem_bytes() {
  return 1024 + fused_bytes<true>() + (size_t)Cfg<TR>::NW * Cfg<TR>::SLOTS * TR * D * sizeof(In)   // track buffers
         + (size_t)Cfg<TR>::NW * 64 * 4                                                   // per-warp scalars
         + (size_t)Cfg<TR>::NW * Cfg<TR>::SLOTS * 8                                       // mbarriers
         + (size_t)Cfg<TR>::NW * 8                                                        // "buffer is free" mbarriers
         + (size_t)Cfg<TR>::NW * Cfg<TR>::SLOTS * 4;                                      // track lengths
}
template <int TR>
constexpr int warp_threads() { return (Cfg<TR>::NW + HELPER_WARPS + Cfg<TR>::LOADER) * 32; }

template <int TR, typename In>
__global__ void __launch_bounds__((Cfg<TR>::NW + HELPER_WARPS + Cfg<TR>::LOADER) * 32, 1)
aggregate_fused_warp_kernel(const __grid_constant__ CUtensorMap tmSeq, const Params p) {
  constexpr int NW = Cfg<TR>::NW, SLOTS = Cfg<TR>::SLOTS;
  constexpr bool LOADER = Cfg<TR>::LOADER != 0;
  static_assert(!LOADER || SLOTS == 1, "the loader warp serves single-buffer producers");
  constexpr int M_INFLIGHT = TR >= 10 ? 4 : 2;     // chunks of M a producer warp has in flight at start
  constexpr uint32_t FRAME_BYTES = D * sizeof(In);
  constexpr size_t XBUF_BYTES = (size_t)NW * SLOTS * TR * FRAME_BYTES;   // every producer's track buffers
  const In* const seq = static_cast<const In*>(p.seq);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* fz = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);        // fused area (1 KB aligned), then producers
  uint8_t* pz = fz + fused_bytes<true>();
  const int lane = threadIdx.x & 31;
  const int warp = __shfl_sync(ptx::FULL_MASK, threadIdx.x >> 5, 0);
  Meta* meta = reinterpret_cast<Meta*>(fz + OFF_META);
  const uint32_t xstep = p.x_on ? xchg::current_step(p.x) : 0u;
  float* const out_local = local_out(p, xstep);

  const long long stride = (long long)gridDim.x * NW;
  const long long first0 = (long long)blockIdx.x * NW;

  In* xbuf = reinterpret_cast<In*>(pz) + (size_t)(warp < NW ? warp : 0) * SLOTS * TR * D;
  float* scal = reinterpret_cast<float*>(pz + XBUF_BYTES) + (warp < NW ? warp : 0) * 64;
  uint64_t* bars = reinterpret_cast<uint64_t*>(pz + XBUF_BYTES + (size_t)NW * 64 * 4) +
                   (warp < NW ? warp : 0) * SLOTS;
  int* slot_len = reinterpret_cast<int*>(pz + XBUF_BYTES + (size_t)NW * 64 * 4 +
                                         (size_t)NW * SLOTS * 8 + (size_t)NW * 8) + (warp < NW ? warp : 0) * SLOTS;
  // loader's view: every producer's buffer, barriers and track length
  In* const xbuf_all = reinterpret_cast<In*>(pz);
  uint64_t* const bars_all = reinterpret_cast<uint64_t*>(pz + XBUF_BYTES + (size_t)NW * 64 * 4);
  uint64_t* const empty_all = bars_all + NW * SLOTS;                                    // producer -> loader: frames are in registers
  int* const slot_len_all = reinterpret_cast<int*>(empty_all + NW);
  if (warp < NW && lane == 0) {
    for (int i = 0; i < SLOTS; ++i) ptx::mbar_init(&bars[i], 1);
    ptx::mbar_init(&empty_all[warp], 1);
    ptx::fence_mbar_init();
  }
  __syncwarp();
  const int Tmax = p.Tmax;
  const long long first = first0 + warp;
  const uint64_t pol = ptx::policy_evict_first();       // frames are read exactly once

  // A track's length comes from lens[] or from its mask row.  peek() only issues that (dependent) load --
  // one track ahead of its use -- and issue() turns the loaded word into the length and starts the copies.
  auto peek = [&](long long track) -> int {
    if (track >= p.Q) return 0;
    if (p.lens) return p.lens[track];
    if (p.mask) return lane <= Tmax ? (int)p.mask[(size_t)track * (1 + Tmax) + lane] : 0;
    return 0;
  };
  auto issue = [&](long long track, int slot, int raw) {
    int len = 0;
    if (track < p.Q) {
      if (p.lens) {
        len = raw;
      } else if (p.mask) {
        // first nonzero of the mask row ends the track; row 0 is the dummy (models/match_head.py:136-139)
        const uint32_t b = __ballot_sync(ptx::FULL_MASK, raw != 0);
        const int end = b ? __ffs(b) - 1 : 1 + Tmax;
        len = end - 1;
      } else {
        len = Tmax;
      }
      len = max(0, min(len, Tmax));
    }
    if (lane == 0) {
      slot_len[slot] = len;
      if (len > 0) ptx::mbar_arrive_expect_tx(&bars[slot], (uint32_t)len * FRAME_BYTES);
      else ptx::mbar_arrive(&bars[slot]);
    }
    __syncwarp();
    if (TR >= 10 && p.use_tm && len == TR) {          // (measured: +4.5 % at 10 frames, +10 % at 16, -7 % at 4)
      // a full track: frames 1..TR of this track as ONE box {256 channels, 1 track, TR frames} (the per-frame loop
      // below costs ~8 instructions and a branch per frame: uniform-datapath copies issued lane by lane)
      if (ptx::elect_one()) ptx::tma_load_3d_hint(xbuf + (size_t)slot * TR * D, &tmSeq, &bars[slot], 0, (int)track, 1, pol);
      __syncwarp();
    } else if (lane < len) {
      const In* src = seq + (long long)(lane + 1) * p.frame_stride + track * p.track_stride;
      ptx::bulk_load_1d_hint(xbuf + ((size_t)slot * TR + lane) * D, src, FRAME_BYTES, &bars[slot], pol);
    }
  };

  // the first tracks are requested before anything else happens in this CTA (barrier set-up, tensor-memory
  // allocation, register re-balancing and a cold instruction cache cost ~3 us)
  constexpr int AHEAD = SLOTS == 1 ? 1 : SLOTS - 1;     // tracks in flight ahead of the one being processed
  int raw_next = 0;
  if (warp < NW) {
#pragma unroll 1
    for (int i = 0; i < AHEAD; ++i) issue(first + i * stride, i, peek(first + i * stride));
    raw_next = peek(first + (long long)AHEAD * stride);
  }
  fused_setup<1>(fz, warp, NW, NW + HELPER_WARPS + Cfg<TR>::LOADER);

  if (LOADER && warp == NW + HELPER_WARPS) {
    // ------------------------------------------------------------------------------ loader warp: lane w serves producer w
    load_m_tmem<NW + HELPER_WARPS + 1, 2>(p, meta, warp, lane);   // its share of M first: sixteen warps fill tensor memory
    auto lane_len = [&](long long track) -> int {       // one lane scans the mask row (independent byte loads)
      int len;
      if (p.lens) {
        len = p.lens[track];
      } else if (p.mask) {
        const uint8_t* m = p.mask + (size_t)track * (1 + Tmax);
        int end = 1 + Tmax;
        for (int i = Tmax; i >= 0; --i)
          if (m[i] != 0) end = i;                       // first nonzero ends the track (models/match_head.py:136-139)
        len = end - 1;
      } else {
        len = Tmax;
      }
      return max(0, min(len, Tmax));
    };
    long long next = first0 + lane + stride;            // the producer's second track (it requested the first itself)
    uint32_t ph = 0u;
    bool active = lane < NW && next < p.Q;
    int len_next = active ? lane_len(next) : 0;
    uint64_t t0 = 0;
    while (__any_sync(ptx::FULL_MASK, active)) {
      const bool ready = active && ptx::mbar_test_wait(&empty_all[lane < NW ? lane : 0], ph);
      if (ready) {
        uint64_t* bar = &bars_all[lane];
        In* dst = xbuf_all + (size_t)lane * TR * D;
        slot_len_all[lane] = len_next;
        if (len_next > 0) ptx::mbar_arrive_expect_tx(bar, (uint32_t)len_next * FRAME_BYTES);
        else ptx::mbar_arrive(bar);
        if (TR >= 10 && p.use_tm && len_next == TR) {
          ptx::tma_load_3d_hint(dst, &tmSeq, bar, 0, (int)next, 1, pol);
        } else {
          for (int t = 0; t < len_next; ++t)
            ptx::bulk_load_1d_hint(dst + (size_t)t * D, seq + (long long)(t + 1) * p.frame_stride + next * p.track_stride,
                                   FRAME_BYTES, bar, pol);
        }
        next += stride;
        ph ^= 1u;
        active = next < p.Q;
        len_next = active ? lane_len(next) : 0;
      }
      if (!__any_sync(ptx::FULL_MASK, ready)) {
        __nanosleep(100);
        const uint64_t now = ptx::globaltimer_ns();     // watchdog: a protocol error traps instead of hanging
        if (t0 == 0) t0 = now;
        else if (now - t0 > 2000000000ull) ptx::watchdog_trap(109u, ptx::smem_u32(&empty_all[lane < NW ? lane : 0]), ph);
      } else {
        t0 = 0;
      }
    }
  } else if (warp >= NW) {
    ptx::reg_dec<Cfg<TR>::REGS_H>();
    // a warp reaches the tensor-memory lanes of ITS quarter (warp % 4): that is the helper's index
    load_m_tmem<NW + HELPER_WARPS + Cfg<TR>::LOADER, 2>(p, meta, warp, lane);
    helper_role<1, true>(p, fz, warp & 3, lane, NW, first0, stride, out_local, xstep);
  } else {
    ptx::reg_inc<Cfg<TR>::REGS_P>();
    load_m_tmem<NW + HELPER_WARPS + Cfg<TR>::LOADER, M_INFLIGHT>(p, meta, warp, lane);   // while the first frames are in flight

    const float* fold = p.fold;
    const Vec8 ut = load_vec8(fold + Fold::U_THETA, lane);
    const Vec8 up = load_vec8(fold + Fold::U_PHI, lane);
    const Vec8 ug = load_vec8(fold + Fold::U_G, lane);
    const Vec8 wa = load_vec8(fold + Fold::W_A, lane);
    const float c_s = fold[Fold::CONSTS + 3];
    // scalar layout per frame: [a, d, b, c]; constants c_theta, 0, c_phi, c_g
    const int comp = lane & 3;
    const float my_const = comp == 0 ? fold[Fold::CONSTS + 0] : comp == 2 ? fold[Fold::CONSTS + 1]
                         : comp == 3 ? fold[Fold::CONSTS + 2] : 0.f;

    int it = 0;
#pragma unroll 1
    for (long long track = first; track < p.Q; track += stride, ++it) {
      const int slot = it % SLOTS;
      const uint32_t phase = (uint32_t)(it / SLOTS) & 1u;
      if constexpr (SLOTS > 1) {
        __syncwarp();                                  // every lane is done with the slot being refilled
        issue(track + (long long)(SLOTS - 1) * stride, (it + SLOTS - 1) % SLOTS, raw_next);
        raw_next = peek(track + (long long)SLOTS * stride);
      }
      ptx::mbar_wait(&bars[slot], phase, 105);
      const int len = slot_len[slot];
      const In* xs = xbuf + (size_t)slot * TR * D;

      // One body, two instantiations: tracks with all TR frames (the common case) run without
      // per-frame guards and with unrolled T x T loops.
      auto process = [&](auto full_tag) {
        constexpr bool FULL = decltype(full_tag)::value;
        // ---- frames -> registers, four dots per frame; every 4 frames a transposing butterfly leaves
        // the 16 totals (a, d, b, c of 4 frames) in lanes 0..15
        // the track's slot in the batch under construction: the shared-memory atomic's round trip (~200 cycles) is
        // started here and used after the weighted sums
        unsigned ticket = 0u;
        if (lane == 0) ticket = atomicAdd(&meta->next_slot, 1u);
        Vec8 x[TR];
#pragma unroll
        for (int t0 = 0; t0 < TR; t0 += 8) {            // 8 frames = 32 totals per butterfly: the 5 dependent shuffle rounds
          const int nf = TR - t0 < 8 ? TR - t0 : 8;     // of a butterfly are the phase's latency (compile time after unrolling)
          float acc[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) acc[i] = 0.f;
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int t = t0 + u;
            if (u < nf) {
              if (FULL || t < len) x[t] = load_frame(xs + t * D, lane);
              else x[t] = zero_vec8();
              acc[4 * u + 0] = dot8(x[t], ut);
              acc[4 * u + 1] = dot8(x[t], wa);
              acc[4 * u + 2] = dot8(x[t], up);
              acc[4 * u + 3] = dot8(x[t], ug);
            }
          }
          float tot;
          if (nf > 4) {
            tot = treduce<32>(acc, lane);
          } else if (nf > 2) {
            float a16[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) a16[i] = acc[i];
            tot = treduce<16>(a16, lane);
          } else {
            float a8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) a8[i] = acc[i];
            tot = treduce<8>(a8, lane);
          }
          if (lane < 4 * nf) scal[4 * t0 + lane] = tot + my_const;
        }
        if constexpr (SLOTS == 1) {
          __syncwarp();                                // all lanes hold their frames in registers:
          if constexpr (LOADER) {
            if (lane == 0) ptx::mbar_arrive(&empty_all[warp]);   // the loader warp may refill the buffer
          } else {
            issue(track + stride, 0, raw_next);        // no loader warp (TR = 16): the producer refills it itself
            raw_next = peek(track + 2 * stride);
          }
        }
        __syncwarp();

        // ---- attention over the track's frames (lane = frame)
        const int L = FULL ? TR : len;
        const bool valid = lane < L;
        const bool many = FULL ? TR > 1 : len > 1;
        const float inv_len = FULL ? 1.f / (float)TR : (len > 0 ? 1.f / (float)len : 0.f);
        float4 sc = make_float4(0.f, 0.f, 0.f, 0.f);
        if (valid) sc = *reinterpret_cast<const float4*>(scal + 4 * lane);   // a, d, b, c of my frame
        float sum = 0.f;
        if (many) {
#pragma unroll
          for (int j = 0; j < (FULL ? TR : len); ++j) {
            const float2 bc = *reinterpret_cast<const float2*>(scal + 4 * j + 2);
            sum = fmaf(fmaxf(sc.x + bc.x, 0.f) * inv_len, bc.y, sum);
          }
        }
        const float s_t = valid ? sc.y + sum + c_s : -INFINITY;
        const float m = ptx::warp_max(s_t);
        const float e_t = valid ? expf(s_t - m) : 0.f;
        __syncwarp();                                    // all lanes have read b, c, d
        if (lane < TR) scal[4 * lane + 1] = e_t;         // d -> e
        __syncwarp();
        // One loop gives the softmax denominator (every lane sums the e_t itself: no reduction) and the second
        // interaction q_j = sum_t p_t relu(a_t + b_j) / T, p_t = e_t / z.
        float z = 0.f, q_j = 0.f;
#pragma unroll
        for (int t = 0; t < (FULL ? TR : len); ++t) {
          const float2 ae = *reinterpret_cast<const float2*>(scal + 4 * t);
          z += ae.y;
          q_j = fmaf(ae.y, fmaxf(ae.x + sc.z, 0.f), q_j);
        }
        const float inv_z = z > 0.f ? 1.f / z : 0.f;
        const float p_t = e_t * inv_z;
        q_j = (many && valid) ? q_j * inv_len * inv_z : 0.f;
        __syncwarp();                                    // all lanes have read the a_t, e_t
        if (lane < TR) *reinterpret_cast<float4*>(scal + 4 * lane) = make_float4(p_t, p_t, q_j, q_j);
        if (p.att && lane < Tmax) p.att[(size_t)track * Tmax + lane] = p_t;
        __syncwarp();

        // ---- weighted sums over frames, 8 channels per lane; sum_j q_j on the way (every lane adds the broadcast q)
        Vec8 pov = zero_vec8(), rv = zero_vec8();
        float qsum = 0.f;
#pragma unroll
        for (int t = 0; t < TR; ++t) {
          if (FULL || t < len) {
            const ulonglong2 pq = *reinterpret_cast<const ulonglong2*>(scal + 4 * t);   // {p,p}, {q,q}
            fma8(pov, pq.x, x[t]);
            fma8(rv, pq.y, x[t]);
            qsum += __uint_as_float((uint32_t)(pq.y & 0xffffffffull));
          }
        }
        float4 po0, po1, r0, r1;
        unpack_vec8(pov, po0, po1);
        unpack_vec8(rv, r0, r1);
        if (many) {
          const float4 wbg0 = *reinterpret_cast<const float4*>(fold + Fold::WBG + 4 * lane);
          const float4 wbg1 = *reinterpret_cast<const float4*>(fold + Fold::WBG + 128 + 4 * lane);
          const float4 bw0 = *reinterpret_cast<const float4*>(fold + Fold::BW + 4 * lane);
          const float4 bw1 = *reinterpret_cast<const float4*>(fold + Fold::BW + 128 + 4 * lane);
          po0.x += fmaf(qsum, wbg0.x, bw0.x);
          po0.y += fmaf(qsum, wbg0.y, bw0.y);
          po0.z += fmaf(qsum, wbg0.z, bw0.z);
          po0.w += fmaf(qsum, wbg0.w, bw0.w);
          po1.x += fmaf(qsum, wbg1.x, bw1.x);
          po1.y += fmaf(qsum, wbg1.y, bw1.y);
          po1.z += fmaf(qsum, wbg1.z, bw1.z);
          po1.w += fmaf(qsum, wbg1.w, bw1.w);
        }
        // ---- publish: pooled' (fp32) and r (two fp16 terms) into the batch under construction
        float mx = fmaxf(fmaxf(fmaxf(fabsf(r0.x), fabsf(r0.y)), fmaxf(fabsf(r0.z), fabsf(r0.w))),
                         fmaxf(fmaxf(fabsf(r1.x), fabsf(r1.y)), fmaxf(fabsf(r1.z), fabsf(r1.w))));
        mx = ptx::warp_max(mx);
        float inv;
        const float s = track_scale(mx, &inv);
        const Slot sl = wait_slot(meta, __shfl_sync(ptx::FULL_MASK, ticket, 0));
        uint8_t* rt = fz + OFF_RT + sl.buf * RT_BYTES;
        store_r4(rt, sl.pos, 4 * lane, r0, s);
        store_r4(rt, sl.pos, 128 + 4 * lane, r1, s);
        float* pool = reinterpret_cast<float*>(fz + OFF_POOL + sl.buf * POOL_BYTES) + sl.pos * D;
        *reinterpret_cast<float4*>(pool + 4 * lane) = po0;
        *reinterpret_cast<float4*>(pool + 128 + 4 * lane) = po1;
        if (lane == 0) {
          meta->slot_track[sl.buf][sl.pos] = (int)track;
          meta->fscale[sl.buf][sl.pos] = inv;
        }
        ptx::fence_proxy_async_smem();                   // the r rows are read by the tensor core (async proxy)
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&meta->tile_full[sl.buf]);
      };
      if (len == TR) process(std::true_type{});
      else process(std::false_type{});
    }
  }
  fused_teardown(fz, warp, NW);
  if (p.x_on && p.x_last) xchg::signal_all(p.x, xchg::KIND_Q, xstep);
}


// ================================================================================================
// Long tracks (17..64 frames): a GROUP of GW = 2 / 4 producer warps per track, 16 frames per warp.
// What crosses the warps of a group goes through a few hundred bytes of shared memory and five
// named barriers per track: the per-frame scalars (a, d, b, c), the softmax maximum and denominator,
// the partial weighted sums.  pooled' goes to global memory (the descriptor row itself) and is picked
// up again from L2 by the helpers: no room for a shared-memory copy next to 128 KB of frame buffers.
// ================================================================================================
constexpr int FB = 16;                 // frames per warp
constexpr int GWARPS = 8;              // producer warps per CTA
constexpr int GTHREADS = (GWARPS + HELPER_WARPS) * 32;
constexpr int GREGS_P = 224, GREGS_H = 56;

template <int GW>
struct alignas(16) GroupSmem {
  float ad[FB * GW / 2][4];            // per pair of frames: a_even, a_odd, d_even -> p_even, d_odd -> p_odd
  float bc[FB * GW / 2][4];            // b_even, b_odd, c_even, c_odd (zero for frames past the track's end)
  float pq[FB * GW][4];                // per frame: p, p, q, q
  float part[GW][2 * D];               // per warp: partial pooled | partial r
  float red_max[GW];
  float red_sum[GW];
  float red_q[GW];
  float red_rmax[GW];
  unsigned int slot;
  float pad[3];
};
template <int GW, typename In>
struct GSmem {
  In x[GWARPS][FB][D];                 // 8 x 16 KB (fp32) / 8 x 8 KB (fp16)
  GroupSmem<GW> g[GWARPS / GW];
  uint64_t bar[GWARPS];
};
template <int GW, typename In>
constexpr size_t group_smem_bytes() { return 1024 + fused_bytes<false>() + sizeof(GSmem<GW, In>); }

template <int GW, typename In>
__global__ void __launch_bounds__(GTHREADS, 1)
aggregate_fused_group_kernel(const __grid_constant__ CUtensorMap tmSeq, const Params p) {
  constexpr int GROUPS_PER_CTA = GWARPS / GW;
  constexpr uint32_t FRAME_BYTES = D * sizeof(In);
  const In* const seq = static_cast<const In*>(p.seq);
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = ptx::smem_u32(smem_raw);
  uint8_t* fz = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  GSmem<GW, In>& s = *reinterpret_cast<GSmem<GW, In>*>(fz + fused_bytes<false>());
  const int lane = threadIdx.x & 31;
  const int warp = __shfl_sync(ptx::FULL_MASK, threadIdx.x >> 5, 0);
  Meta* meta = reinterpret_cast<Meta*>(fz + OFF_META);
  const uint32_t xstep = p.x_on ? xchg::current_step(p.x) : 0u;
  float* const out_local = local_out(p, xstep);
  const long long stride = (long long)gridDim.x * GROUPS_PER_CTA;
  const long long first0 = (long long)blockIdx.x * GROUPS_PER_CTA;

  if (warp < GWARPS && lane == 0) {
    ptx::mbar_init(&s.bar[warp], 1);
    ptx::fence_mbar_init();
  }
  __syncwarp();
  const int pw = warp < GWARPS ? warp : 0;            // helper warps never use what follows
  const int grp = pw / GW, wg = pw % GW;
  GroupSmem<GW>& gs = s.g[grp];
  In* xs = &s.x[pw][0][0];
  uint64_t* bar = &s.bar[pw];
  const int Tmax = p.Tmax;
  const uint32_t bar_id = 2 + grp;                     // named barrier 1 belongs to the helpers
  const long long first = first0 + grp;
  const uint64_t pol = ptx::policy_evict_first();

  // length of a track (every warp of the group derives it on its own).  peek() only issues the (dependent) loads --
  // one track ahead of their use, so that their latency hides behind the current track's dots -- and decode() turns
  // the loaded words into the length.
  auto peek = [&](long long track) -> uint32_t {
    if (track >= p.Q) return 0u;
    if (p.lens) return (uint32_t)p.lens[track];
    if (p.mask) {
      const uint8_t* m = p.mask + (size_t)track * (1 + Tmax);
      const uint32_t m0 = lane <= Tmax ? m[lane] : 0u;
      const uint32_t m1 = 32 + lane <= Tmax ? m[min(32 + lane, Tmax)] : 0u;
      const uint32_t m2 = lane == 0 && Tmax >= 64 ? m[min(64, Tmax)] : 0u;
      return m0 | (m1 << 8) | (m2 << 16);
    }
    return 0u;
  };
  auto decode = [&](long long track, uint32_t raw) -> int {
    if (track >= p.Q) return 0;
    int len;
    if (p.lens) {
      len = (int)raw;
    } else if (p.mask) {
      // first nonzero of the mask row ends the track; row 0 is the dummy (models/match_head.py:136-139)
      const uint32_t b0 = __ballot_sync(ptx::FULL_MASK, (raw & 0xffu) != 0u);
      const uint32_t b1 = __ballot_sync(ptx::FULL_MASK, (raw & 0xff00u) != 0u);
      const uint32_t b2 = __ballot_sync(ptx::FULL_MASK, (raw & 0xff0000u) != 0u);
      const int end = b0 ? __ffs(b0) - 1 : b1 ? 32 + __ffs(b1) - 1 : b2 ? 64 : 1 + Tmax;
      len = end - 1;
    } else {
      len = Tmax;
    }
    return max(0, min(len, Tmax));
  };
  // start the copies of this warp's frame block of one track.  Frames past the block's end are read as ZEROS from the
  // buffer (the dots and the weighted sums run unguarded, straight-line): whenever a block is shorter than the one
  // the buffer held before, the stale frames in between are cleared first.
  int nw_buf = FB;                     // frames of the buffer that may hold something else than zeros
  auto issue = [&](long long track, int len) {
    const int nw = max(0, min(len - FB * wg, FB));
    if (nw < nw_buf) {                 // warp-uniform
      float4* z = reinterpret_cast<float4*>(xs + (size_t)nw * D);   // 16-byte chunks of zeros
      for (int i = lane; i < (nw_buf - nw) * (int)(FRAME_BYTES / 16); i += 32) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      ptx::fence_proxy_async_smem();   // these generic-proxy writes come before any later copy into the same bytes
    }
    nw_buf = nw;
    if (lane == 0) {
      if (nw > 0) ptx::mbar_arrive_expect_tx(bar, (uint32_t)nw * FRAME_BYTES);
      else ptx::mbar_arrive(bar);
    }
    __syncwarp();
    if (p.use_tm && nw == FB) {
      // a full block: frames FB wg + 1 .. FB wg + 16 of this track as ONE box {256 channels, 1 track, 16 frames}
      // (the per-frame loop below is ~10 instructions and a branch per frame: uniform-datapath copies issued lane by lane)
      if (ptx::elect_one()) ptx::tma_load_3d_hint(xs, &tmSeq, bar, 0, (int)track, FB * wg + 1, pol);
      __syncwarp();
    } else if (lane < nw) {
      const In* src = seq + (long long)(FB * wg + lane + 1) * p.frame_stride + track * p.track_stride;
      ptx::bulk_load_1d_hint(xs + (size_t)lane * D, src, FRAME_BYTES, bar, pol);
    }
  };
  // the first track is requested before the CTA-wide set-up
  int len = 0;
  if (warp < GWARPS) {
    len = decode(first, peek(first));
    issue(first, len);
  }
  fused_setup<GW>(fz, warp, GWARPS, GWARPS + HELPER_WARPS);

  if (warp >= GWARPS) {
    ptx::reg_dec<GREGS_H>();
    load_m_tmem<GWARPS + HELPER_WARPS, 2>(p, meta, warp, lane);
    helper_role<GW, false>(p, fz, warp - GWARPS, lane, GROUPS_PER_CTA, first0, stride, out_local, xstep);
  } else {
    ptx::reg_inc<GREGS_P>();
    const float* fold = p.fold;
    const Vec8 ut = load_vec8(fold + Fold::U_THETA, lane);
    const Vec8 up = load_vec8(fold + Fold::U_PHI, lane);
    const Vec8 ug = load_vec8(fold + Fold::U_G, lane);
    const Vec8 wa = load_vec8(fold + Fold::W_A, lane);
    const float c_s = fold[Fold::CONSTS + 3];
    const int comp = lane & 3;
    const float my_const = comp == 0 ? fold[Fold::CONSTS + 0] : comp == 2 ? fold[Fold::CONSTS + 1]
                         : comp == 3 ? fold[Fold::CONSTS + 2] : 0.f;
    // where this lane's butterfly total (component comp of frame SF0 + t0) goes: the T x T loops read PAIRS of frames
    const int SF0 = FB * wg + (lane >> 2);
    float* const sc_dst = (comp < 2 ? &gs.ad[0][0] : &gs.bc[0][0]) + (SF0 >> 1) * 4 + ((comp & 1) << 1) + (SF0 & 1);

    load_m_tmem<GWARPS + HELPER_WARPS, 2>(p, meta, warp, lane);   // while the first frames are in flight
    int it = 0;
#pragma unroll 1
    for (long long track = first; track < p.Q; track += stride, ++it) {
      ptx::mbar_wait(bar, (uint32_t)it & 1u, 106);
      const int nw = max(0, min(len - FB * wg, FB));

      // ---- my 16 frames -> registers (zeros past the block's end), four dots per frame, the 32 totals of 8 frames per
      // butterfly (five dependent shuffle rounds per 8 frames instead of per 4: the rounds are the phase's latency)
      const uint32_t raw_next = peek(track + stride);
      Vec8 x[FB];
#pragma unroll
      for (int t0 = 0; t0 < FB; t0 += 8) {
        float acc[32];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int t = t0 + u;
          x[t] = load_frame(xs + t * D, lane);
          acc[4 * u + 0] = dot8(x[t], ut);
          acc[4 * u + 1] = dot8(x[t], wa);
          acc[4 * u + 2] = dot8(x[t], up);
          acc[4 * u + 3] = dot8(x[t], ug);
        }
        const float tot = treduce<32>(acc, lane);
        // frame F = FB wg + t0 + (lane >> 2): a, d -> ad[F / 2][F % 2 (+ 2)], b, c -> bc[...], zero past the track's end
        sc_dst[2 * t0] = (comp < 2 || SF0 + t0 < len) ? tot + my_const : 0.f;
      }
      // the buffer is free again: fetch this warp's block of the group's next track
      const int len_next = decode(track + stride, raw_next);
      __syncwarp();
      issue(track + stride, len_next);
      ptx::named_bar_sync(bar_id, GW * 32);                       // #1 all scalars of the track are visible
      // the track's slot in the batch under construction is claimed now, its (~200 cycle) round trip used much later
      unsigned my_slot = 0u;
      if (wg == 0 && lane == 0) my_slot = atomicAdd(&meta->next_slot, 1u);

      // ---- attention over the track's frames: lane = (frame f of my block, half of the j / t range).  The loops
      // take two frames per step ({b_e, b_o, c_e, c_o}: one 16-byte load, one packed add, one packed fma) and run over
      // ALL FB GW frames without bounds (straight-line code): past the track's end c, and later e, are zero.  The 1/T
      // factor is applied once at the end.
      const int f = lane & 15, half = lane >> 4;
      const int F = FB * wg + f;
      const bool valid = F < len;
      const float inv_len = len > 0 ? 1.f / (float)len : 0.f;
      const float a_f = gs.ad[F >> 1][F & 1], d_f = gs.ad[F >> 1][2 + (F & 1)], b_f = gs.bc[F >> 1][F & 1];
      // sum over the 8 pairs of block w this lane's half takes: relu(own + tab.x) * tab.y; *ysum += sum of tab.y
      auto block_sum = [&](const u64 o2, const float (*tab)[4], int w, u64* ysum) -> float {
        u64 acc_a = 0ull, acc_b = 0ull;
#pragma unroll
        for (int i = 0; i < FB / 2; i += 4) {
          const ulonglong2 v0 = *reinterpret_cast<const ulonglong2*>(&tab[(FB / 2) * w + i + half][0]);
          const ulonglong2 v1 = *reinterpret_cast<const ulonglong2*>(&tab[(FB / 2) * w + i + 2 + half][0]);
          float s0, s1, s2, s3;
          upk(add2(o2, v0.x), s0, s1);
          upk(add2(o2, v1.x), s2, s3);
          acc_a = fma2(pk(fmaxf(s0, 0.f), fmaxf(s1, 0.f)), v0.y, acc_a);
          acc_b = fma2(pk(fmaxf(s2, 0.f), fmaxf(s3, 0.f)), v1.y, acc_b);
          if (ysum) *ysum = add2(*ysum, add2(v0.y, v1.y));
        }
        float lo, hi, lo2, hi2;
        upk(acc_a, lo, hi);
        upk(acc_b, lo2, hi2);
        return (lo + hi) + (lo2 + hi2);
      };
      float sum = 0.f;
      if (len > 1) {
        const u64 a2 = pk(a_f, a_f);
#pragma unroll
        for (int w = 0; w < GW; ++w) sum += block_sum(a2, gs.bc, w, nullptr);
        sum += __shfl_xor_sync(ptx::FULL_MASK, sum, 16);
        sum *= inv_len;
      }
      const float s_t = valid ? d_f + sum + c_s : -INFINITY;
      // Softmax over the track with ONE barrier and no second pass over p: every warp publishes the maximum m_w of its
      // block and e_t = exp(s_t - m_w) for its frames.  After the barrier m = max_w m_w; the second interaction sums
      // e_t block by block -- and the e_t themselves on the way: z = sum_w exp(m_w - m) sum_{t in w} e_t, no reduction
      // of its own -- scaling each block's sums by exp(m_w - m); p_t = e_t exp(m_w - m) / z.
      const float m_w = ptx::warp_max(s_t);
      const float e_t = valid ? expf(s_t - m_w) : 0.f;
      if (half == 0) gs.ad[F >> 1][2 + (F & 1)] = e_t;            // d (read above by both lanes of the frame) -> e
      if (lane == 0) gs.red_max[wg] = m_w;
      ptx::named_bar_sync(bar_id, GW * 32);                       // #2 e and m_w of the whole track are visible
      float m = gs.red_max[0];
#pragma unroll
      for (int w = 1; w < GW; ++w) m = fmaxf(m, gs.red_max[w]);
      float scale[GW];
#pragma unroll
      for (int w = 0; w < GW; ++w) {
        const float mw = gs.red_max[w];
        scale[w] = mw > -INFINITY ? expf(mw - m) : 0.f;            // a warp without frames of this track: -inf
      }
      float q_j = 0.f, z = 0.f;                                    // q_j = sum_t relu(b_j + a_t) p_t / T
      {
        const u64 b2 = pk(b_f, b_f);
#pragma unroll
        for (int w = 0; w < GW; ++w) {
          u64 ys = 0ull;
          q_j = fmaf(block_sum(b2, gs.ad, w, &ys), scale[w], q_j);
          float y0, y1;
          upk(ys, y0, y1);
          z = fmaf(y0 + y1, scale[w], z);
        }
        q_j += __shfl_xor_sync(ptx::FULL_MASK, q_j, 16);
        z += __shfl_xor_sync(ptx::FULL_MASK, z, 16);
      }
      const float inv_z = z > 0.f ? 1.f / z : 0.f;
      const float p_t = e_t * scale[wg] * inv_z;
      q_j = len > 1 ? q_j * inv_len * inv_z : 0.f;
      if (p.att && half == 0 && F < Tmax) p.att[(size_t)track * Tmax + F] = p_t;
      if (!valid) q_j = 0.f;
      const float qsum_w = ptx::warp_sum(half == 0 ? q_j : 0.f);
      if (half == 0) *reinterpret_cast<float4*>(&gs.pq[F][0]) = make_float4(p_t, p_t, q_j, q_j);
      __syncwarp();

      // ---- partial weighted sums over my frames, 8 channels per lane.  {p, p}, {q, q} come from shared memory (one
      // broadcast load per frame, four in flight); frames past the block's end are zero in registers and need no guard.
      Vec8 pov = zero_vec8(), rv = zero_vec8();
#pragma unroll
      for (int t0 = 0; t0 < FB; t0 += 4) {
        ulonglong2 w2[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) w2[u] = *reinterpret_cast<const ulonglong2*>(&gs.pq[FB * wg + t0 + u][0]);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          fma8(pov, w2[u].x, x[t0 + u]);
          fma8(rv, w2[u].y, x[t0 + u]);
        }
      }
      float4 po0, po1, r0, r1;
      unpack_vec8(pov, po0, po1);
      unpack_vec8(rv, r0, r1);
      {
        float* pw = &gs.part[wg][0];
        *reinterpret_cast<float4*>(pw + 4 * lane) = po0;
        *reinterpret_cast<float4*>(pw + 128 + 4 * lane) = po1;
        *reinterpret_cast<float4*>(pw + D + 4 * lane) = r0;
        *reinterpret_cast<float4*>(pw + D + 128 + 4 * lane) = r1;
        // the sum of the warps' partial maxima bounds max |r|: it fixes the track's fp16 scale
        float pm = fmaxf(fmaxf(fmaxf(fabsf(r0.x), fabsf(r0.y)), fmaxf(fabsf(r0.z), fabsf(r0.w))),
                         fmaxf(fmaxf(fabsf(r1.x), fabsf(r1.y)), fmaxf(fabsf(r1.z), fabsf(r1.w))));
        pm = ptx::warp_max(pm);
        if (lane == 0) {
          gs.red_q[wg] = qsum_w;
          gs.red_rmax[wg] = pm;
          if (wg == 0) gs.slot = my_slot;
        }
      }
      ptx::named_bar_sync(bar_id, GW * 32);                       // #5 partial sums, maxima and the slot are visible

      // ---- warp w finishes channels [CW w, CW (w+1)), CW = 256 / GW, and publishes them
      {
        const unsigned slot = gs.slot;
        const unsigned batch = slot / NB;
        const int buf = (int)(batch & 1u), pos = (int)(slot % NB);
        float rb = gs.red_rmax[0];
#pragma unroll
        for (int w = 1; w < GW; ++w) rb += gs.red_rmax[w];
        float inv;
        const float scale = track_scale(rb, &inv);
        ptx::mbar_wait(&meta->buf_free[buf], ((batch >> 1) & 1u) ^ 1u, 107);
        uint8_t* rt = fz + OFF_RT + buf * RT_BYTES;
        constexpr int CW = D / GW;
#pragma unroll
        for (int c0 = 0; c0 < CW; c0 += 64) {
          const int c = CW * wg + c0 + 2 * lane;
          float2 po = make_float2(0.f, 0.f), rr = po;
#pragma unroll
          for (int w = 0; w < GW; ++w) {
            const float2 a = *reinterpret_cast<const float2*>(&gs.part[w][c]);
            const float2 b = *reinterpret_cast<const float2*>(&gs.part[w][D + c]);
            po.x += a.x;
            po.y += a.y;
            rr.x += b.x;
            rr.y += b.y;
          }
          if (len > 1) {
            float qsum = gs.red_q[0];
#pragma unroll
            for (int w = 1; w < GW; ++w) qsum += gs.red_q[w];
            const float2 wbg = *reinterpret_cast<const float2*>(fold + Fold::WBG + c);
            const float2 bw = *reinterpret_cast<const float2*>(fold + Fold::BW + c);
            po.x += fmaf(qsum, wbg.x, bw.x);
            po.y += fmaf(qsum, wbg.y, bw.y);
          }
          *reinterpret_cast<float2*>(out_local + (size_t)track * D + c) = po;
          store_r2(rt, pos, c, rr.x, rr.y, scale);
        }
        if (wg == 0 && lane == 0) {
          meta->slot_track[buf][pos] = (int)track;
          meta->fscale[buf][pos] = inv;
        }
        ptx::fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&meta->tile_full[buf]);
      }
      len = len_next;
    }
  }
  fused_teardown(fz, warp, GWARPS);
  if (p.x_on && p.x_last) xchg::signal_all(p.x, xchg::KIND_Q, xstep);
}


}  // namespace aggf
}  // namespace seam
