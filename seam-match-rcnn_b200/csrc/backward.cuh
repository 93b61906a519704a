// f4: backward of the hot path for training (SURVEY.md section 8 f4).
//
// The reference trains through the aggregator with autograd (models/match_head.py:339, 429: the losses consume
// x5 = last((x3_1b - x3_2)^2) of TemporalAggregationNLB.forward's x-branch; stuffs/engine.py:158-185).  The block
// differentiated is models/nlb.py:66-101 followed by the attention pooling of match_head.py:144-151:
//
//   theta_t = Wt x_t + bt   phi_j = Wp x_j + bp   g_j = Wg x_j + bg                        nlb.py:72-79
//   pre_tj = wt.theta_t + wp.phi_j ;  f_tj = relu(pre_tj) / T                               nlb.py:84-93
//   z_t = WW (sum_j f_tj g_j) + bW + x_t ;  s_t = wa.z_t + ba ;  p = softmax_t(s) ;  out = sum_t p_t z_t
//   (T == 1: the block is skipped, out = x_0: match_head.py:145-147)
//
// Its backward collapses the way the forward does (DESIGN.md "K1 algebra", fold.cuh): with the folded vectors
//   u_theta = Wt^T wt, u_phi = Wp^T wp, nu = WW^T wa, u_g = Wg^T nu (and their constants)
// and per track, from the upstream gradient o = d loss / d out,
//   mu = WW^T o, m = Wg^T mu, c_mu = bg.mu, e0 = bW.o,
// every frame needs six dots (a_t, b_t, c_t, d_t with the folded vectors, gamma_t = m.x_t + c_mu, e_t = o.x_t) and
// O(T^2) scalar work; every per-frame gradient is a combination of six fixed 256-vectors
//   dx_t = p_t o + ds_t wa + alpha_t u_theta + beta_t u_phi + q_t m + q'_t u_g
// and every parameter gradient an outer product of fixed vectors and per-track weighted sums of the frames (DESIGN.md
// section 4 f4 lists them).  The work per track is O(T*256 + T^2) and three 128x256 matrix-vector products.
//
// agg_backward_folded_kernel: persistent CTAs of 256 threads (thread = channel), each folding the weights it was
// given once and then taking tracks blockIdx.x, blockIdx.x + gridDim.x, ...  A track is handled by one CTA in a
// fixed order, so dseq (written once per frame, no atomics) does not depend on the grid.  The parameter gradients
// are accumulated with atomicAdd: the two outer products whose left vector changes with the track (g.weight:
// mu (x) r, W.weight: o (x) hr) per track, everything with a fixed left vector summed over the CTA's tracks in
// registers and added once at the end.
// scorer_backward_{q,g}_kernel: gradients of x5 = last((q - g)^2) (match_head.py:160-162) for the dense (Q,G,2)
// logits training uses.
#pragma once
#include <cstdint>
#include "../../include/seam_b200.h"
#include "sm100_ptx.cuh"

namespace seam {
namespace bwd {

constexpr int D = 256, DI = 128, MAXT = SEAM_MAX_T;

struct AggWeights {     // the reference's parameters, fp32, device pointers
  const float *theta_w, *theta_b, *phi_w, *phi_b, *g_w, *g_b, *W_w, *W_b, *concat_w, *att_w, *att_b;
};
struct AggGrads {       // same shapes, accumulated into (caller zero-fills)
  float *theta_w, *theta_b, *phi_w, *phi_b, *g_w, *g_b, *W_w, *W_b, *concat_w, *att_w, *att_b;
};
struct AggBwdParams {
  const float* seq;
  const uint8_t* mask;
  const int32_t* lens;
  int Tmax, Q;
  long long frame_stride, track_stride;
  const float* dout;      // (Q,256)
  float* dseq;            // (1+Tmax, Q, 256) contiguous; row 0 and padded frames are zero-filled by the caller
  AggWeights w;
  AggGrads g;
};

// dynamic shared memory: the track's frames, fp32
constexpr size_t agg_bwd_smem_bytes(int Tmax) { return (size_t)Tmax * D * sizeof(float); }

// out[i] = sum_k A[i*lda + k] * v[k] + s * bias[i], i < n; one warp per row (v in shared memory)
__device__ __forceinline__ void rows_dot(float* out, const float* __restrict__ A, int lda, const float* v, int n,
                                         int K, float s, const float* __restrict__ bias) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = warp; i < n; i += 8) {
    float acc = 0.f;
    for (int k = lane; k < K; k += 32) acc = fmaf(A[(size_t)i * lda + k], v[k], acc);
    acc = ptx::warp_sum(acc);
    if (lane == 0) out[i] = fmaf(s, bias[i], acc);
  }
}

// out[c] = sum_o WW[o][c] v[o] (WW: 256 x 128, v in shared memory), both thread halves sum half of o; two barriers
__device__ __forceinline__ void ww_t_mv(float* out, float* part, const float* __restrict__ WW, const float* v) {
  const int c = threadIdx.x & 127, o0 = threadIdx.x & 128;
  float a = 0.f;
#pragma unroll 4
  for (int o = o0; o < o0 + 128; ++o) a = fmaf(WW[(size_t)o * DI + c], v[o], a);
  part[threadIdx.x] = a;
  __syncthreads();
  if (threadIdx.x < DI) out[c] = part[c] + part[DI + c];
  __syncthreads();
}

// out[k] = sum_c M[c][k] v[c] (M: 128 x 256, v in shared memory); thread = k
__device__ __forceinline__ float mt_mv(const float* __restrict__ M, const float* v) {
  float a = 0.f;
#pragma unroll 4
  for (int c = 0; c < DI; ++c) a = fmaf(M[(size_t)c * D + threadIdx.x], v[c], a);
  return a;
}

// sum of v over a warp's lanes 0..31 and 32..63 (T <= 64 values, zero past T)
__device__ __forceinline__ float sum64(const float* v, int T) {
  const int lane = threadIdx.x & 31;
  float a = lane < T ? v[lane] : 0.f;
  if (lane + 32 < T) a += v[lane + 32];
  return ptx::warp_sum(a);
}

__global__ void __launch_bounds__(256, 3) agg_backward_folded_kernel(const AggBwdParams p) {
  extern __shared__ __align__(16) float xs[];               // [T][256] the track's frames
  __shared__ float s_uth[D], s_uph[D], s_ug[D], s_wa[D];    // folded vectors
  __shared__ float s_o[D], s_m[D], s_r[D], s_part[D];
  __shared__ float s_wt[DI], s_wp[DI], s_nu[DI], s_mu[DI], s_hr[DI];
  __shared__ float fa[MAXT], fb[MAXT], fc[MAXT], fd[MAXT], fgam[MAXT], fe[MAXT];
  __shared__ float fp[MAXT], fds[MAXT], fq[MAXT], fqp[MAXT], fal[MAXT], fbe[MAXT];
  __shared__ float sc[8];   // c_theta, c_phi, c_g, c_s, c_mu, e0, S
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const AggWeights& W = p.w;

  // ---- fold the weights of this call (fold_vectors_kernel's vectors, fp32 accumulation)
  s_wa[tid] = W.att_w[tid];
  if (tid < DI) {
    s_wt[tid] = W.concat_w[tid];
    s_wp[tid] = W.concat_w[DI + tid];
  }
  __syncthreads();
  ww_t_mv(s_nu, s_part, W.W_w, s_wa);                       // nu = WW^T wa
  s_uth[tid] = mt_mv(W.theta_w, s_wt);
  s_uph[tid] = mt_mv(W.phi_w, s_wp);
  s_ug[tid] = mt_mv(W.g_w, s_nu);
  if (warp < 4) {
    const float* bias = warp == 0 ? W.theta_b : warp == 1 ? W.phi_b : warp == 2 ? W.g_b : W.W_b;
    const float* v = warp == 0 ? s_wt : warp == 1 ? s_wp : warp == 2 ? s_nu : s_wa;
    const int n = warp == 3 ? D : DI;
    float a = 0.f;
    for (int k = lane; k < n; k += 32) a = fmaf(bias[k], v[k], a);
    a = ptx::warp_sum(a);
    if (lane == 0) sc[warp] = warp == 3 ? a + W.att_b[0] : a;
  }
  // (the first barrier of the track loop publishes the folded vectors)

  // sums over this CTA's tracks of the terms with a fixed left vector
  float accA = 0.f, accB = 0.f, accE = 0.f, accRp = 0.f, accWb = 0.f, accGb = 0.f;
  float sumAl = 0.f, sumBe = 0.f, sumS = 0.f, sumQp = 0.f;
  bool any = false;

  for (int track = blockIdx.x; track < p.Q; track += gridDim.x) {
    // ---- track length (models/match_head.py:136-139)
    int len;
    if (p.lens) {
      len = p.lens[track];
    } else if (p.mask) {
      len = p.Tmax;
      for (int t = 0; t <= p.Tmax; ++t)
        if (p.mask[(size_t)track * (1 + p.Tmax) + t]) {
          len = t - 1;
          break;
        }
    } else {
      len = p.Tmax;
    }
    len = max(0, min(len, p.Tmax));
    if (len == 0) continue;
    const float o_k = p.dout[(size_t)track * D + tid];
    if (len == 1) {                                         // block skipped, softmax of one logit: out = x_0
      p.dseq[((size_t)1 * p.Q + track) * D + tid] = o_k;
      continue;
    }
    const int T = len;
    const float invT = 1.f / (float)T;
    any = true;
    __syncthreads();                                        // the previous track is done with the shared buffers
    s_o[tid] = o_k;
    for (int t = 0; t < T; ++t)
      xs[t * D + tid] = p.seq[(long long)(t + 1) * p.frame_stride + (long long)track * p.track_stride + tid];
    __syncthreads();
    ww_t_mv(s_mu, s_part, W.W_w, s_o);                      // mu = WW^T o
    s_m[tid] = mt_mv(W.g_w, s_mu);                          // m = Wg^T mu
    if (warp == 0) {
      float a = 0.f;
      for (int c = lane; c < DI; c += 32) a = fmaf(W.g_b[c], s_mu[c], a);
      a = ptx::warp_sum(a);
      if (lane == 0) sc[4] = a;                             // c_mu
    } else if (warp == 1) {
      float a = 0.f;
      for (int k = lane; k < D; k += 32) a = fmaf(W.W_b[k], s_o[k], a);
      a = ptx::warp_sum(a);
      if (lane == 0) sc[5] = a;                             // e0
    }
    __syncthreads();
    // ---- six dots per frame: one warp per frame, lanes over channels
    for (int t = warp; t < T; t += 8) {
      float a = 0.f, b = 0.f, c = 0.f, d = 0.f, g = 0.f, e = 0.f;
#pragma unroll 2
      for (int i = 0; i < 8; ++i) {
        const int k = lane + 32 * i;
        const float xv = xs[t * D + k];
        a = fmaf(xv, s_uth[k], a);
        b = fmaf(xv, s_uph[k], b);
        c = fmaf(xv, s_ug[k], c);
        d = fmaf(xv, s_wa[k], d);
        g = fmaf(xv, s_m[k], g);
        e = fmaf(xv, s_o[k], e);
      }
      a = ptx::warp_sum(a);
      b = ptx::warp_sum(b);
      c = ptx::warp_sum(c);
      d = ptx::warp_sum(d);
      g = ptx::warp_sum(g);
      e = ptx::warp_sum(e);
      if (lane == 0) {
        fa[t] = a + sc[0];
        fb[t] = b + sc[1];
        fc[t] = c + sc[2];
        fd[t] = d;
        fgam[t] = g + sc[4];
        fe[t] = e;
      }
    }
    __syncthreads();
    // ---- forward logits s_t and h_t = o.z_t (thread t)
    if (tid < T) {
      const float at = fa[tid];
      float s = 0.f, h = 0.f;
      for (int j = 0; j < T; ++j) {
        const float f = fmaxf(at + fb[j], 0.f) * invT;
        s = fmaf(f, fc[j], s);
        h = fmaf(f, fgam[j], h);
      }
      fp[tid] = fd[tid] + s + sc[3];
      fds[tid] = fe[tid] + h + sc[5];
    }
    __syncthreads();
    // ---- softmax and its backward (one warp: T <= 64 = two values per lane)
    if (warp == 0) {
      const bool v0 = lane < T, v1 = lane + 32 < T;
      const float s0 = v0 ? fp[lane] : -INFINITY, s1 = v1 ? fp[lane + 32] : -INFINITY;
      float mx = fmaxf(s0, s1);
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
      const float e0 = v0 ? expf(s0 - mx) : 0.f, e1 = v1 ? expf(s1 - mx) : 0.f;
      const float inv = 1.f / ptx::warp_sum(e0 + e1);
      const float p0 = e0 * inv, p1 = e1 * inv;
      const float h0 = v0 ? fds[lane] : 0.f, h1 = v1 ? fds[lane + 32] : 0.f;
      const float H = ptx::warp_sum(fmaf(p0, h0, p1 * h1));
      const float d0 = p0 * (h0 - H), d1 = p1 * (h1 - H);
      __syncwarp();
      if (v0) { fp[lane] = p0; fds[lane] = d0; }
      if (v1) { fp[lane + 32] = p1; fds[lane + 32] = d1; }
      const float S = ptx::warp_sum(d0 + d1);
      if (lane == 0) sc[6] = S;
    }
    __syncthreads();
    // ---- q_j, q'_j, beta_j (thread j) and alpha_t (thread 64 + t):  g_tj = [pre_tj > 0] (p_t gamma_j + ds_t c_j) / T
    if (tid < T) {
      const int j = tid;
      const float bj = fb[j], cj = fc[j], gj = fgam[j];
      float q = 0.f, qp = 0.f, be = 0.f;
      for (int t = 0; t < T; ++t) {
        const float pre = fa[t] + bj;
        const float f = fmaxf(pre, 0.f) * invT;
        q = fmaf(fp[t], f, q);
        qp = fmaf(fds[t], f, qp);
        if (pre > 0.f) be += fmaf(fp[t], gj, fds[t] * cj) * invT;
      }
      fq[j] = q;
      fqp[j] = qp;
      fbe[j] = be;
    } else if (tid >= MAXT && tid < MAXT + T) {
      const int t = tid - MAXT;
      const float at = fa[t], pt = fp[t], dst = fds[t];
      float al = 0.f;
      for (int j = 0; j < T; ++j)
        if (at + fb[j] > 0.f) al += fmaf(pt, fgam[j], dst * fc[j]) * invT;
      fal[t] = al;
    }
    __syncthreads();
    // ---- dx_t (thread = channel), weighted sums of the frames
    const float uth = s_uth[tid], uph = s_uph[tid], ug = s_ug[tid], wa = s_wa[tid], m = s_m[tid];
    float r = 0.f, rp = 0.f, A = 0.f, B = 0.f, E = 0.f;
    float Qs = 0.f, Qps = 0.f, Als = 0.f, Bes = 0.f;
    for (int t = 0; t < T; ++t) {
      const float pt = fp[t], dst = fds[t], al = fal[t], be = fbe[t], q = fq[t], qp = fqp[t];
      const float dx = fmaf(pt, o_k, fmaf(dst, wa, fmaf(al, uth, fmaf(be, uph, fmaf(q, m, qp * ug)))));
      p.dseq[((size_t)(t + 1) * p.Q + track) * D + tid] = dx;
      const float xv = xs[t * D + tid];
      r = fmaf(q, xv, r);
      rp = fmaf(qp, xv, rp);
      A = fmaf(al, xv, A);
      B = fmaf(be, xv, B);
      E = fmaf(dst, xv, E);
      Qs += q;
      Qps += qp;
      Als += al;
      Bes += be;
    }
    const float S = sc[6];
    s_r[tid] = r;
    accA += A;
    accB += B;
    accE += E;
    accRp += rp;
    accWb += fmaf(S, wa, o_k);
    if (tid < DI) accGb += fmaf(Qs, s_mu[tid], Qps * s_nu[tid]);
    sumAl += Als;
    sumBe += Bes;
    sumS += S;
    sumQp += Qps;
    // g.weight[c][k] += mu[c] r[k] + nu[c] r'[k]
#pragma unroll 4
    for (int c = 0; c < DI; ++c) atomicAdd(p.g.g_w + (size_t)c * D + tid, fmaf(s_mu[c], r, s_nu[c] * rp));
    __syncthreads();
    rows_dot(s_hr, W.g_w, D, s_r, DI, D, Qs, W.g_b);      // hr = Wg r + Q bg
    __syncthreads();
    // W.weight[o][c] += o[o] hr[c]   (warp = rows, lanes = columns: coalesced)
    for (int o = warp; o < D; o += 8) {
      const float ov = s_o[o];
#pragma unroll
      for (int i = 0; i < DI / 32; ++i) atomicAdd(p.g.W_w + (size_t)o * DI + lane + 32 * i, ov * s_hr[lane + 32 * i]);
    }
  }
  if (!any) return;                                         // uniform: every thread saw the same tracks

  // ---- once per CTA: the terms with a fixed left vector, summed over its tracks
  __syncthreads();
  s_o[tid] = accA;                                          // reuse: A, B, r' sums
  s_m[tid] = accB;
  s_r[tid] = accRp;
  __syncthreads();
#pragma unroll 4
  for (int c = 0; c < DI; ++c) {
    atomicAdd(p.g.theta_w + (size_t)c * D + tid, s_wt[c] * accA);
    atomicAdd(p.g.phi_w + (size_t)c * D + tid, s_wp[c] * accB);
  }
  rows_dot(s_hr, W.g_w, D, s_r, DI, D, sumQp, W.g_b);       // sum of hr' = Wg r' + Q' bg
  rows_dot(s_part, W.theta_w, D, s_o, DI, D, sumAl, W.theta_b);        // concat[:128]  = Wt A + alpha bt
  rows_dot(s_part + DI, W.phi_w, D, s_m, DI, D, sumBe, W.phi_b);       // concat[128:]  = Wp B + beta bp
  __syncthreads();
  if (tid < DI) {
    atomicAdd(p.g.theta_b + tid, sumAl * s_wt[tid]);
    atomicAdd(p.g.phi_b + tid, sumBe * s_wp[tid]);
    atomicAdd(p.g.g_b + tid, accGb);
  }
  atomicAdd(p.g.concat_w + tid, s_part[tid]);
  atomicAdd(p.g.W_b + tid, accWb);
  if (tid == 0) atomicAdd(p.g.att_b, sumS);
  for (int o = warp; o < D; o += 8) {                       // W.weight[o][c] += wa[o] hr'[c]
    const float wv = s_wa[o];
#pragma unroll
    for (int i = 0; i < DI / 32; ++i) atomicAdd(p.g.W_w + (size_t)o * DI + lane + 32 * i, wv * s_hr[lane + 32 * i]);
  }
  __syncthreads();                                          // s_part is reused below
  rows_dot(s_part, W.W_w, DI, s_hr, D, DI, sumS, W.W_b);    // att_w += E + WW hr' + S bW
  __syncthreads();
  atomicAdd(p.g.att_w + tid, accE + s_part[tid]);
}

// ---------------------------------------------------------------------------------------- pair scorer backward
// x5[i,j,c] = sum_k W[c,k] (q_ik - g_jk)^2 + b_c.  One CTA per query (thread = channel k): dq, and this query's
// contribution to dW / db.
__global__ void __launch_bounds__(256) scorer_backward_q_kernel(const float* __restrict__ q, int Q,
                                                                const float* __restrict__ g, int G,
                                                                const float* __restrict__ last_w,
                                                                const float* __restrict__ dx5, float* __restrict__ dq,
                                                                float* __restrict__ dlast_w, float* __restrict__ dlast_b) {
  const int i = blockIdx.x, k = threadIdx.x;
  const float qv = q[(size_t)i * 256 + k], w0 = last_w[k], w1 = last_w[256 + k];
  float dqv = 0.f, dw0 = 0.f, dw1 = 0.f, db0 = 0.f, db1 = 0.f;
  for (int j = 0; j < G; ++j) {
    const float2 e = *reinterpret_cast<const float2*>(dx5 + ((size_t)i * G + j) * 2);
    const float diff = qv - g[(size_t)j * 256 + k];
    dqv = fmaf(2.f * fmaf(e.x, w0, e.y * w1), diff, dqv);
    const float d2 = diff * diff;
    dw0 = fmaf(e.x, d2, dw0);
    dw1 = fmaf(e.y, d2, dw1);
    db0 += e.x;
    db1 += e.y;
  }
  dq[(size_t)i * 256 + k] = dqv;
  atomicAdd(dlast_w + k, dw0);
  atomicAdd(dlast_w + 256 + k, dw1);
  if (k == 0) {
    atomicAdd(dlast_b, db0);
    atomicAdd(dlast_b + 1, db1);
  }
}
// one CTA per gallery row: dg (no atomics)
__global__ void __launch_bounds__(256) scorer_backward_g_kernel(const float* __restrict__ q, int Q,
                                                                const float* __restrict__ g, int G,
                                                                const float* __restrict__ last_w,
                                                                const float* __restrict__ dx5, float* __restrict__ dg) {
  const int j = blockIdx.x, k = threadIdx.x;
  const float gv = g[(size_t)j * 256 + k], w0 = last_w[k], w1 = last_w[256 + k];
  float d = 0.f;
  for (int i = 0; i < Q; ++i) {
    const float2 e = *reinterpret_cast<const float2*>(dx5 + ((size_t)i * G + j) * 2);
    d = fmaf(-2.f * fmaf(e.x, w0, e.y * w1), q[(size_t)i * 256 + k] - gv, d);
  }
  dg[(size_t)j * 256 + k] = d;
}

}  // namespace bwd
}  // namespace seam
