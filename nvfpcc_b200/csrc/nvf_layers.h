// Layer-at-a-time kernels: every layer of the NVF decoder (forward), its data
// gradient and its weight gradient as grid-wide kernels over (block, tile).
// Used for the training path (activations are stashed for the backward pass
// anyway, and at --batchsize 16 they are L2-resident) and for decoding channel
// configurations that have no fused kernel.  Reference maths: SURVEY.md 3.4/3.5
// (utils/network.py:4758-4768 forward; autograd of the same ops backward).
#pragma once
#include <stddef.h>
#include <type_traits>
#include "nvf_common.h"
#include "nvf_tiles.h"
#include "../../include/nvf_b200.h"

namespace nvf {

enum LayerOp { OP_CORR3 = 0, OP_CORR4 = 1, OP_CONVT = 2, OP_CORR_S2 = 3 };
enum Act { ACT_NONE = 0, ACT_RELU = 1, ACT_SIGMOID = 2 };

struct LayerParams {
  const float* in;    // [n][CI][Din][Din][inPitch]
  float* out;         // [n][CO][Dout][Dout][outPitch]
  const float* Wp;    // packed [CI][K^3][CO]
  const float* bias;  // [CO] or null
  const float* add;   // same layout as out, added before act/mask, or null
  const float* mask;  // same layout as out: out = mask > 0 ? out : 0, or null
  int32_t n, CI, CO, Din, inPitch, Dout, outPitch, P, act, op;
  float* out2;        // optional second copy of the output (same layout) or null
};

template <int COT>
struct LayerKernel {
  typedef LayerParams Params;
  static NVF_HD void thread(const LayerParams& p, int bid, int tid, int nbid) {
    const int XT = (p.Dout + 3) >> 2;
    const int groups = p.CO / COT;
    const int64_t per_block = (int64_t)groups * p.Dout * p.Dout * XT;
    const int64_t total = per_block * p.n;
    const int64_t in_bs = (int64_t)p.CI * p.Din * p.Din * p.inPitch;
    const int64_t out_cs = (int64_t)p.Dout * p.Dout * p.outPitch;
    for (int64_t t = (int64_t)bid * kThreads + tid; t < total; t += (int64_t)nbid * kThreads) {
      const int b = (int)(t / per_block);
      int r = (int)(t - (int64_t)b * per_block);
      const int xt = r % XT; r /= XT;
      const int oy = r % p.Dout; r /= p.Dout;
      const int oz = r % p.Dout; r /= p.Dout;
      const int co0 = r * COT;
      const int ox0 = xt * 4;
      View in{p.in + b * in_bs, p.Din * p.Din * p.inPitch, p.Din * p.inPitch, p.inPitch, p.Din};
      float acc[COT][4];
      zero_acc<COT>(acc);
      if (p.op == OP_CORR3) corr_s1_tile<3, COT>(in, p.CI, p.P, p.Wp, p.CO, co0, oz, oy, ox0, acc);
      else if (p.op == OP_CORR4) corr_s1_tile<4, COT>(in, p.CI, p.P, p.Wp, p.CO, co0, oz, oy, ox0, acc);
      else if (p.op == OP_CONVT) convT5_tile<COT>(in, p.CI, p.P, p.Wp, p.CO, co0, oz, oy, ox0, acc);
      else corr_s2_tile<COT>(in, p.CI, p.P, p.Wp, p.CO, co0, oz, oy, ox0, acc);
      NVF_UNROLL
      for (int c = 0; c < COT; ++c) {
        const int64_t o = ((int64_t)b * p.CO + co0 + c) * out_cs + ((int64_t)oz * p.Dout + oy) * p.outPitch + ox0;
        const float bb = p.bias ? p.bias[co0 + c] : 0.f;
        NVF_UNROLL
        for (int j = 0; j < 4; ++j) {
          if (ox0 + j >= p.Dout) continue;
          float v = acc[c][j] + bb;
          if (p.add) v += p.add[o + j];
          if (p.act == ACT_RELU) v = relu(v);
          else if (p.act == ACT_SIGMOID) v = sigmoidf(v);
          if (p.mask) v = p.mask[o + j] > 0.f ? v : 0.f;
          p.out[o + j] = v;
          if (p.out2) p.out2[o + j] = v;
        }
      }
    }
  }
};

// ---------------------------------------------------------------------------
// Weight gradients.  Both families share one formulation:
//   dW[a][s][kz][ky][kx] = sum_{b,pos} A[b][a][pos] * Sft[b][s][S*pos + k - P]
//   conv  : A = g (Cout), Sft = x (Cin), S = 1  -> dW (Cout,Cin,K,K,K)
//   convT : A = x (Cin),  Sft = g (Cout), S = 2 -> dW (Cin,Cout,K,K,K)
// One CTA per (a-group, s, kz, ky): every thread accumulates COT x K partial
// sums over its share of positions, then a fixed-order tree reduction in
// shared memory makes the result deterministic (no atomics).
// ---------------------------------------------------------------------------
struct WgradParams {
  const float* A;    // [n][CA][Da][Da][aPitch]
  const float* Sft;  // [n][CS][Ds][Ds][sPitch]
  float* dW;         // [CA][CS][K][K][K]
  int32_t n, CA, CS, Da, aPitch, Ds, sPitch, K, S, P;
};

template <int COT, int K>
struct WgradBlock {
  static constexpr int NACC = COT * K;
  // smem: kThreads * NACC floats
  template <class Env>
  static NVF_HD void run(Env& env, const WgradParams& p, float* sm, int bid) {
    int r = bid;
    const int ky = r % K; r /= K;
    const int kz = r % K; r /= K;
    const int s = r % p.CS; r /= p.CS;
    const int a0 = r * COT;
    const int XT = (p.Da + 3) >> 2;
    const int64_t a_cs = (int64_t)p.Da * p.Da * p.aPitch, s_cs = (int64_t)p.Ds * p.Ds * p.sPitch;
    env.phase([&](int tid, int&) {
      float acc[COT][K];
      NVF_UNROLL
      for (int c = 0; c < COT; ++c) {
        NVF_UNROLL
        for (int k = 0; k < K; ++k) acc[c][k] = 0.f;
      }
      const int64_t per_block = (int64_t)p.Da * p.Da * XT;
      const int64_t total = per_block * p.n;
      for (int64_t t = tid; t < total; t += kThreads) {
        const int b = (int)(t / per_block);
        int q = (int)(t - (int64_t)b * per_block);
        const int xt = q % XT; q /= XT;
        const int y = q % p.Da; q /= p.Da;
        const int z = q;
        const int sz = p.S * z + kz - p.P, sy = p.S * y + ky - p.P;
        if (sz < 0 || sz >= p.Ds || sy < 0 || sy >= p.Ds) continue;
        const int x0 = xt * 4;
        const float* srow = p.Sft + ((int64_t)b * p.CS + s) * s_cs + ((int64_t)sz * p.Ds + sy) * p.sPitch;
        float sv[2 * 3 + K + 1];
        const int nsv = p.S * 3 + K;
        NVF_UNROLL
        for (int i = 0; i < 2 * 3 + K; ++i) {
          const int sx = p.S * x0 + i - p.P;
          sv[i] = (i < nsv && sx >= 0 && sx < p.Ds) ? srow[sx] : 0.f;
        }
        NVF_UNROLL
        for (int c = 0; c < COT; ++c) {
          const float* arow = p.A + ((int64_t)b * p.CA + a0 + c) * a_cs + ((int64_t)z * p.Da + y) * p.aPitch + x0;
          NVF_UNROLL
          for (int j = 0; j < 4; ++j) {
            const float av = (x0 + j < p.Da) ? arow[j] : 0.f;
            NVF_UNROLL
            for (int k = 0; k < K; ++k) {
              const float v = p.S == 1 ? sv[j + k] : sv[2 * j + k];
              acc[c][k] = fmaf(av, v, acc[c][k]);
            }
          }
        }
      }
      NVF_UNROLL
      for (int c = 0; c < COT; ++c) {
        NVF_UNROLL
        for (int k = 0; k < K; ++k) sm[(c * K + k) * kThreads + tid] = acc[c][k];
      }
    });
    for (int stride = kThreads / 2; stride >= 1; stride >>= 1) {
      env.phase([&](int tid, int&) {
        if (tid < stride) {
          for (int e = 0; e < NACC; ++e) sm[e * kThreads + tid] += sm[e * kThreads + tid + stride];
        }
      });
    }
    env.phase([&](int tid, int&) {
      if (tid < NACC) {
        const int c = tid / K, k = tid % K;
        p.dW[((((int64_t)(a0 + c) * p.CS + s) * K + kz) * K + ky) * K + k] = sm[tid * kThreads];
      }
    });
  }
};

// Per-channel sum (bias gradients): out[c] = sum_{b,pos} g[b][c][pos] over the valid cube.
struct ChanSumParams {
  const float* g;
  float* out;
  int32_t n, C, D, pitch;
};
struct ChanSumBlock {
  template <class Env>
  static NVF_HD void run(Env& env, const ChanSumParams& p, float* sm, int c) {
    env.phase([&](int tid, int&) {
      float s = 0.f;
      const int64_t cs = (int64_t)p.D * p.D * p.pitch;
      const int64_t rows = (int64_t)p.n * p.D * p.D;
      for (int64_t r = tid; r < rows; r += kThreads) {
        const int b = (int)(r / (p.D * p.D));
        const int zy = (int)(r - (int64_t)b * p.D * p.D);
        const float* row = p.g + ((int64_t)b * p.C + c) * cs + (int64_t)zy * p.pitch;
        for (int x = 0; x < p.D; ++x) s += row[x];
      }
      sm[tid] = s;
    });
    for (int stride = kThreads / 2; stride >= 1; stride >>= 1) {
      env.phase([&](int tid, int&) {
        if (tid < stride) sm[tid] += sm[tid + stride];
      });
    }
    env.phase([&](int tid, int&) {
      if (tid == 0) p.out[c] = sm[0];
    });
  }
};

// ---------------------------------------------------------------------------
// IGDN (gdn_3d.py:137-159): y_i = x_i * sqrt(beta_i + sum_j gamma_ij x_j^2)
// ---------------------------------------------------------------------------
struct IgdnParams {
  const float* x;      // [n][C][64]
  float* y;            // forward out / backward dx
  const float* g;      // backward: dL/dy
  const float* beta;   // [C]
  const float* gamma;  // [C][C]
  float* dbeta;        // [C]      (backward, may be null)
  float* dgamma;       // [C][C]   (backward, may be null)
  int32_t n, C;
};
struct IgdnFwdKernel {
  typedef IgdnParams Params;
  static NVF_HD void thread(const IgdnParams& p, int bid, int tid, int nbid) {
    const int64_t total = (int64_t)p.n * p.C * 64;
    for (int64_t t = (int64_t)bid * kThreads + tid; t < total; t += (int64_t)nbid * kThreads) {
      const int pos = (int)(t & 63), c = (int)((t >> 6) % p.C), b = (int)(t / (64 * p.C));
      const float* xb = p.x + (int64_t)b * p.C * 64 + pos;
      float n = p.beta[c];
      for (int j = 0; j < p.C; ++j) n = fmaf(p.gamma[c * p.C + j], xb[j * 64] * xb[j * 64], n);
      p.y[t] = xb[c * 64] * sqrtf(n);
    }
  }
};
// dx_k = g_k n_k + x_k sum_i g_i x_i gamma_ik / n_i      (SURVEY.md 3.5)
struct IgdnBwdDxKernel {
  typedef IgdnParams Params;
  static NVF_HD void thread(const IgdnParams& p, int bid, int tid, int nbid) {
    const int64_t total = (int64_t)p.n * p.C * 64;
    for (int64_t t = (int64_t)bid * kThreads + tid; t < total; t += (int64_t)nbid * kThreads) {
      const int pos = (int)(t & 63), k = (int)((t >> 6) % p.C), b = (int)(t / (64 * p.C));
      const float* xb = p.x + (int64_t)b * p.C * 64 + pos;
      const float* gb = p.g + (int64_t)b * p.C * 64 + pos;
      float acc = 0.f, nk = 0.f;
      for (int i = 0; i < p.C; ++i) {
        float n = p.beta[i];
        for (int j = 0; j < p.C; ++j) n = fmaf(p.gamma[i * p.C + j], xb[j * 64] * xb[j * 64], n);
        n = sqrtf(n);
        if (i == k) nk = n;
        acc += gb[i * 64] * xb[i * 64] * p.gamma[i * p.C + k] / n;
      }
      p.y[t] = gb[k * 64] * nk + xb[k * 64] * acc;
    }
  }
};
// dbeta_i = sum g_i x_i/(2 n_i);  dgamma_ij = sum g_i x_i x_j^2/(2 n_i).  One CTA, thread = (i,j).
struct IgdnBwdParamKernel {
  typedef IgdnParams Params;
  static NVF_HD void thread(const IgdnParams& p, int bid, int tid, int nbid) {
    if (bid != 0 || tid >= p.C * p.C) return;
    const int i = tid / p.C, j = tid % p.C;
    float dg = 0.f, db = 0.f;
    for (int64_t q = 0; q < (int64_t)p.n * 64; ++q) {
      const int b = (int)(q >> 6), pos = (int)(q & 63);
      const float* xb = p.x + (int64_t)b * p.C * 64 + pos;
      float n = p.beta[i];
      for (int l = 0; l < p.C; ++l) n = fmaf(p.gamma[i * p.C + l], xb[l * 64] * xb[l * 64], n);
      const float t = p.g[(int64_t)b * p.C * 64 + i * 64 + pos] * xb[i * 64] / (2.f * sqrtf(n));
      dg = fmaf(t, xb[j * 64] * xb[j * 64], dg);
      db += t;
    }
    if (p.dgamma) p.dgamma[i * p.C + j] = dg;
    if (p.dbeta && j == 0) p.dbeta[i] = db;
  }
};

// ---------------------------------------------------------------------------
// element-wise helpers
// ---------------------------------------------------------------------------
// g_logit = g_p * p * (1 - p)   (d sigmoid)
struct SigBwdParams {
  const float* gp;
  const float* p;
  float* out;
  int64_t n;
};
struct SigBwdKernel {
  typedef SigBwdParams Params;
  static NVF_HD void thread(const SigBwdParams& p, int bid, int tid, int nbid) {
    for (int64_t t = (int64_t)bid * kThreads + tid; t < p.n; t += (int64_t)nbid * kThreads) {
      const float pr = p.p[t];
      p.out[t] = p.gp ? p.gp[t] * pr * (1.f - pr) : 0.f;
    }
  }
};

// the three heads in one launch: segment h covers n[h] elements
struct SigBwd3Params {
  const float* gp[3];
  const float* p[3];
  float* out[3];
  int64_t n[3];
};
struct SigBwd3Kernel {
  typedef SigBwd3Params Params;
  static NVF_HD void thread(const SigBwd3Params& q, int bid, int tid, int nbid) {
    const int64_t total = q.n[0] + q.n[1] + q.n[2];
    for (int64_t t = (int64_t)bid * kThreads + tid; t < total; t += (int64_t)nbid * kThreads) {
      const int h = t < q.n[0] ? 0 : (t < q.n[0] + q.n[1] ? 1 : 2);
      const int64_t i = t - (h == 0 ? 0 : (h == 1 ? q.n[0] : q.n[0] + q.n[1]));
      const float pr = q.p[h][i];
      q.out[h][i] = q.gp[h] ? q.gp[h][i] * pr * (1.f - pr) : 0.f;
    }
  }
};

// probability grid -> occupancy mask words + per-block counts (generic decode path)
struct MaskParams {
  const float* prob;  // [n][32768]
  uint32_t* mask;     // [n][1024]
  int32_t* counts;    // [n]
  float thh;
  int32_t n;
};
struct MaskBlock {
  // one CTA per block
  template <class Env>
  static NVF_HD void run(Env& env, const MaskParams& p, int* sm, int b) {
    env.phase([&](int tid, int&) {
      int c = 0;
      for (int w = tid; w < 1024; w += kThreads) {
        const float* row = p.prob + (int64_t)b * kVox + w * 32;
        uint32_t bits = 0;
        for (int k = 0; k < 32; ++k)
          if (row[k] > p.thh) bits |= 1u << k;
        p.mask[(int64_t)b * 1024 + w] = bits;
        c += popc32(bits);
      }
      sm[tid] = c;
    });
    env.phase([&](int tid, int&) {
      if (tid == 0) {
        int s = 0;
        for (int i = 0; i < kThreads; ++i) s += sm[i];
        p.counts[b] = s;
      }
    });
  }
};

// ---------------------------------------------------------------------------
// Distortion losses, metrics and gradient seeds (see include/nvf_b200.h).
//   main head  utils/loss.py:94-111  l = -a (1-F)^2 (dist + [occ]) ln F
//   aux heads  utils/loss.py:61-72   l = -a (1-F)^2 ln F on max-pooled GT (NVFPCC.py:81-85)
//   F = max(F0,1e-9), F0 = p (occupied) | 1-p (empty); a = alpha | 1-alpha (fp32)
//   dl/dp = -+ a w ((1-F)^2/F - 2(1-F) ln F), zero where the clamp is active.
// One CTA per block; per-block partial sums are reduced in fixed order.
// ---------------------------------------------------------------------------
struct LossParams {
  const float* out;   // [n][32768]
  const float* cls1;  // [n][4096]
  const float* cls0;  // [n][512]
  const float* gt;    // [n][32768]
  const float* dist;  // [n][32768]
  float* g_out;       // or null
  float* g_cls1;
  float* g_cls0;
  double* partial;    // [n * kLossChunks][NVF_LOSS_SUMS]
  float alpha_main, alpha_aux, thh_metric;
  int32_t n;
};

NVF_HD void focal_term(float p, bool occ, float a_occ, float a_emp, float w, float& loss, float& dldp) {
  const float F0 = occ ? p : 1.f - p;
  const float a = occ ? a_occ : a_emp;
  const bool clamped = F0 < 1e-9f;
  const float Fv = clamped ? 1e-9f : F0;
  const float om = 1.f - Fv;
  const float lg = logf(Fv);
  loss = -a * om * om * w * lg;
  const float dF = -a * w * (om * om / Fv - 2.f * om * lg);
  dldp = clamped ? 0.f : (occ ? dF : -dF);
}

constexpr int kLossChunks = 16;  // CTAs per block: chunk c covers main-head slices 2c, 2c+1 and the aux voxels below them
struct LossBlock {
  // smem: kThreads * NVF_LOSS_SUMS doubles
  template <class Env>
  static NVF_HD void run(Env& env, const LossParams& p, double* sm, int bc) {
    const int b = bc / kLossChunks, chunk = bc % kLossChunks;
    env.phase([&](int tid, int&) {
      double s[NVF_LOSS_SUMS];
      for (int i = 0; i < NVF_LOSS_SUMS; ++i) s[i] = 0.0;
      const float a_occ = p.alpha_main, a_emp = 1.f - p.alpha_main;
      const float x_occ = p.alpha_aux, x_emp = 1.f - p.alpha_aux;
      const float* gt = p.gt + (int64_t)b * kVox;
      const float* dist = p.dist + (int64_t)b * kVox;
      const float* out = p.out + (int64_t)b * kVox;
      for (int v = chunk * (kVox / kLossChunks) + tid; v < (chunk + 1) * (kVox / kLossChunks); v += kThreads) {
        const bool occ = gt[v] != 0.f;
        const float pr = out[v], d = dist[v];
        float l, g;
        focal_term(pr, occ, a_occ, a_emp, d + (occ ? 1.f : 0.f), l, g);
        s[0] += l;
        if (p.g_out) p.g_out[(int64_t)b * kVox + v] = g;
        if (pr > p.thh_metric) { s[3] += (double)(d * d); s[4] += 1.0; }
        if (occ) { s[6] += 1.0; if (pr > 0.5f) s[5] += 1.0; }
        else { s[8] += 1.0; if (!(pr > 0.5f)) s[7] += 1.0; }
      }
      // 16^3 head (cls1): GT = max over 2x2x2
      for (int v = chunk * (4096 / kLossChunks) + tid; v < (chunk + 1) * (4096 / kLossChunks); v += kThreads) {
        const int z = v >> 8, y = (v >> 4) & 15, x = v & 15;
        bool occ = false;
        for (int dz = 0; dz < 2; ++dz)
          for (int dy = 0; dy < 2; ++dy)
            for (int dx = 0; dx < 2; ++dx)
              occ = occ || gt[((2 * z + dz) * 32 + 2 * y + dy) * 32 + 2 * x + dx] != 0.f;
        const float pr = p.cls1[(int64_t)b * 4096 + v];
        float l, g;
        focal_term(pr, occ, x_occ, x_emp, 1.f, l, g);
        s[2] += l;
        if (p.g_cls1) p.g_cls1[(int64_t)b * 4096 + v] = g;
        if (occ) { s[14] += 1.0; if (pr > 0.5f) s[13] += 1.0; }
        else { s[16] += 1.0; if (!(pr > 0.5f)) s[15] += 1.0; }
      }
      // 8^3 head (cls0): GT = max over 4x4x4
      for (int v = chunk * (512 / kLossChunks) + tid; v < (chunk + 1) * (512 / kLossChunks); v += kThreads) {
        const int z = v >> 6, y = (v >> 3) & 7, x = v & 7;
        bool occ = false;
        for (int dz = 0; dz < 4; ++dz)
          for (int dy = 0; dy < 4; ++dy)
            for (int dx = 0; dx < 4; ++dx)
              occ = occ || gt[((4 * z + dz) * 32 + 4 * y + dy) * 32 + 4 * x + dx] != 0.f;
        const float pr = p.cls0[(int64_t)b * 512 + v];
        float l, g;
        focal_term(pr, occ, x_occ, x_emp, 1.f, l, g);
        s[1] += l;
        if (p.g_cls0) p.g_cls0[(int64_t)b * 512 + v] = g;
        if (occ) { s[10] += 1.0; if (pr > 0.5f) s[9] += 1.0; }
        else { s[12] += 1.0; if (!(pr > 0.5f)) s[11] += 1.0; }
      }
      for (int i = 0; i < NVF_LOSS_SUMS; ++i) sm[i * kThreads + tid] = s[i];
    });
    for (int stride = kThreads / 2; stride >= 1; stride >>= 1) {
      env.phase([&](int tid, int&) {
        if (tid < stride)
          for (int i = 0; i < NVF_LOSS_SUMS; ++i) sm[i * kThreads + tid] += sm[i * kThreads + tid + stride];
      });
    }
    env.phase([&](int tid, int&) {
      if (tid < NVF_LOSS_SUMS) p.partial[(int64_t)bc * NVF_LOSS_SUMS + tid] = sm[tid * kThreads];
    });
  }
};
// final fixed-order reduction of the per-block partials: sums[i] = sum_b partial[b][i]
struct LossFinalKernel {
  struct Params {
    const double* partial;
    double* sums;
    int32_t n;
  };
  // launched with kGrid CTAs: one warp per sum, lanes stride over the partials, fixed-order shuffle tree
  // (deterministic; a single thread per sum was a serial chain of n dependent double adds - 20 k of them
  // in the full-batch embedding step)
  static constexpr int kGrid = (NVF_LOSS_SUMS * 32 + kThreads - 1) / kThreads;
  static NVF_HD void thread(const Params& p, int bid, int tid, int nbid) {
#if defined(__CUDA_ARCH__)
    const int w = (bid * kThreads + tid) >> 5, lane = tid & 31;
    if (w >= NVF_LOSS_SUMS) return;
    double s = 0.0;
    for (int b = lane; b < p.n; b += 32) s += p.partial[(int64_t)b * NVF_LOSS_SUMS + w];
    for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) p.sums[w] = s;
#else
    if (bid != 0 || tid >= NVF_LOSS_SUMS) return;
    double s = 0.0;
    for (int b = 0; b < p.n; ++b) s += p.partial[(int64_t)b * NVF_LOSS_SUMS + tid];
    p.sums[tid] = s;
#endif
  }
};

// ---------------------------------------------------------------------------
// geometry / workspace layouts shared by the host launchers
// ---------------------------------------------------------------------------
inline bool generic_supported(const NvfDesc& d) {
  auto ok = [](int c) { return c == 8 || c == 16 || c == 32; };
  return d.ch >= 1 && d.ch <= 16 && ok(d.c0) && ok(d.c1) && ok(d.c2) && ok(d.c3);
}

// per-block activation stash (floats)
struct Stash {
  int64_t x0, a0, a1, a2, a3, a4, a5, per_block;
  static Stash make(const NvfDesc& d) {
    Stash s{};
    int64_t o = 0;
    s.x0 = o; o += (int64_t)d.c0 * 64;
    s.a0 = o; o += (int64_t)d.c0 * 64;
    s.a1 = o; o += (int64_t)d.c1 * 512;
    s.a2 = o; o += (int64_t)d.c2 * 19 * 19 * 20;
    s.a3 = o; o += (int64_t)d.c2 * 4096;
    s.a4 = o; o += (int64_t)d.c3 * 35 * 35 * 36;
    s.a5 = o; o += (int64_t)d.c3 * 32768;
    s.per_block = o;
    return s;
  }
};

// The decoder's nine convolutions in NvfParamSet order; the auxiliary heads cls1 and cls0 come last.
enum ConvLayer { L_UP0, L_CONV0, L_UP1, L_CONV1, L_UP2, L_CONV2, L_CLS2, L_CLS1, L_CLS0 };
struct ConvGeom {
  int A, B, K;   // PyTorch weight (A, B, K, K, K): convT (Cin, Cout, ...), conv (Cout, Cin, ...)
  bool convT;
  int nb;        // bias length
  int slot;      // index of the layer's `_w` pointer in NvfWeights / NvfWeightGrads; `_b` is the next one
  constexpr int K3() const { return K * K * K; }
  constexpr int64_t n() const { return (int64_t)A * B * K3(); }   // weight elements
};
constexpr ConvGeom conv_geom(const NvfDesc& d, int l) {
  const ConvGeom g[NVF_NUM_CONV] = {
      // A     B   K  convT    nb  slot
      {d.ch, d.c0, 5, true, d.c0, 0},     // up0
      {d.c0, d.c1, 5, true, d.c1, 4},     // conv0 (igdn_beta, igdn_gamma sit in slots 2, 3)
      {d.c1, d.c2, 5, true, d.c2, 6},     // up1
      {d.c2, d.c2, 4, false, d.c2, 8},    // conv1
      {d.c2, d.c3, 5, true, d.c3, 10},    // up2
      {d.c3, d.c3, 4, false, d.c3, 12},   // conv2
      {1, d.c3, 3, false, 1, 14},         // cls2 (conv2_cls)
      {1, d.c2, 3, false, 1, 16},         // cls1 (conv1_cls)
      {1, d.c1, 3, false, 1, 18},         // cls0 (conv0_cls)
  };
  return g[l];
}

// NvfWeights / NvfWeightGrads as the array of their pointers in field order
constexpr int kEffTensors = 20;
template <class W>
auto slots(W& w) {
  return reinterpret_cast<std::remove_reference_t<decltype((w.up0_w))>*>(&w);
}
static_assert(sizeof(NvfWeights) == kEffTensors * sizeof(float*) && sizeof(NvfWeightGrads) == sizeof(NvfWeights),
              "NvfWeights / NvfWeightGrads are plain arrays of pointers");
#define NVF_CHECK_SLOT(l, f)                                                                          \
  static_assert(offsetof(NvfWeights, f##_w) == conv_geom(NvfDesc{}, l).slot * sizeof(float*) &&      \
                    offsetof(NvfWeights, f##_b) == offsetof(NvfWeights, f##_w) + sizeof(float*) &&    \
                    offsetof(NvfWeightGrads, f##_w) == offsetof(NvfWeights, f##_w) &&                 \
                    offsetof(NvfWeightGrads, f##_b) == offsetof(NvfWeights, f##_b),                   \
                #f " slot of conv_geom")
NVF_CHECK_SLOT(L_UP0, up0);
NVF_CHECK_SLOT(L_CONV0, conv0);
NVF_CHECK_SLOT(L_UP1, up1);
NVF_CHECK_SLOT(L_CONV1, conv1);
NVF_CHECK_SLOT(L_UP2, up2);
NVF_CHECK_SLOT(L_CONV2, conv2);
NVF_CHECK_SLOT(L_CLS2, cls2);
NVF_CHECK_SLOT(L_CLS1, cls1);
NVF_CHECK_SLOT(L_CLS0, cls0);
#undef NVF_CHECK_SLOT

// packed weights for the layer-wise path (forward + dgrad layouts of every layer), floats
struct GenericPacked {
  int64_t fwd[NVF_NUM_CONV], dg[NVF_NUM_CONV];   // by ConvLayer
  int64_t cls_is;  // PACK_CLS_IS copy of cls2 for the fused decode head
  int64_t total;
  static GenericPacked make(const NvfDesc& d) {
    GenericPacked g{};
    int64_t o = 0;
    auto take = [&](int64_t n) { int64_t r = o; o += (n + 3) / 4 * 4; return r; };
    for (int l = 0; l < NVF_NUM_CONV; ++l) g.fwd[l] = take(conv_geom(d, l).n());
    for (int l = 0; l < NVF_NUM_CONV; ++l) g.dg[l] = take(conv_geom(d, l).n());
    g.cls_is = take((int64_t)d.c3 * 36);
    g.total = o;
    return g;
  }
  static int64_t floats(const NvfDesc& d) { return make(d).total; }
};

}  // namespace nvf
