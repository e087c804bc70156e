// Host-side orchestration of the C ABI (include/nvf_b200.h), templated on a
// launcher so that the CUDA build (nvf_capi.cu) and the test-only CPU emulator
// (tests/emu/nvf_emu.cpp) execute the same sequencing, workspace layouts and
// weight packing.
#pragma once
#include <stdlib.h>
#include "../../include/nvf_b200.h"
#include "nvf_common.h"
#include "nvf_emit.h"
#include "nvf_layers.h"

namespace nvf {

constexpr int kMaxCtas = 160;  // upper bound on persistent CTAs (B200: 148 SMs)
constexpr size_t kAlign = 256;
inline size_t align_up(size_t v) { return (v + kAlign - 1) / kAlign * kAlign; }
constexpr int64_t kGenericDecodeChunk = 128;  // blocks per pass of the layer-wise decode path
// per-leaf scratch of the two-pass (wide) head: conv2 rows next to the cut + their partial logits
inline size_t head_brow_floats(const NvfDesc& d) { return d.c3 == 16 ? (size_t)2 * d.c3 * 1024 : 0; }
inline size_t head_pl_floats(const NvfDesc& d) { return d.c3 == 16 ? (size_t)2048 : 0; }
// blocks per pass of the fused-head decode path: the stem activations of a pass live in the workspace (8,16,8,8:
// 0.6 MB per block; 16,32,16,16: 1.4 MB), so a cloud is one pass up to 8 GiB of them (vox11 wide: 6.7 GB) and is
// otherwise cut into EQUAL passes - every pass ends with one partial round of the head kernel, and equal passes keep
// those few
inline int64_t head_chunk(const NvfDesc& d, int64_t n) {
  const int64_t per_block = 4 * (Stash::make(d).a4 + (int64_t)d.c2 * 16 * 480 + (int64_t)head_brow_floats(d) + (int64_t)head_pl_floats(d));
  int64_t cmax = ((int64_t)8 << 30) / per_block;
  if (cmax < 148) cmax = 148;
  if (const char* e = getenv("NVF_DECODE_PASS_LEAVES")) {   // tests: force several passes on a small cloud
    const long v = atol(e);
    if (v > 0) cmax = v;
  }
  if (n <= cmax) return n;
  const int64_t passes = (n + cmax - 1) / cmax;
  return (n + passes - 1) / passes;
}
// configurations the warp-specialised fused decode head (nvf_decode_head.cuh) is instantiated for
inline bool head_cfg(const NvfDesc& d) { return (d.c2 == 8 && d.c3 == 8) || (d.c2 == 16 && d.c3 == 16); }
constexpr int kQueueSlots = 16;                // work-queue slots (16 bytes each) of one forward / backward pass
constexpr int kMaxPartialCtas = 304;          // persistent CTAs of a split-K weight-gradient kernel (2 per SM)
// scratch for the split-K partial results of one backward pass: every weight-gradient kernel
// writes <= kMaxPartialCtas partial copies of its layer's gradient; per-block partials of the
// stem / bias sums need n-proportional room.
inline size_t partial_floats(const NvfDesc& d, int64_t n) {
  size_t params = 2 * (size_t)(d.c0 + d.c1 + d.c2 + d.c3) + 64 * 24;
  for (int l = 0; l < NVF_NUM_CONV; ++l) params += (size_t)conv_geom(d, l).n();
  const size_t stem = (size_t)d.c0 * d.c1 * 125 + d.c1 + (size_t)d.c0 * d.c0 + d.c0 + (size_t)d.ch * d.c0 * 125 + d.c0;
  return (size_t)kMaxPartialCtas * params +
         (size_t)n * (stem + (size_t)d.c0 * d.c0 + 8 * (size_t)(d.c0 + d.c1 + d.c2 + d.c3) + 64 * 16);
}

struct DecodeWs {
  size_t off_packed, off_scratch, off_sp, off_brow, off_pl, off_mask, off_offsets, total;
  // head: stem layers batched over a chunk of blocks (stash up to conv1's output), then the fused head kernel
  static DecodeWs make(const NvfDesc& d, int64_t n, bool head) {
    DecodeWs L{};
    size_t o = 0;
    L.off_packed = o;
    o += align_up(sizeof(float) * (size_t)GenericPacked::floats(d));
    L.off_scratch = o;
    if (head) {
      const int64_t chunk = head_chunk(d, n);
      o += align_up(sizeof(float) * (size_t)Stash::make(d).a4 * (size_t)chunk);
      L.off_sp = o;
      o += align_up(sizeof(float) * (size_t)d.c2 * 16 * 480 * (size_t)chunk);
      L.off_brow = o;
      o += align_up(sizeof(float) * head_brow_floats(d) * (size_t)chunk);
      L.off_pl = o;
      o += align_up(sizeof(float) * head_pl_floats(d) * (size_t)chunk);
    } else {
      const int64_t chunk = n < kGenericDecodeChunk ? n : kGenericDecodeChunk;
      o += align_up(sizeof(float) * (size_t)(Stash::make(d).per_block + kVox) * (size_t)chunk);
    }
    L.off_mask = o;
    o += align_up(sizeof(uint32_t) * 1024 * (size_t)n);
    L.off_offsets = o;
    o += align_up(sizeof(int64_t) * (size_t)(n + 1));
    L.total = o;
    return L;
  }
};

struct TrainWs {
  size_t off_packed, off_stash, off_grad, off_tmp3, off_tmp1, off_gl2, off_gl1, off_gl0, off_p2, off_p1, off_p0, off_loss, off_partial, off_queue, total;
  static TrainWs make(const NvfDesc& d, int64_t n) {
    TrainWs L{};
    const Stash s = Stash::make(d);
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes); return r; };
    L.off_packed = take(sizeof(float) * (size_t)GenericPacked::floats(d));
    L.off_stash = take(sizeof(float) * (size_t)s.per_block * n);
    L.off_grad = take(sizeof(float) * (size_t)s.per_block * n);
    L.off_tmp3 = take(sizeof(float) * (size_t)d.c2 * 4096 * n);
    L.off_tmp1 = take(sizeof(float) * (size_t)d.c1 * 512 * n);
    L.off_gl2 = take(sizeof(float) * (size_t)kVox * n);
    L.off_gl1 = take(sizeof(float) * (size_t)4096 * n);
    L.off_gl0 = take(sizeof(float) * (size_t)512 * n);
    L.off_p2 = take(sizeof(float) * (size_t)kVox * n);   // probabilities of the three heads (forward -> backward)
    L.off_p1 = take(sizeof(float) * (size_t)4096 * n);
    L.off_p0 = take(sizeof(float) * (size_t)512 * n);
    L.off_loss = take(sizeof(double) * (size_t)NVF_LOSS_SUMS * (n * kLossChunks + 1));
    L.off_partial = take(sizeof(float) * partial_floats(d, n));
    L.off_queue = take(2 * 16 * kQueueSlots);   // forward slots, then backward slots
    L.total = o;
    return L;
  }
};

// arguments of the fused decode head (mirrors fast::HeadParams, which only the CUDA build sees)
struct HeadArgs {
  const float *sp, *w_up2, *w_c2, *w_cls, *up2_b, *conv2_b, *cls2_b;
  float* prob_out;
  uint32_t* mask_out;
  int32_t* counts_out;
  float *brow, *pl;
  float thh;
  int32_t n_blocks;
};

template <class L>
struct Api {
  static void layer(L& l, const LayerParams& p) {
    if (l.fast_layer(p)) return;
    // generic kernel: the per-thread channel tile shrinks when the layer is too small to fill the GPU
    const int64_t pos = (int64_t)p.n * p.Dout * p.Dout * ((p.Dout + 3) / 4);
    const int64_t want = (int64_t)l.sms() * 2 * kThreads;
    if (p.CO % 16 == 0 && pos * (p.CO / 16) >= want) l.template layer<16>(p);
    else if (p.CO % 8 == 0 && pos * (p.CO / 8) >= want) l.template layer<8>(p);
    else if (p.CO % 4 == 0) l.template layer<4>(p);
    else l.template layer<1>(p);
  }
  // weight gradient + bias gradient (db = per-channel sum of the output gradient `c.g`)
  // Runs on the auxiliary stream: weight gradients only feed the final reduction, not the dgrad chain.
  static void wgrad_bias(L& l, const WgradParams& p, const ChanSumParams& c) {
    l.side_begin();
    if (!l.fast_wgrad(p, c)) {
      wgrad(l, p);
      l.chansum(c, c.C);
    }
    l.side_end();
  }
  static void wgrad(L& l, const WgradParams& p) {
    const bool c8 = p.CA % 8 == 0;
    const int groups = c8 ? p.CA / 8 : p.CA;
    const int grid = groups * p.CS * p.K * p.K;
    if (p.K == 3) { if (c8) l.template wgrad<8, 3>(p, grid); else l.template wgrad<1, 3>(p, grid); }
    else if (p.K == 4) { if (c8) l.template wgrad<8, 4>(p, grid); else l.template wgrad<1, 4>(p, grid); }
    else { if (c8) l.template wgrad<8, 5>(p, grid); else l.template wgrad<1, 5>(p, grid); }
  }

  static int pack_all(L& l, const NvfDesc& d, const NvfWeights& w, float* packed, bool fwd_aux, bool dgrad) {
    const GenericPacked g = GenericPacked::make(d);
    PackParams pp{};
    auto job = [&](int i, int64_t off, int mode) {
      const ConvGeom c = conv_geom(d, i);
      if (pp.njobs == kMaxPackJobs) { l.pack(pp); pp.njobs = 0; }
      pp.job[pp.njobs++] = PackJob{slots(w)[c.slot], packed + off, mode, c.A, c.B, c.K};
    };
    for (int i = 0; i < (fwd_aux ? NVF_NUM_CONV : L_CLS1); ++i)
      job(i, g.fwd[i], conv_geom(d, i).convT ? PACK_CONVT_FWD : PACK_CONV_FWD);
    if (dgrad)
      for (int i = 0; i < NVF_NUM_CONV; ++i) job(i, g.dg[i], conv_geom(d, i).convT ? PACK_CONVT_DGRAD : PACK_CONV_DGRAD);
    if (pp.njobs) l.pack(pp);
    return NVF_OK;
  }

  // Layer-wise forward over `n` blocks.  stash: n * Stash::per_block floats.
  // p2/p1/p0: optional second copies of the three heads' probabilities (kept for the backward pass)
  static void forward_layers(L& l, const NvfDesc& d, const NvfWeights& w, const float* packed, const float* latent,
                             int n, float* stash, float* out, float* cls1, float* cls0, float* p2 = nullptr,
                             float* p1 = nullptr, float* p0 = nullptr, bool stem_only = false,
                             float* pad_scratch = nullptr) {
    const Stash s = Stash::make(d);
    const GenericPacked g = GenericPacked::make(d);
    // NOTE: the stash is laid out tensor-major ([tensor][n][...]) so that every layer sees a dense batch.
    float* x0 = stash + s.x0 * n; float* a0 = stash + s.a0 * n; float* a1 = stash + s.a1 * n;
    float* a2 = stash + s.a2 * n; float* a3 = stash + s.a3 * n; float* a4 = stash + s.a4 * n;
    float* a5 = stash + s.a5 * n;
    LayerParams p{};
    p.n = n;
    if (!l.fast_stem_fwd(d, w, packed + g.fwd[L_UP0], packed + g.fwd[L_CONV0], packed + g.fwd[L_CLS0], latent, n, x0,
                         a0, a1, cls0, p0)) {
      // up0: convT k5 s2 p2 op1 (utils/network.py:4671-4680)
      p = LayerParams{latent, x0, packed + g.fwd[L_UP0], w.up0_b, nullptr, nullptr, n, d.ch, d.c0, 2, 2, 4, 4, 2, ACT_NONE, OP_CONVT};
      layer(l, p);
      IgdnParams ip{x0, a0, nullptr, w.igdn_beta, w.igdn_gamma, nullptr, nullptr, n, d.c0};
      l.template generic<IgdnFwdKernel>(ip, (int)((int64_t)n * d.c0 * 64 + kThreads - 1) / kThreads);
      // conv0: convT k5 s2 p2 op1 + ReLU (:4682-4691, :4760)
      p = LayerParams{a0, a1, packed + g.fwd[L_CONV0], w.conv0_b, nullptr, nullptr, n, d.c0, d.c1, 4, 4, 8, 8, 2, ACT_RELU, OP_CONVT};
      layer(l, p);
      if (cls0) {  // conv0_cls + sigmoid (:4743-4751, :4761)
        p = LayerParams{a1, cls0, packed + g.fwd[L_CLS0], w.cls0_b, nullptr, nullptr, n, d.c1, 1, 8, 8, 8, 8, 1, ACT_SIGMOID, OP_CORR3};
        p.out2 = p0;
        layer(l, p);
      }
    }
    // up1: convT k5 s2 p0 + ReLU (:4693-4700, :4762)
    p = LayerParams{a1, a2, packed + g.fwd[L_UP1], w.up1_b, nullptr, nullptr, n, d.c1, d.c2, 8, 8, 19, 20, 0, ACT_RELU, OP_CONVT};
    // fused-head decode (pad_scratch): polyphase kernel on a zero-padded copy of conv0's output; else the tile kernels
    if (!(pad_scratch && l.up_poly(p, pad_scratch))) layer(l, p);
    // conv1: conv k4 + ReLU (:4702-4710, :4763)
    p = LayerParams{a2, a3, packed + g.fwd[L_CONV1], w.conv1_b, nullptr, nullptr, n, d.c2, d.c2, 19, 20, 16, 16, 0, ACT_RELU, OP_CORR4};
    layer(l, p);
    if (cls1) {  // conv1_cls + sigmoid (:4733-4741, :4764)
      p = LayerParams{a3, cls1, packed + g.fwd[L_CLS1], w.cls1_b, nullptr, nullptr, n, d.c2, 1, 16, 16, 16, 16, 1, ACT_SIGMOID, OP_CORR3};
      p.out2 = p1;
      l.side_begin();   // auxiliary head: off the critical path
      layer(l, p);
      l.side_end();
    }
    if (stem_only) {   // the fused decode head takes over from conv1's output
      l.join();
      return;
    }
    // up2: convT k5 s2 p0 + ReLU (:4712-4719, :4765)
    p = LayerParams{a3, a4, packed + g.fwd[L_UP2], w.up2_b, nullptr, nullptr, n, d.c2, d.c3, 16, 16, 35, 36, 0, ACT_RELU, OP_CONVT};
    layer(l, p);
    // conv2: conv k4 + ReLU (:4721-4729, :4766)
    p = LayerParams{a4, a5, packed + g.fwd[L_CONV2], w.conv2_b, nullptr, nullptr, n, d.c3, d.c3, 35, 36, 32, 32, 0, ACT_RELU, OP_CORR4};
    layer(l, p);
    // conv2_cls + sigmoid (:4731, :4767-4768)
    p = LayerParams{a5, out, packed + g.fwd[L_CLS2], w.cls2_b, nullptr, nullptr, n, d.c3, 1, 32, 32, 32, 32, 1, ACT_SIGMOID, OP_CORR3};
    p.out2 = p2;
    layer(l, p);
    l.join();
  }

  static int decode(L& l, const NvfDesc* desc, const NvfWeights* w, const float* latent, const int32_t* origins,
                    int64_t n_blocks, float thh, float* prob_out, uint32_t* mask_out, int32_t* counts_out,
                    int32_t* coords_out, int64_t cap, int64_t* total_out, void* workspace, size_t workspace_bytes) {
    if (!desc || !w || !workspace || n_blocks < 0 || cap < 0) return NVF_ERR_INVALID_ARG;
    if (n_blocks > 0 && (!latent || !counts_out)) return NVF_ERR_INVALID_ARG;  // empty input: nothing to read
    if (n_blocks > 0x7fffffff / 1024) return NVF_ERR_INVALID_ARG;
    if (!generic_supported(*desc)) return NVF_ERR_UNSUPPORTED;
    const bool head = l.has_head(*desc);
    const DecodeWs W = DecodeWs::make(*desc, n_blocks, head);
    if (workspace_bytes < W.total) return NVF_ERR_WORKSPACE;
    char* ws = (char*)workspace;
    float* packed = (float*)(ws + W.off_packed);
    uint32_t* mask = mask_out ? mask_out : (uint32_t*)(ws + W.off_mask);
    int64_t* offsets = (int64_t*)(ws + W.off_offsets);
    if (n_blocks > 0) {
      if (head) {
        // stem (up0 .. conv1, 13 % of the multiply-adds) as batched layer kernels over a chunk of blocks, then
        // one persistent fused kernel per chunk for up2 -> conv2 -> conv2_cls -> sigmoid -> threshold
        const GenericPacked g = GenericPacked::make(*desc);
        pack_all(l, *desc, *w, packed, false, false);
        PackParams pp{};
        pp.job[pp.njobs++] = PackJob{w->cls2_w, packed + g.cls_is, PACK_CLS_IS, 1, desc->c3, 3};
        l.pack(pp);
        const int64_t chunk = head_chunk(*desc, n_blocks);
        float* stash = (float*)(ws + W.off_scratch);
        float* sp = (float*)(ws + W.off_sp);
        l.zero_ints(counts_out, n_blocks);
        for (int64_t b0 = 0; b0 < n_blocks; b0 += chunk) {
          const int nb = (int)(n_blocks - b0 < chunk ? n_blocks - b0 : chunk);
          forward_layers(l, *desc, *w, packed, latent + b0 * desc->ch * 8, nb, stash, nullptr, nullptr, nullptr, nullptr,
                         nullptr, nullptr, true, sp);   // sp doubles as the padded conv0 output until conv1 is done
          l.pad_conv1(stash + Stash::make(*desc).a3 * nb, sp, (int64_t)nb * desc->c2 * 16);
          HeadArgs ha{sp, packed + g.fwd[L_UP2], packed + g.fwd[L_CONV2], packed + g.cls_is, w->up2_b, w->conv2_b, w->cls2_b,
                      prob_out ? prob_out + b0 * kVox : nullptr, mask + b0 * 1024, counts_out + b0,
                      (float*)(ws + W.off_brow), (float*)(ws + W.off_pl), thh, nb};
          // always one CTA per SM: with fewer (leaf, pass) units than SMs the kernel cuts them along z
          l.head(*desc, ha, l.sms() < kMaxCtas ? l.sms() : kMaxCtas);
        }
      } else {
        pack_all(l, *desc, *w, packed, false, false);
        const int64_t chunk = n_blocks < kGenericDecodeChunk ? n_blocks : kGenericDecodeChunk;
        float* stash = (float*)(ws + W.off_scratch);
        float* prob_tmp = stash + Stash::make(*desc).per_block * chunk;
        for (int64_t b0 = 0; b0 < n_blocks; b0 += chunk) {
          const int nb = (int)(n_blocks - b0 < chunk ? n_blocks - b0 : chunk);
          float* pr = prob_out ? prob_out + b0 * kVox : prob_tmp;
          forward_layers(l, *desc, *w, packed, latent + b0 * desc->ch * 8, nb, stash, pr, nullptr, nullptr);
          MaskParams mp{pr, mask + b0 * 1024, counts_out + b0, thh, nb};
          l.mask(mp, nb);
        }
      }
    }
    EmitParams ep{};
    ep.mask = mask;
    ep.counts = counts_out;
    ep.origins = origins;
    ep.offsets = offsets;
    ep.coords = coords_out;
    ep.total_out = total_out;
    ep.cap = cap;
    ep.n_blocks = (int32_t)n_blocks;
    l.scan(ep);
    if (n_blocks > 0 && coords_out) l.emit(ep, (int)n_blocks);
    return l.error();
  }

  static int emit_points(L& l, const uint32_t* mask, const int32_t* counts, const int32_t* origins, int64_t n_blocks,
                         int32_t* coords_out, int64_t cap, int64_t* total_out, void* workspace,
                         size_t workspace_bytes) {
    if (!mask || !counts || !workspace || n_blocks < 0 || cap < 0) return NVF_ERR_INVALID_ARG;
    if (workspace_bytes < sizeof(int64_t) * (size_t)(n_blocks + 1)) return NVF_ERR_WORKSPACE;
    EmitParams ep{};
    ep.mask = mask;
    ep.counts = counts;
    ep.origins = origins;
    ep.offsets = (int64_t*)workspace;
    ep.coords = coords_out;
    ep.total_out = total_out;
    ep.cap = cap;
    ep.n_blocks = (int32_t)n_blocks;
    l.scan(ep);
    if (n_blocks > 0 && coords_out) l.emit(ep, (int)n_blocks);
    return l.error();
  }

  static int train_forward(L& l, const NvfDesc* desc, const NvfWeights* w, const float* latent, int64_t n, float* out,
                           float* cls1, float* cls0, void* workspace, size_t workspace_bytes) {
    if (!desc || !w || !latent || !out || !cls1 || !cls0 || !workspace || n <= 0 || n > 1 << 20) return NVF_ERR_INVALID_ARG;
    if (!w->cls1_w || !w->cls0_w || !w->cls1_b || !w->cls0_b) return NVF_ERR_INVALID_ARG;
    if (!generic_supported(*desc)) return NVF_ERR_UNSUPPORTED;
    const TrainWs W = TrainWs::make(*desc, n);
    if (workspace_bytes < W.total) return NVF_ERR_WORKSPACE;
    char* ws = (char*)workspace;
    float* packed = (float*)(ws + W.off_packed);
    l.zero_queue(ws + W.off_queue, 2 * 16 * kQueueSlots);   // the caller's workspace is not zero-filled on this path
    l.set_queue(ws + W.off_queue);
    pack_all(l, *desc, *w, packed, true, true);
    forward_layers(l, *desc, *w, packed, latent, (int)n, (float*)(ws + W.off_stash), out, cls1, cls0,
                   (float*)(ws + W.off_p2), (float*)(ws + W.off_p1), (float*)(ws + W.off_p0));
    return l.error();
  }

  static int loss_seeds(L& l, const float* out, const float* cls1, const float* cls0, const float* gt,
                        const float* dist, int64_t n, float alpha_main, float alpha_aux, float thh_metric,
                        double* sums_out, float* g_out, float* g_cls1, float* g_cls0, void* workspace,
                        size_t workspace_bytes) {
    if (!out || !cls1 || !cls0 || !gt || !dist || !sums_out || !workspace || n <= 0) return NVF_ERR_INVALID_ARG;
    if (workspace_bytes < sizeof(double) * NVF_LOSS_SUMS * (size_t)n * kLossChunks) return NVF_ERR_WORKSPACE;
    LossParams lp{out, cls1, cls0, gt, dist, g_out, g_cls1, g_cls0, (double*)workspace, alpha_main, alpha_aux,
                  thh_metric, (int32_t)n};
    l.loss(lp, (int)n * kLossChunks);
    LossFinalKernel::Params fp{(const double*)workspace, sums_out, (int32_t)n * kLossChunks};
    l.template generic<LossFinalKernel>(fp, LossFinalKernel::kGrid);
    return l.error();
  }

  static int train_backward(L& l, const NvfDesc* desc, const NvfWeights* w, const float* latent, int64_t n64,
                            const float* g_out, const float* g_cls1, const float* g_cls0, int flags,
                            const NvfWeightGrads* gw, float* g_latent, void* workspace, size_t workspace_bytes) {
    if (!desc || !w || !latent || !workspace || n64 <= 0 || n64 > 1 << 20) return NVF_ERR_INVALID_ARG;
    if ((flags & NVF_BWD_WGRAD) && !gw) return NVF_ERR_INVALID_ARG;
    if ((flags & NVF_BWD_DLATENT) && !g_latent) return NVF_ERR_INVALID_ARG;
    if (!generic_supported(*desc)) return NVF_ERR_UNSUPPORTED;
    const NvfDesc& d = *desc;
    const int n = (int)n64;
    const TrainWs W = TrainWs::make(d, n);
    if (workspace_bytes < W.total) return NVF_ERR_WORKSPACE;
    char* ws = (char*)workspace;
    const float* packed = (const float*)(ws + W.off_packed);
    const GenericPacked g = GenericPacked::make(d);
    const Stash s = Stash::make(d);
    const float* stash = (const float*)(ws + W.off_stash);
    float* grad = (float*)(ws + W.off_grad);
    const float *x0 = stash + s.x0 * n, *a0 = stash + s.a0 * n, *a1 = stash + s.a1 * n, *a2 = stash + s.a2 * n,
                *a3 = stash + s.a3 * n, *a4 = stash + s.a4 * n, *a5 = stash + s.a5 * n;
    float *gx0 = grad + s.x0 * n, *gy0 = grad + s.a0 * n, *g1 = grad + s.a1 * n, *g2 = grad + s.a2 * n,
          *g3 = grad + s.a3 * n, *g4 = grad + s.a4 * n, *g5 = grad + s.a5 * n;
    float* tmp3 = (float*)(ws + W.off_tmp3);
    float* tmp1 = (float*)(ws + W.off_tmp1);
    const float* gl2 = (const float*)(ws + W.off_gl2);
    const float* gl1 = (const float*)(ws + W.off_gl1);
    const float* gl0 = (const float*)(ws + W.off_gl0);
    l.set_partial((float*)(ws + W.off_partial), partial_floats(d, n));
    l.set_queue(ws + W.off_queue + 16 * kQueueSlots);
    const bool wg = (flags & NVF_BWD_WGRAD) != 0;
    LayerParams p{};
    if (flags & NVF_BWD_DLOGIT) {
      // the caller's gradients are already w.r.t. the logits (the fused step's loss kernel folds the sigmoid in)
      if (!g_out || !g_cls1 || !g_cls0) return NVF_ERR_INVALID_ARG;
      gl2 = g_out; gl1 = g_cls1; gl0 = g_cls0;
    } else {
      // the heads' probabilities were kept by nvf_train_forward: dL/dlogit = dL/dp * p (1 - p)
      SigBwd3Params sp{{g_out, g_cls1, g_cls0},
                       {(const float*)(ws + W.off_p2), (const float*)(ws + W.off_p1), (const float*)(ws + W.off_p0)},
                       {(float*)(ws + W.off_gl2), (float*)(ws + W.off_gl1), (float*)(ws + W.off_gl0)},
                       {(int64_t)n * kVox, (int64_t)n * 4096, (int64_t)n * 512}};
      int64_t grid = ((int64_t)n * (kVox + 4096 + 512) + kThreads - 1) / kThreads;
      if (grid > 4096) grid = 4096;
      l.template generic<SigBwd3Kernel>(sp, (int)grid);
    }

    // ---- conv2_cls ----
    if (wg) {
      WgradParams q{gl2, a5, gw->cls2_w, n, 1, d.c3, 32, 32, 32, 32, 3, 1, 1};
      ChanSumParams c{gl2, gw->cls2_b, n, 1, 32, 32};
      wgrad_bias(l, q, c);
    }
    p = LayerParams{gl2, g5, packed + g.dg[L_CLS2], nullptr, nullptr, a5, n, 1, d.c3, 32, 32, 32, 32, 1, ACT_NONE, OP_CORR3};
    layer(l, p);
    // ---- conv2 ----
    if (wg) {
      WgradParams q{g5, a4, gw->conv2_w, n, d.c3, d.c3, 32, 32, 35, 36, 4, 1, 0};
      ChanSumParams c{g5, gw->conv2_b, n, d.c3, 32, 32};
      wgrad_bias(l, q, c);
    }
    p = LayerParams{g5, g4, packed + g.dg[L_CONV2], nullptr, nullptr, a4, n, d.c3, d.c3, 32, 32, 35, 36, 3, ACT_NONE, OP_CORR4};
    layer(l, p);
    // ---- up2 (+ conv1_cls branch) ----
    if (wg) {
      WgradParams q{a3, g4, gw->up2_w, n, d.c2, d.c3, 16, 16, 35, 36, 5, 2, 0};
      ChanSumParams c{g4, gw->up2_b, n, d.c3, 35, 36};
      wgrad_bias(l, q, c);
      WgradParams q1{gl1, a3, gw->cls1_w, n, 1, d.c2, 16, 16, 16, 16, 3, 1, 1};
      ChanSumParams c1{gl1, gw->cls1_b, n, 1, 16, 16};
      wgrad_bias(l, q1, c1);
    }
    p = LayerParams{gl1, tmp3, packed + g.dg[L_CLS1], nullptr, nullptr, nullptr, n, 1, d.c2, 16, 16, 16, 16, 1, ACT_NONE, OP_CORR3};
    layer(l, p);
    p = LayerParams{g4, g3, packed + g.dg[L_UP2], nullptr, tmp3, a3, n, d.c3, d.c2, 35, 36, 16, 16, 0, ACT_NONE, OP_CORR_S2};
    layer(l, p);
    // ---- conv1 ----
    if (wg) {
      WgradParams q{g3, a2, gw->conv1_w, n, d.c2, d.c2, 16, 16, 19, 20, 4, 1, 0};
      ChanSumParams c{g3, gw->conv1_b, n, d.c2, 16, 16};
      wgrad_bias(l, q, c);
    }
    p = LayerParams{g3, g2, packed + g.dg[L_CONV1], nullptr, nullptr, a2, n, d.c2, d.c2, 16, 16, 19, 20, 3, ACT_NONE, OP_CORR4};
    layer(l, p);
    // ---- up1 (+ conv0_cls branch) ----
    if (wg) {
      WgradParams q{a1, g2, gw->up1_w, n, d.c1, d.c2, 8, 8, 19, 20, 5, 2, 0};
      ChanSumParams c{g2, gw->up1_b, n, d.c2, 19, 20};
      wgrad_bias(l, q, c);
      WgradParams q0{gl0, a1, gw->cls0_w, n, 1, d.c1, 8, 8, 8, 8, 3, 1, 1};
      ChanSumParams c0{gl0, gw->cls0_b, n, 1, 8, 8};
      wgrad_bias(l, q0, c0);
    }
    p = LayerParams{gl0, tmp1, packed + g.dg[L_CLS0], nullptr, nullptr, nullptr, n, 1, d.c1, 8, 8, 8, 8, 1, ACT_NONE, OP_CORR3};
    layer(l, p);
    p = LayerParams{g2, g1, packed + g.dg[L_UP1], nullptr, tmp1, a1, n, d.c2, d.c1, 19, 20, 8, 8, 0, ACT_NONE, OP_CORR_S2};
    layer(l, p);
    if (!l.fast_stem_bwd(d, *w, latent, n, x0, a0, g1, gy0, wg ? gw : nullptr, (flags & NVF_BWD_DLATENT) ? g_latent : nullptr)) {
      // ---- conv0 ----
      if (wg) {
        WgradParams q{a0, g1, gw->conv0_w, n, d.c0, d.c1, 4, 4, 8, 8, 5, 2, 2};
        ChanSumParams c{g1, gw->conv0_b, n, d.c1, 8, 8};
        wgrad_bias(l, q, c);
      }
      p = LayerParams{g1, gy0, packed + g.dg[L_CONV0], nullptr, nullptr, nullptr, n, d.c1, d.c0, 8, 8, 4, 4, 2, ACT_NONE, OP_CORR_S2};
      layer(l, p);
      // ---- IGDN ----
      {
        IgdnParams ip{x0, gx0, gy0, w->igdn_beta, w->igdn_gamma, wg ? gw->igdn_beta : nullptr,
                      wg ? gw->igdn_gamma : nullptr, n, d.c0};
        l.template generic<IgdnBwdDxKernel>(ip, (int)(((int64_t)n * d.c0 * 64 + kThreads - 1) / kThreads));
        if (wg && !l.fast_igdn_param(ip)) l.template generic<IgdnBwdParamKernel>(ip, 1);
      }
      // ---- up0 ----
      if (wg) {
        WgradParams q{latent, gx0, gw->up0_w, n, d.ch, d.c0, 2, 2, 4, 4, 5, 2, 2};
        ChanSumParams c{gx0, gw->up0_b, n, d.c0, 4, 4};
        wgrad_bias(l, q, c);
      }
      if (flags & NVF_BWD_DLATENT) {
        p = LayerParams{gx0, g_latent, packed + g.dg[L_UP0], nullptr, nullptr, nullptr, n, d.c0, d.ch, 4, 4, 2, 2, 2, ACT_NONE, OP_CORR_S2};
        layer(l, p);
      }
    }
    l.join();
    l.flush_reduce();
    return l.error();
  }
};

}  // namespace nvf
