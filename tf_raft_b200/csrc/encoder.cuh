// Feature / context encoders (tf_raft/layers/extractor.py:88-175) on the tensor-core path.
//   conv1 7x7 s2 (Cin = 3, K = 147: CUDA cores, image normalisation 2*(x/255)-1 fused into the load)
//   6 ResBlocks (extractor.py:19-49): 3x3 convs on conv_tc_kernel; stride-2 convs fetch their A operand with
//   TMA elementStrides = 2 (Keras 'same' is asymmetric there: pad 0 before / 1 after); 1x1 s2 downsample.
//   conv2 1x1.
// Norms: 'batch' in inference is a per-channel affine folded into the conv epilogue (everything fuses);
// 'instance' (and 'batch' in training) need statistics of the raw conv output: two deterministic reduction
// passes + one apply kernel that also does ReLU, the residual add and the fp16 hi/lo re-split.
#pragma once
#include <algorithm>

#include "lookup.cuh"
#include "update.cuh"

namespace raft {

enum { NORM_NONE = 0, NORM_INSTANCE = 1, NORM_BATCH = 2 };

struct EncSpec { int c0; int c[3]; int s[3]; };
inline EncSpec enc_spec(int variant) {
  if (variant == RAFT_VARIANT_BASIC) return {64, {64, 96, 128}, {1, 2, 2}};
  return {32, {32, 64, 96}, {1, 2, 2}};
}
inline int pad64(int c) { return round_up(c, 64); }

struct EncConvSlot { size_t hi, lo, bias, scale, absmax; int kh, kw, cin, cout, cin_pad, cout_pad; };
struct EncNormSlot { size_t gamma, beta, fscale, fshift; int C; };
struct EncLayout {
  EncConvSlot conv1;                          // stem as a 1x1 conv over the 147 (->192) im2col channels
  EncNormSlot norm1;
  EncConvSlot bc1[6], bc2[6], bds[6];
  EncNormSlot bn1[6], bn2[6], bnd[6];
  int has_ds[6], bcin[6], bc[6], bstride[6];
  EncConvSlot conv2;
  size_t total;
};

inline EncLayout enc_layout(int variant, int out_dim) {
  EncLayout L;
  memset(&L, 0, sizeof(L));
  const EncSpec S = enc_spec(variant);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; };
  auto conv_slot = [&](int kh, int kw, int cin, int cout) {
    EncConvSlot s;
    s.kh = kh; s.kw = kw; s.cin = cin; s.cout = cout; s.cin_pad = pad64(cin); s.cout_pad = round_up(cout, 32);
    const size_t plane = (size_t)kh * kw * s.cout_pad * s.cin_pad * sizeof(__half);
    s.hi = take(plane); s.lo = take(plane);
    s.bias = take(sizeof(float) * (s.cout_pad + 64));
    s.scale = take(2 * sizeof(float));
    s.absmax = take(sizeof(unsigned int));
    return s;
  };
  auto norm_slot = [&](int C) {
    EncNormSlot n;
    n.C = C;
    n.gamma = take(sizeof(float) * (C + 64)); n.beta = take(sizeof(float) * (C + 64));
    n.fscale = take(sizeof(float) * (C + 64)); n.fshift = take(sizeof(float) * (C + 64));
    return n;
  };
  L.conv1 = conv_slot(1, 1, 147, S.c0);
  L.norm1 = norm_slot(S.c0);
  int cin = S.c0;
  for (int k = 0; k < 6; ++k) {
    const int c = S.c[k / 2], st = (k % 2 == 0) ? S.s[k / 2] : 1;
    L.bcin[k] = cin; L.bc[k] = c; L.bstride[k] = st;
    L.bc1[k] = conv_slot(3, 3, cin, c);
    L.bc2[k] = conv_slot(3, 3, c, c);
    L.bn1[k] = norm_slot(c);
    L.bn2[k] = norm_slot(c);
    L.has_ds[k] = st != 1;
    if (L.has_ds[k]) { L.bds[k] = conv_slot(1, 1, cin, c); L.bnd[k] = norm_slot(c); }
    cin = c;
  }
  L.conv2 = conv_slot(1, 1, cin, out_dim);
  L.total = off;
  return L;
}

struct EncWs {
  float *X32, *O32, *Y32, *D32;
  __half *Xh, *Xl, *Oh, *Ol, *Fh, *Fl, *Ih, *Il;
  float *part, *mean, *mult;
  size_t total;
};
constexpr int kNormSplit = 64;
inline EncWs enc_ws_layout(void* base, int variant, int N, int H, int W) {
  EncWs E;
  memset(&E, 0, sizeof(E));
  const EncSpec S = enc_spec(variant);
  size_t max32 = 0, max16 = 0;
  for (int l = 0; l < 3; ++l) {
    const int d = 2 << l;
    const size_t np = (size_t)N * ((H + d - 1) / d) * ((W + d - 1) / d);
    const int c = l == 0 ? (S.c0 > S.c[0] ? S.c0 : S.c[0]) : S.c[l];
    if (np * c > max32) max32 = np * c;
    if (np * pad64(c) > max16) max16 = np * pad64(c);
  }
  uint8_t* b8 = reinterpret_cast<uint8_t*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) { uint8_t* p = b8 + off; off = align_up(off + bytes, 1024); return p; };
  E.X32 = (float*)take(max32 * 4); E.O32 = (float*)take(max32 * 4);
  E.Y32 = (float*)take(max32 * 4); E.D32 = (float*)take(max32 * 4);
  E.Xh = (__half*)take(max16 * 2); E.Xl = (__half*)take(max16 * 2);
  E.Oh = (__half*)take(max16 * 2); E.Ol = (__half*)take(max16 * 2);
  E.Fh = (__half*)take(max16 * 2); E.Fl = (__half*)take(max16 * 2);
  {
    const size_t np1 = (size_t)N * ((H + 1) / 2) * ((W + 1) / 2);
    E.Ih = (__half*)take(np1 * 192 * 2); E.Il = (__half*)take(np1 * 192 * 2);
  }
  E.part = (float*)take((size_t)N * kNormSplit * 3 * 256 * 4);
  E.mean = (float*)take((size_t)N * 256 * 4);
  E.mult = (float*)take((size_t)N * 256 * 4);
  E.total = off;
  return E;
}

// ---- prepare ----------------------------------------------------------------------------------
inline int enc_pack_conv(const raft_conv& cv, const EncConvSlot& s, uint8_t* base, cudaStream_t st) {
  if (!cv.kernel || !cv.bias) return RAFT_ERR_BAD_ARG;
  if (cv.kh != s.kh || cv.kw != s.kw || cv.cin != s.cin || cv.cout != s.cout) return RAFT_ERR_BAD_SHAPE;
  const size_t nw = (size_t)s.kh * s.kw * s.cin * s.cout;
  unsigned int* amax = reinterpret_cast<unsigned int*>(base + s.absmax);
  float* scale = reinterpret_cast<float*>(base + s.scale);
  absmax_kernel<<<grid_for(nw), 256, 0, st>>>(cv.kernel, nw, amax);
  weight_scale_kernel<<<1, 1, 0, st>>>(amax, scale);
  PackParams pp;
  memset(&pp, 0, sizeof(pp));
  pp.w = cv.kernel; pp.kh = s.kh; pp.kw = s.kw; pp.cin = s.cin; pp.cout = s.cout;
  pp.hi = reinterpret_cast<__half*>(base + s.hi); pp.lo = reinterpret_cast<__half*>(base + s.lo);
  pp.cout_pad = s.cout_pad; pp.cin_pad = s.cin_pad; pp.cout_off = 0;
  pp.nrange = 1; pp.r_src0[0] = 0; pp.r_n[0] = s.cin; pp.r_dst0[0] = 0;
  pp.scale = scale;
  pack_weights_kernel<<<grid_for(nw), 256, 0, st>>>(pp);
  g_launches += 3;
  RAFT_CUDA_TRY(cudaMemcpyAsync(base + s.bias, cv.bias, s.cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return raft_launch_status();
}

inline int enc_pack_norm(const raft_norm& nm, const EncNormSlot& s, int norm_type, uint8_t* base, cudaStream_t st) {
  if (norm_type == NORM_NONE) return 0;
  if (!nm.gamma || !nm.beta) return RAFT_ERR_BAD_ARG;
  float* g = reinterpret_cast<float*>(base + s.gamma);
  float* b = reinterpret_cast<float*>(base + s.beta);
  RAFT_CUDA_TRY(cudaMemcpyAsync(g, nm.gamma, s.C * sizeof(float), cudaMemcpyDeviceToDevice, st));
  RAFT_CUDA_TRY(cudaMemcpyAsync(b, nm.beta, s.C * sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (norm_type == NORM_BATCH) {
    if (!nm.moving_mean || !nm.moving_variance) return RAFT_ERR_BAD_ARG;
    bn_fold_kernel<<<ceil_div(s.C, 128), 128, 0, st>>>(nm.gamma, nm.beta, nm.moving_mean, nm.moving_variance, 1e-3f, s.C,
                                                       reinterpret_cast<float*>(base + s.fscale),
                                                       reinterpret_cast<float*>(base + s.fshift));
    ++g_launches;
  }
  return raft_launch_status();
}

inline int encoder_prepare(int variant, int norm_type, int out_dim, const raft_encoder_weights* w, void* prepared,
                           size_t bytes, cudaStream_t st) {
  const EncLayout L = enc_layout(variant, out_dim);
  if (L.total > bytes) return RAFT_ERR_WORKSPACE;
  const EncSpec S = enc_spec(variant);
  uint8_t* base = reinterpret_cast<uint8_t*>(prepared);
  RAFT_CUDA_TRY(cudaMemsetAsync(base, 0, L.total, st));
  if (!w->conv1.kernel || !w->conv1.bias) return RAFT_ERR_BAD_ARG;
  if (w->conv1.kh != 7 || w->conv1.kw != 7 || w->conv1.cin != 3 || w->conv1.cout != S.c0) return RAFT_ERR_BAD_SHAPE;
  {
    raft_conv flat = w->conv1;            // HWIO (7,7,3,c0) is already [tap*3 + c][cout]: view it as 1x1 over 147
    flat.kh = 1; flat.kw = 1; flat.cin = 147;
    RAFT_TRY(enc_pack_conv(flat, L.conv1, base, st));
  }
  RAFT_TRY(enc_pack_norm(w->norm1, L.norm1, norm_type, base, st));
  for (int k = 0; k < 6; ++k) {
    RAFT_TRY(enc_pack_conv(w->block[k].conv1, L.bc1[k], base, st));
    RAFT_TRY(enc_pack_conv(w->block[k].conv2, L.bc2[k], base, st));
    RAFT_TRY(enc_pack_norm(w->block[k].norm1, L.bn1[k], norm_type, base, st));
    RAFT_TRY(enc_pack_norm(w->block[k].norm2, L.bn2[k], norm_type, base, st));
    if (L.has_ds[k]) {
      RAFT_TRY(enc_pack_conv(w->block[k].downsample, L.bds[k], base, st));
      RAFT_TRY(enc_pack_norm(w->block[k].downsample_norm, L.bnd[k], norm_type, base, st));
    }
  }
  RAFT_TRY(enc_pack_conv(w->conv2, L.conv2, base, st));
  return raft_launch_status();
}

// ---- forward ----------------------------------------------------------------------------------
struct EncCtx {
  const uint8_t* prep; EncLayout L; EncWs W; cudaStream_t st;
  int N, norm_type, stats;    // stats: 1 = statistics from the data (instance, or batch in training)
  int per_image;              // instance: one group per image; batch-training: one group
};

// y (npix, C) raw conv output -> normalised, activated, (+skip), re-split.  (Statistics partials from the convolution
// epilogue and operand-swapped narrow layers were built and measured in round 2 -- both slower than this form
// (profiles/README.md) -- and removed.)
inline int enc_norm_apply(const EncCtx& c, const EncNormSlot& ns, const float* y, size_t npix, int P, int relu,
                          const float* skip32, const __half* skip_hi, const __half* skip_lo, float* out32, __half* hi,
                          __half* lo) {
  const int C = ns.C, G = c.per_image ? c.N : 1;
  const int Pg = c.per_image ? P : (int)npix;
  const float* gamma = reinterpret_cast<const float*>(c.prep + ns.gamma);
  const float* beta = reinterpret_cast<const float*>(c.prep + ns.beta);
  // (Finalisation inside norm_stats_kernel by the last block of a group was measured twice -- +33 us per launch: the merge
  //  of C channels by one block is serial where norm_final_kernel spreads it over G*C warps; profiles/README.md.)
  norm_stats_kernel<<<dim3((unsigned)G, kNormSplit), kNormStatsThreads, 0, c.st>>>(y, Pg, C, kNormSplit, c.W.part);
  norm_final_kernel<<<ceil_div(G * C * 32, 256), 256, 0, c.st>>>(c.W.part, G, C, kNormSplit, gamma, 1e-3f, c.W.mean, c.W.mult);
  norm_apply_kernel<<<grid_for(npix * (pad64(C) / 8)), 256, 0, c.st>>>(y, npix, P, C, c.per_image, c.W.mean, c.W.mult, beta, relu,
                                                                 skip32, skip_hi, skip_lo, out32, hi, lo, pad64(C));
  g_launches += 3;
  return raft_launch_status();
}

// One tensor-core convolution of the encoder.  When the norm needs data statistics the raw output goes to
// `raw32` (bias only); otherwise the folded affine, activation and skip are applied in the epilogue.
inline int enc_conv_tc(const EncCtx& c, const EncConvSlot& cs, const EncNormSlot* ns, const __half* ahi, const __half* alo,
                       int Hin, int Win, int Hout, int Wout, int stride, int relu, const float* skip, float* out32,
                       __half* ohi, __half* olo) {
  TcConvParams p;
  memset(&p, 0, sizeof(p));
  int tw, th;
  tc_pick_tile(Wout, Hout, &tw, &th);
  if (tw * stride > 256) tw = 128 / stride, th = 128 / tw;
  // Wide 3x3 stride-1 layers with few output channels (layer1 / layer2 of both encoders at >= 128 feature columns): one
  // activation box and one weight box per kernel ROW (conv_tc.cuh kRow3).  RAFT_B200_ROW3=0 disables (A/B timing).
  static const int row3_flag = [] { const char* e = getenv("RAFT_B200_ROW3"); return e ? atoi(e) : 1; }();
  const bool row3 = row3_flag && cs.kh == 3 && cs.kw == 3 && stride == 1 && tw == kTileM && th == 1 && cs.cout_pad <= 96 &&
                    cs.cout_pad % 8 == 0;
  if (row3) {
    RAFT_TRY(make_tmap_act2(&p.a_map[0], ahi, alo, c.N, Hin, Win, cs.cin_pad, kARow3Pixels, 1, 1));
    RAFT_TRY(make_tmap_wgt3(&p.b_map, reinterpret_cast<const __half*>(c.prep + cs.hi),
                            reinterpret_cast<const __half*>(c.prep + cs.lo), cs.kh * cs.kw, cs.cout_pad, cs.cin_pad, cs.cout_pad));
    p.row3 = 1;
    // (Keeping the nine taps of the 64-channel layers resident in shared memory was measured in round 2: slower, 489 vs 496
    // pairs/s -- it leaves 68 KB of activation stages in flight against an HBM latency of ~3.1 k cycles.)
  } else {
    RAFT_TRY(make_tmap_act2(&p.a_map[0], ahi, alo, c.N, Hin, Win, cs.cin_pad, tw, th, stride));
    RAFT_TRY(make_tmap_wgt2(&p.b_map, reinterpret_cast<const __half*>(c.prep + cs.hi),
                            reinterpret_cast<const __half*>(c.prep + cs.lo), cs.kh * cs.kw, cs.cout_pad, cs.cin_pad,
                            cs.cout_pad));
  }
  p.nseg = 1; p.seg_chunks[0] = cs.cin_pad / kChunkK; p.seg_c0[0] = 0;
  p.kh = cs.kh; p.kw = cs.kw; p.stride = stride;
  // Keras 'same': stride 1 -> (k-1)/2 before; stride 2 on even input -> total k-2, before = (k-2)/2 (0 for 3x3);
  // 1x1 convs are 'valid' (no padding).
  if (stride == 1) { p.ph = (cs.kh - 1) / 2; p.pw = (cs.kw - 1) / 2; }
  else {
    const int tot_h = (Hout - 1) * stride + cs.kh - Hin, tot_w = (Wout - 1) * stride + cs.kw - Win;
    p.ph = (tot_h > 0 ? tot_h : 0) / 2; p.pw = (tot_w > 0 ? tot_w : 0) / 2;
  }
  p.B = c.N; p.H = Hout; p.W = Wout; p.TH = th; p.TW = tw;
  p.bn = cs.cout_pad; p.n_total = cs.cout;
  p.mode = EPI_LINEAR; p.out_scale = 1.0f;
  p.bias = reinterpret_cast<const float*>(c.prep + cs.bias);
  p.inv_scale = reinterpret_cast<const float*>(c.prep + cs.scale) + 1;
  p.out_f32 = out32; p.f32_stride = cs.cout; p.f32_c0 = 0;
  p.out_hi = ohi; p.out_lo = olo; p.h_stride = pad64(cs.cout); p.h_c0 = 0;
  if (ns && !c.stats && c.norm_type == NORM_BATCH) {
    p.post_scale = reinterpret_cast<const float*>(c.prep + ns->fscale);
    p.post_shift = reinterpret_cast<const float*>(c.prep + ns->fshift);
  }
  const bool fused = !(ns && c.stats);
  if (fused) {
    p.act = relu ? ACT_RELU : ACT_NONE;
    p.residual = skip; p.res_stride = cs.cout; p.res_c0 = 0;
  } else {
    p.act = ACT_NONE; p.out_hi = nullptr; p.out_lo = nullptr;
  }
  // (An L2 tensor prefetch of the next tile's activation boxes was measured in round 2: no effect, 494 vs 496 pairs/s -- the
  //  ~3 k-cycle load latency of these layers is TMA service time, not HBM latency; profiles/README.md.)
  if (g_dbg_layer >= 1000 && g_dbg_count++ == g_dbg_layer - 1000) p.dbg = g_dbg_buf;   // timeline of the k-th encoder conv
  {
    // Promotion group of the encoder convolutions: their contractions are short (K <= 1152, 18 chunks), so the fp32
    // accumulator may stay in TMEM for 5 chunks (60 MMA steps) between IEEE promotions instead of the update block's 2
    // (its K = 1920 GRU contractions feed a 12-iteration recurrence).  Measured: 433 -> 447 pairs/s, parity tests green.
    static const int grp = [] { const char* e = getenv("RAFT_B200_ENC_GROUP"); return e ? atoi(e) : 5; }();
    if (grp > 0) p.group_chunks = grp;
    if (row3) p.group_chunks = 2;       // a kRow3 stage carries three taps: 2 stages = 72 MMA steps per accumulation chain
  }
  ++g_launches;
  return tc_launch(p, 1, c.st);
}

// (Processing a large batch in groups of 2 or 4 images, so that a group's raw convolution output stays in L2 between the
// convolution, the statistics pass and the normalise pass, was measured in round 2: 408 / 456 vs 482 pairs/s -- the
// smaller launches cost more than the L2 hits save -- and removed.)
inline int encoder_forward(int variant, int norm_type, int out_dim, const void* prepared, const float* images, int N,
                           int H, int W, int training, int image_norm, float* out, void* ws, size_t ws_bytes, cudaStream_t st) {
  EncCtx c;
  c.prep = reinterpret_cast<const uint8_t*>(prepared);
  c.L = enc_layout(variant, out_dim);
  c.W = enc_ws_layout(ws, variant, N, H, W);
  if (c.W.total > ws_bytes) return RAFT_ERR_WORKSPACE;
  c.st = st; c.N = N; c.norm_type = norm_type;
  c.stats = (norm_type == NORM_INSTANCE) || (norm_type == NORM_BATCH && training);
  c.per_image = norm_type == NORM_INSTANCE;
  const EncSpec S = enc_spec(variant);
  const EncLayout& L = c.L;
  const EncWs& E = c.W;

  // ---- stem: conv1 7x7 s2 + norm1 + relu (extractor.py:120) ----
  // K = 7*7*3 = 147: gather the (normalised) input window of every output pixel into 192-channel fp16 planes
  // and run the stem as a 1x1 tensor-core convolution.
  int h = (H + 1) / 2, w = (W + 1) / 2;
  {
    const size_t npix = (size_t)N * h * w;
    const int tot_h = (h - 1) * 2 + 7 - H, tot_w = (w - 1) * 2 + 7 - W;
    stem_gather_kernel<<<dim3(ceil_div(w, kStemSeg), h, N), 256, 0, st>>>(images, H, W, h, w, (tot_h > 0 ? tot_h : 0) / 2,
                                                                          (tot_w > 0 ? tot_w : 0) / 2, image_norm, E.Ih, E.Il);
    ++g_launches;
    if (!c.stats && pad64(S.c0) != S.c0) {
      RAFT_CUDA_TRY(cudaMemsetAsync(E.Xh, 0, npix * pad64(S.c0) * 2, st));
      RAFT_CUDA_TRY(cudaMemsetAsync(E.Xl, 0, npix * pad64(S.c0) * 2, st));
    }
    RAFT_TRY(enc_conv_tc(c, L.conv1, &L.norm1, E.Ih, E.Il, h, w, h, w, 1, 1, nullptr, c.stats ? E.Y32 : E.X32, E.Xh, E.Xl));
    if (c.stats) RAFT_TRY(enc_norm_apply(c, L.norm1, E.Y32, npix, h * w, 1, nullptr, nullptr, nullptr, nullptr, E.Xh, E.Xl));
  }

  float *X32 = E.X32, *O32 = E.O32;
  __half *Xh = E.Xh, *Xl = E.Xl, *Oh = E.Oh, *Ol = E.Ol;
  for (int k = 0; k < 6; ++k) {
    const int st2 = L.bstride[k], cin = L.bcin[k], cc = L.bc[k];
    const int ho = (h + st2 - 1) / st2, wo = (w + st2 - 1) / st2;
    const size_t npo = (size_t)N * ho * wo;
    (void)cin;
    const bool zero_pad_out = pad64(cc) != cc;     // fused epilogues write 32-column chunks: clear the 64-pad tail
    // conv1 + norm1 + relu -> F
    if (!c.stats && zero_pad_out) {
      RAFT_CUDA_TRY(cudaMemsetAsync(E.Fh, 0, npo * pad64(cc) * 2, st));
      RAFT_CUDA_TRY(cudaMemsetAsync(E.Fl, 0, npo * pad64(cc) * 2, st));
      RAFT_CUDA_TRY(cudaMemsetAsync(Oh, 0, npo * pad64(cc) * 2, st));
      RAFT_CUDA_TRY(cudaMemsetAsync(Ol, 0, npo * pad64(cc) * 2, st));
    }
    RAFT_TRY(enc_conv_tc(c, L.bc1[k], &L.bn1[k], Xh, Xl, h, w, ho, wo, st2, 1, nullptr, c.stats ? E.Y32 : nullptr, E.Fh, E.Fl));
    if (c.stats) RAFT_TRY(enc_norm_apply(c, L.bn1[k], E.Y32, npo, ho * wo, 1, nullptr, nullptr, nullptr, nullptr, E.Fh, E.Fl));
    // skip branch
    const float* skip = X32;
    if (L.has_ds[k]) {
      RAFT_TRY(enc_conv_tc(c, L.bds[k], &L.bnd[k], Xh, Xl, h, w, ho, wo, st2, 0, nullptr, c.stats ? E.Y32 : E.D32, nullptr, nullptr));
      if (c.stats) RAFT_TRY(enc_norm_apply(c, L.bnd[k], E.Y32, npo, ho * wo, 0, nullptr, nullptr, nullptr, E.D32, nullptr, nullptr));
      skip = E.D32;
    }
    // conv2 + norm2 + relu, then relu(skip + fx) -> O
    RAFT_TRY(enc_conv_tc(c, L.bc2[k], &L.bn2[k], E.Fh, E.Fl, ho, wo, ho, wo, 1, 1, skip, c.stats ? E.Y32 : O32, Oh, Ol));
    if (c.stats) {   // skip = block input: from D32 after a downsample, else from the block's own fp16 operand planes
      if (L.has_ds[k]) RAFT_TRY(enc_norm_apply(c, L.bn2[k], E.Y32, npo, ho * wo, 1, E.D32, nullptr, nullptr, nullptr, Oh, Ol));
      else RAFT_TRY(enc_norm_apply(c, L.bn2[k], E.Y32, npo, ho * wo, 1, nullptr, Xh, Xl, nullptr, Oh, Ol));
    }
    // next block reads O
    float* t32 = X32; X32 = O32; O32 = t32;
    __half* th_ = Xh; Xh = Oh; Oh = th_;
    __half* tl_ = Xl; Xl = Ol; Ol = tl_;
    h = ho; w = wo;
  }
  // conv2 1x1 -> (N, H/8, W/8, out_dim), bias only (extractor.py:125)
  RAFT_TRY(enc_conv_tc(c, L.conv2, nullptr, Xh, Xl, h, w, h, w, 1, 0, nullptr, out, nullptr, nullptr));
  return raft_launch_status();
}

}  // namespace raft
