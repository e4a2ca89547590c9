// extern "C" entry points of libraft_b200.so (see include/raft_b200.h for the contract and the
// reference file:line each one replaces).  Host code only decides shapes and launches kernels;
// there is no CPU compute path.
#include <algorithm>

#include "corr_tc.cuh"
#include "encoder.cuh"
#include "train.cuh"

namespace raft {
thread_local long long g_launches = 0;
int g_dbg_layer = -1;
long long* g_dbg_buf = nullptr;
int g_dbg_count = 0;               // encoder convolutions launched since the timeline was armed (tc_layer >= 1000)

static int check_dims(int B, int h, int w) { return (B > 0 && h > 0 && w > 0) ? 0 : RAFT_ERR_BAD_SHAPE; }

// Per-kernel timing of raft_b200_forward_loop for bench.py's roofline objects: CUDA events on the launching stream around
// the lookup and around the update-block kernel(s) of every iteration (raft_b200_profile_loop / _read).  Off by default;
// never armed while a CUDA graph is being captured.
struct LoopProfile {
  bool on = false;
  int n = 0;                                   // iterations recorded by the last forward_loop call
  cudaEvent_t ev[64][3];                       // [iteration]: before lookup, after lookup (+ im2col), after the update block
  bool created = false;
};
static LoopProfile g_prof;

// ------------------------------------------------------------------------------------------------
// Correlation pyramid
// ------------------------------------------------------------------------------------------------
struct CorrWs {
  float* f2_lvl[RAFT_MAX_LEVELS];            // pooled fmap2 per level (level 0 = fmap2 itself, not stored)
  __half *f1_hi, *f1_lo;
  __half *f2_hi[RAFT_MAX_LEVELS], *f2_lo[RAFT_MAX_LEVELS];
  size_t total;
};
static CorrWs corr_ws_layout(void* base, int B, int h, int w, int C, int levels, int precision) {
  CorrWs W;
  memset(&W, 0, sizeof(W));
  if (precision != RAFT_PREC_F16X2) return W;
  uint8_t* b8 = reinterpret_cast<uint8_t*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) {
    uint8_t* p = b8 + off;
    off = align_up(off + bytes, 1024);
    return p;
  };
  W.f1_hi = reinterpret_cast<__half*>(take((size_t)B * h * w * C * 2));
  W.f1_lo = reinterpret_cast<__half*>(take((size_t)B * h * w * C * 2));
  int lh = h, lw = w;
  for (int l = 0; l < levels; ++l) {
    if (l > 0) W.f2_lvl[l] = reinterpret_cast<float*>(take((size_t)B * lh * lw * C * 4));
    W.f2_hi[l] = reinterpret_cast<__half*>(take((size_t)B * lh * lw * C * 2));
    W.f2_lo[l] = reinterpret_cast<__half*>(take((size_t)B * lh * lw * C * 2));
    lh /= 2;
    lw /= 2;
  }
  W.total = off;
  return W;
}

static int corr_build_fp32(const float* f1, const float* f2, int B, int h, int w, int C, int levels, float* const pyr[],
                           cudaStream_t st) {
  const int N = h * w;
  dim3 grid((unsigned)ceil_div(N, 64), (unsigned)ceil_div(N, 64), (unsigned)B);
  corr_fp32_kernel<<<grid, 256, 0, st>>>(f1, f2, pyr[0], N, C, sqrtf((float)C));
  RAFT_COUNT_LAUNCH();
  RAFT_TRY(raft_launch_status());
  int lh = h, lw = w;
  for (int l = 1; l < levels; ++l) {        // corr.py:112-114: pool the volume itself
    const size_t M = (size_t)B * N;
    const size_t total = M * (lh / 2) * (lw / 2);
    avgpool2x2_kernel<<<grid_for(total), 256, 0, st>>>(pyr[l - 1], pyr[l], M, lh, lw, 1);
    RAFT_COUNT_LAUNCH();
    RAFT_TRY(raft_launch_status());
    lh /= 2;
    lw /= 2;
  }
  return 0;
}

// Tensor-core path: level l = fmap1 . avgpool^l(fmap2)^T / sqrt(C).  Pooling is linear, so pooling
// the 256-channel features (a few MB) before the GEMM equals pooling the N x N volume after it
// (up to fp32 summation order) and every level is written exactly once, straight from TMEM.
// Two launches: corr_prep_kernel (pool + hi/lo split of both feature maps) and corr_tc_kernel (all levels).
static int corr_build_tc(const float* f1, const float* f2, int B, int h, int w, int C, int levels, float* const pyr[],
                         void* ws, cudaStream_t st) {
  if (C % kChunkK != 0) return RAFT_ERR_BAD_SHAPE;
  CorrWs W = corr_ws_layout(ws, B, h, w, C, levels, RAFT_PREC_F16X2);
  const int N = h * w;
  const size_t npix = (size_t)B * N;
  if (levels <= 4) {
    CorrPrepParams q;
    memset(&q, 0, sizeof(q));
    q.f1 = f1; q.f2 = f2; q.f1_hi = W.f1_hi; q.f1_lo = W.f1_lo;
    for (int l = 0; l < levels; ++l) { q.f2_hi[l] = W.f2_hi[l]; q.f2_lo[l] = W.f2_lo[l]; }
    q.B = B; q.h = h; q.w = w; q.C = C; q.levels = levels;
    q.patches_x = ceil_div(w, 8); q.patches_y = ceil_div(h, 8);
    q.npatch = B * q.patches_x * q.patches_y;
    const int split_blocks = (int)std::min<size_t>((npix * C / 4 + 127) / 128, (size_t)kNumSMs * 8);
    corr_prep_kernel<<<q.npatch + split_blocks, 128, 0, st>>>(q);
    RAFT_COUNT_LAUNCH();
  } else {                                   // deeper pyramids: generic pooling / split kernels, level by level
    split_plane_kernel<<<grid_for(npix * C), 256, 0, st>>>(f1, C, 0, C, C, W.f1_hi, W.f1_lo, C, 0, npix, 1.0f);
    RAFT_COUNT_LAUNCH();
    int lh = h, lw = w;
    const float* src = f2;
    for (int l = 0; l < levels; ++l) {
      if (l > 0) {
        const size_t total = (size_t)B * (lh / 2) * (lw / 2) * C;
        avgpool2x2_kernel<<<grid_for(total), 256, 0, st>>>(src, W.f2_lvl[l], (size_t)B, lh, lw, C);
        RAFT_COUNT_LAUNCH();
        src = W.f2_lvl[l];
        lh /= 2;
        lw /= 2;
      }
      const size_t np2 = (size_t)B * lh * lw;
      split_plane_kernel<<<grid_for(np2 * C), 256, 0, st>>>(src, C, 0, C, C, W.f2_hi[l], W.f2_lo[l], C, 0, np2, 1.0f);
      RAFT_COUNT_LAUNCH();
    }
  }
  RAFT_TRY(raft_launch_status());

  CorrTcParams p;
  memset(&p, 0, sizeof(p));
  // A: fmap1 as a (B, 1, N, C) "image" -> 128 consecutive queries per tile
  RAFT_TRY(make_tmap_act2(&p.a_map, W.f1_hi, W.f1_lo, B, 1, N, C, 128, 1));
  p.levels = levels; p.B = B; p.N = N; p.chunks = C / kChunkK;
  p.mtiles_img = ceil_div(N, kTileM);
  const int mtiles = B * p.mtiles_img;
  int lh = h, lw = w;
  for (int l = 0; l < levels; ++l) {
    const int N2 = lh * lw;
    const int ntn = ceil_div(N2, kCorrBn);
    const int bn = round_up(ceil_div(N2, ntn), 16);
    // B: level-l features [B][N2][C] -> the batch index rides in the "tap" coordinate
    RAFT_TRY(make_tmap_wgt2(&p.b_map[l], W.f2_hi[l], W.f2_lo[l], B, N2, C, bn));
    p.out[l] = pyr[l];
    p.n2[l] = N2; p.bn[l] = bn;
    p.tile0[l + 1] = p.tile0[l] + mtiles * ntn;
    lh /= 2;
    lw /= 2;
  }
  p.corr_div = sqrtf((float)C);
  {
    int e = 0;
    const float m = frexpf(p.corr_div, &e);          // sqrt(C) = m * 2^e; m == 0.5 <=> exact power of two
    p.corr_mul = (m == 0.5f && p.corr_div * p.corr_div == (float)C) ? 1.0f / p.corr_div : 0.0f;
  }
  if (g_dbg_layer == 2000) p.dbg = g_dbg_buf;
  int dev = 0;
  RAFT_CUDA_TRY(cudaGetDevice(&dev));
  static unsigned long long attr_mask = 0;          // per-device attribute (benign race: idempotent)
  if (!(attr_mask & (1ull << (dev & 63)))) {
    RAFT_CUDA_TRY(cudaFuncSetAttribute(corr_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCorrSmemBytes));
    attr_mask |= 1ull << (dev & 63);
  }
  const int ntiles = p.tile0[levels];
  corr_tc_kernel<<<ntiles < kNumSMs ? ntiles : kNumSMs, kCorrThreads, kCorrSmemBytes, st>>>(p);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

// ------------------------------------------------------------------------------------------------
// Update block, fp32 FFMA path: the reference's op sequence, one launch per Conv2D.
// ------------------------------------------------------------------------------------------------
static int gru_fp32(const UpdateCtx& c, float* h, int iz, int ir, int iq, int hid, int xs, int xn) {
  const Workspace& W = c.W;
  const size_t n = (size_t)c.B * c.h * c.w * hid;
  RAFT_TRY(simt2(c, iz, h, hid, hid, W.x, xs, xn, W.z, hid, SACT_SIGMOID));
  RAFT_TRY(simt2(c, ir, h, hid, hid, W.x, xs, xn, W.r, hid, SACT_SIGMOID));
  gru_rh_kernel<<<grid_for(n), 256, 0, c.stream>>>(W.r, h, W.rh, n);
  RAFT_COUNT_LAUNCH();
  RAFT_TRY(simt2(c, iq, W.rh, hid, hid, W.x, xs, xn, W.q, hid, SACT_TANH));
  gru_update_kernel<<<grid_for(n), 256, 0, c.stream>>>(W.z, W.q, h, n);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

static int update_core_fp32(const UpdateCtx& c, float* h, float* delta, float* mask) {
  const Workspace& W = c.W;
  const VariantDims d = variant_dims(c.variant);
  const size_t npix = (size_t)c.B * c.h * c.w;
  if (c.variant == RAFT_VARIANT_BASIC) {
    RAFT_TRY(simt1(c, BC1, W.corr, 324, 0, 324, W.cor1, 256, 0, SACT_RELU));           // update.py:98
    RAFT_TRY(simt1(c, BC2, W.cor1, 256, 0, 256, W.cf, 256, 0, SACT_RELU));              // :99
    RAFT_TRY(simt1(c, BF1, W.flow, 2, 0, 2, W.flo1, 128, 0, SACT_RELU));                // :100
    RAFT_TRY(simt1(c, BF2, W.flo1, 128, 0, 128, W.cf, 256, 192, SACT_RELU));            // :101,104
    RAFT_TRY(simt1(c, BCV, W.cf, 256, 0, 256, W.x, 256, 128, SACT_RELU));               // :105
    copy_channels_kernel<<<grid_for(npix * 2), 256, 0, c.stream>>>(W.flow, 2, 0, W.x, 256, 254, 2, npix);   // :106
    RAFT_COUNT_LAUNCH();
    RAFT_TRY(gru_fp32(c, h, BZ1, BR1, BQ1, 128, 256, 256));                             // :53-58
    RAFT_TRY(gru_fp32(c, h, BZ2, BR2, BQ2, 128, 256, 256));                             // :60-65
    RAFT_TRY(simt1(c, BFH1, h, 128, 0, 128, W.fm, 512, 0, SACT_RELU));                  // :14
    RAFT_TRY(simt1(c, BFH2, W.fm, 512, 0, 256, delta, 2, 0, SACT_NONE));
    if (mask) {
      RAFT_TRY(simt1(c, BM0, h, 128, 0, 128, W.fm, 512, 256, SACT_RELU));               // :137-141
      RAFT_TRY(simt1(c, BM2, W.fm, 512, 256, 256, mask, 576, 0, SACT_NONE, 0.25f));     // :152
    }
  } else {
    RAFT_TRY(simt1(c, SC1, W.corr, 196, 0, 196, W.cf, 128, 0, SACT_RELU));              // update.py:80
    RAFT_TRY(simt1(c, SF1, W.flow, 2, 0, 2, W.flo1, 64, 0, SACT_RELU));                 // :81
    RAFT_TRY(simt1(c, SF2, W.flo1, 64, 0, 64, W.cf, 128, 96, SACT_RELU));               // :82-83
    RAFT_TRY(simt1(c, SCV, W.cf, 128, 0, 128, W.x, d.c_x, 64, SACT_RELU));              // :84
    copy_channels_kernel<<<grid_for(npix * 2), 256, 0, c.stream>>>(W.flow, 2, 0, W.x, d.c_x, 144, 2, npix);  // :85
    RAFT_COUNT_LAUNCH();
    RAFT_TRY(gru_fp32(c, h, SZ, SR, SQ, 96, d.c_x, 146));                               // :26-35
    RAFT_TRY(simt1(c, SFH1, h, 96, 0, 96, W.fm, 128, 0, SACT_RELU));
    RAFT_TRY(simt1(c, SFH2, W.fm, 128, 0, 128, delta, 2, 0, SACT_NONE));
  }
  return raft_launch_status();
}

// ------------------------------------------------------------------------------------------------
// Update block, tensor-core path.  Operands travel between layers as fp16 hi/lo planes written by
// the producing layer's epilogue; z||r and flow_head.conv1||mask[0] are single GEMMs.
// ------------------------------------------------------------------------------------------------
static void tc_params_init(TcConvParams& p, int mode, int act, int n_total) {
  memset(&p, 0, sizeof(p));
  p.mode = mode;
  p.act = act;
  p.n_total = n_total;
  p.out_scale = 1.0f;
}

static TcDeps dep1(int layer, int ntile = -1) { return TcDeps{1, {layer, -1}, {ntile, -1}}; }
static TcDeps dep2(int l0, int l1) { return TcDeps{2, {l0, l1}, {-1, -1}}; }

static int gru_tc(const UpdateCtx& c, float* h, int lzr, int lq, int hid, int x_chunks, int src_layer) {
  const Workspace& W = c.W;
  const VariantDims d = variant_dims(c.variant);
  TcConvParams p;
  {
    tc_params_init(p, EPI_GRU_ZR, ACT_NONE, 2 * hid);
    p.z = W.z; p.h = h; p.hid = hid;
    p.out_hi = W.rh_hi; p.out_lo = W.rh_lo; p.h_stride = d.s_h; p.h_c0 = 0;
    TcSeg segs[2] = {{W.h_hi, W.h_lo, d.s_h, 0, d.s_h / kChunkK}, {W.x_hi, W.x_lo, d.s_x, 0, x_chunks}};
    RAFT_TRY(launch_tc_layer(c, lzr, 2, segs, p, -1, dep1(src_layer)));
  }
  {
    tc_params_init(p, EPI_GRU_Q, ACT_NONE, hid);
    p.z = W.z; p.h = h; p.hid = hid;
    p.out_hi = W.h_hi; p.out_lo = W.h_lo; p.h_stride = d.s_h; p.h_c0 = 0;
    TcSeg segs[2] = {{W.rh_hi, W.rh_lo, d.s_h, 0, d.s_h / kChunkK}, {W.x_hi, W.x_lo, d.s_x, 0, x_chunks}};
    RAFT_TRY(launch_tc_layer(c, lq, 2, segs, p, -1, dep1(lzr)));
  }
  return 0;
}

// Flow branch of BasicMotionEncoder (update.py:98-99): convf1 7x7 2->128 + relu, convf2 3x3 128->64 + relu ->
// cor_flo[192:256).  Depends only on the current flow, so it may run beside the lookup and the correlation branch.
// (two parts, so that the work list of update_mega_kernel can interleave them with the correlation branch: the list order is
//  the order in which free CTAs claim items)
static int flow_branch_basic_tc(const UpdateCtx& c, int part) {
  const Workspace& W = c.W;
  const VariantDims d = variant_dims(c.variant);
  TcConvParams p;
  if (part == 0) {  // convf1 7x7 2->128 + relu: K = 98 -> gather the window into 128-channel planes, run as a 1x1 GEMM
    const size_t npix = (size_t)c.B * c.h * c.w;
    if (!c.fim_ready) {              // (the iteration loop's lookup kernel has already produced the planes)
      flow_im2col_kernel<<<grid_for(npix * 128), 256, 0, c.stream>>>(W.flow, c.B, c.h, c.w, W.fim_hi, W.fim_lo);
      RAFT_COUNT_LAUNCH();
    }
    tc_params_init(p, EPI_LINEAR, ACT_RELU, 128);
    p.out_hi = W.flo1_hi; p.out_lo = W.flo1_lo; p.h_stride = d.s_flo1;
    TcSeg s[1] = {{W.fim_hi, W.fim_lo, 128, 0, 2}};
    RAFT_TRY(launch_tc_layer(c, 11, 1, s, p));
  } else {  // convf2 3x3 128->64 + relu -> cor_flo[192:256)
    tc_params_init(p, EPI_LINEAR, ACT_RELU, 64);
    p.out_hi = W.cf_hi; p.out_lo = W.cf_lo; p.h_stride = d.s_cf; p.h_c0 = 192;
    TcSeg s[1] = {{W.flo1_hi, W.flo1_lo, d.s_flo1, 0, 2}};
    RAFT_TRY(launch_tc_layer(c, 2, 1, s, p, -1, dep1(11)));
  }
  return 0;
}

// adv_coords != null (iteration loop): the flow-head epilogue also applies coords1 += delta and flow = coords1 - grid.
static int update_core_tc(const UpdateCtx& c, float* h, float* delta, float* mask, float* adv_coords = nullptr) {
  const Workspace& W = c.W;
  const VariantDims d = variant_dims(c.variant);
  TcConvParams p;
  if (c.variant == RAFT_VARIANT_BASIC) {
    {  // convc1 1x1 324->256 + relu
      tc_params_init(p, EPI_LINEAR, ACT_RELU, 256);
      p.out_hi = W.cor1_hi; p.out_lo = W.cor1_lo; p.h_stride = d.s_cor1;
      TcSeg s[1] = {{W.corr_hi, W.corr_lo, d.s_corr, 0, d.s_corr / kChunkK}};
      RAFT_TRY(launch_tc_layer(c, 0, 1, s, p));
    }
    RAFT_TRY(flow_branch_basic_tc(c, 0));                   // convf1 (update.py:98)
    {  // convc2 3x3 256->192 + relu -> cor_flo[0:192)
      tc_params_init(p, EPI_LINEAR, ACT_RELU, 192);
      p.out_hi = W.cf_hi; p.out_lo = W.cf_lo; p.h_stride = d.s_cf;
      TcSeg s[1] = {{W.cor1_hi, W.cor1_lo, d.s_cor1, 0, 4}};
      RAFT_TRY(launch_tc_layer(c, 1, 1, s, p, -1, dep1(0)));
    }
    RAFT_TRY(flow_branch_basic_tc(c, 1));                   // convf2 (update.py:99)
    {  // conv 3x3 256->126 + relu, concat flow -> x[128:256)
      tc_params_init(p, EPI_LINEAR, ACT_RELU, 126);
      p.out_hi = W.x_hi; p.out_lo = W.x_lo; p.h_stride = d.s_x; p.h_c0 = 128;
      p.concat_src = W.flow; p.concat_n = 2;
      TcSeg s[1] = {{W.cf_hi, W.cf_lo, d.s_cf, 0, 4}};
      RAFT_TRY(launch_tc_layer(c, 3, 1, s, p, -1, dep2(1, 2)));
    }
    RAFT_TRY(gru_tc(c, h, 4, 5, 128, 4, 3));
    RAFT_TRY(gru_tc(c, h, 6, 7, 128, 4, 5));
    {  // flow_head.conv1 || mask[0], 3x3 128->512 + relu
      tc_params_init(p, EPI_LINEAR, ACT_RELU, mask ? 512 : 256);
      p.out_hi = W.fm_hi; p.out_lo = W.fm_lo; p.h_stride = d.s_fm;
      TcSeg s[1] = {{W.h_hi, W.h_lo, d.s_h, 0, 2}};
      RAFT_TRY(launch_tc_layer(c, 8, 1, s, p, mask ? 2 : 1, dep1(7)));
    }
    {  // flow_head.conv2 3x3 256->2
      tc_params_init(p, EPI_LINEAR, ACT_NONE, 2);
      p.out_f32 = delta; p.f32_stride = 2;
      p.adv_coords = adv_coords; p.adv_flow = adv_coords ? W.flow : nullptr;
      TcSeg s[1] = {{W.fm_hi, W.fm_lo, d.s_fm, 0, 4}};
      RAFT_TRY(launch_tc_layer(c, 9, 1, s, p, -1, dep1(8, 0)));
    }
    if (mask) {  // mask[2] 1x1 256->576, x0.25
      tc_params_init(p, EPI_LINEAR, ACT_NONE, 576);
      p.out_f32 = mask; p.f32_stride = 576; p.out_scale = 0.25f;
      TcSeg s[1] = {{W.fm_hi, W.fm_lo, d.s_fm, 256, 4}};
      RAFT_TRY(launch_tc_layer(c, 10, 1, s, p, -1, dep1(8, 1)));
    }
  } else {
    {  // convc1 1x1 196->96 + relu -> cor_flo[0:96)
      tc_params_init(p, EPI_LINEAR, ACT_RELU, 96);
      p.out_hi = W.cf_hi; p.out_lo = W.cf_lo; p.h_stride = d.s_cf;
      TcSeg s[1] = {{W.corr_hi, W.corr_lo, d.s_corr, 0, 4}};
      RAFT_TRY(launch_tc_layer(c, 0, 1, s, p));
    }
    {  // convf1 7x7 2->64 + relu via im2col + 1x1 GEMM
      const size_t npix = (size_t)c.B * c.h * c.w;
      if (!c.fim_ready) {
        flow_im2col_kernel<<<grid_for(npix * 128), 256, 0, c.stream>>>(W.flow, c.B, c.h, c.w, W.fim_hi, W.fim_lo);
        RAFT_COUNT_LAUNCH();
      }
      tc_params_init(p, EPI_LINEAR, ACT_RELU, 64);
      p.out_hi = W.flo1_hi; p.out_lo = W.flo1_lo; p.h_stride = d.s_flo1;
      TcSeg s[1] = {{W.fim_hi, W.fim_lo, 128, 0, 2}};
      RAFT_TRY(launch_tc_layer(c, 7, 1, s, p));
    }
    {  // convf2 3x3 64->32 + relu -> cor_flo[96:128)
      tc_params_init(p, EPI_LINEAR, ACT_RELU, 32);
      p.out_hi = W.cf_hi; p.out_lo = W.cf_lo; p.h_stride = d.s_cf; p.h_c0 = 96;
      TcSeg s[1] = {{W.flo1_hi, W.flo1_lo, d.s_flo1, 0, 1}};
      RAFT_TRY(launch_tc_layer(c, 1, 1, s, p, -1, dep1(7)));
    }
    {  // conv 3x3 128->80 + relu, concat flow -> x[64:160)
      tc_params_init(p, EPI_LINEAR, ACT_RELU, 80);
      p.out_hi = W.x_hi; p.out_lo = W.x_lo; p.h_stride = d.s_x; p.h_c0 = 64;
      p.concat_src = W.flow; p.concat_n = 2;
      TcSeg s[1] = {{W.cf_hi, W.cf_lo, d.s_cf, 0, 2}};
      RAFT_TRY(launch_tc_layer(c, 2, 1, s, p, -1, dep2(0, 1)));
    }
    RAFT_TRY(gru_tc(c, h, 3, 4, 96, 3, 2));
    {  // flow_head.conv1 3x3 96->128 + relu
      tc_params_init(p, EPI_LINEAR, ACT_RELU, 128);
      p.out_hi = W.fm_hi; p.out_lo = W.fm_lo; p.h_stride = d.s_fm;
      TcSeg s[1] = {{W.h_hi, W.h_lo, d.s_h, 0, 2}};
      RAFT_TRY(launch_tc_layer(c, 5, 1, s, p, -1, dep1(4)));
    }
    {  // flow_head.conv2 3x3 128->2
      tc_params_init(p, EPI_LINEAR, ACT_NONE, 2);
      p.out_f32 = delta; p.f32_stride = 2;
      p.adv_coords = adv_coords; p.adv_flow = adv_coords ? W.flow : nullptr;
      TcSeg s[1] = {{W.fm_hi, W.fm_lo, d.s_fm, 0, 2}};
      RAFT_TRY(launch_tc_layer(c, 6, 1, s, p, -1, dep1(5)));
    }
  }
  return 0;
}

// Per-pair setup shared by the update_* entry points and the loop: zero the fp16 planes (their
// padded channels must hold exact zeros), stage inp and the hidden state in operand format.
static int update_begin(const UpdateCtx& c, const float* h, const float* inp) {
  const Workspace& W = c.W;
  const VariantDims d = variant_dims(c.variant);
  const size_t npix = (size_t)c.B * c.h * c.w;
  if (c.precision == RAFT_PREC_F16X2) {
    RAFT_CUDA_TRY(cudaMemsetAsync(W.f16_begin, 0, W.f16_bytes, c.stream));
    split_plane_kernel<<<grid_for(npix * d.ctx), 256, 0, c.stream>>>(inp, d.ctx, 0, d.ctx, d.ctx, W.x_hi, W.x_lo, d.s_x,
                                                                      0, npix, 1.0f);
    RAFT_COUNT_LAUNCH();
    split_plane_kernel<<<grid_for(npix * d.hid), 256, 0, c.stream>>>(h, d.hid, 0, d.hid, d.hid, W.h_hi, W.h_lo, d.s_h, 0,
                                                                      npix, 1.0f);
    RAFT_COUNT_LAUNCH();
  } else {
    RAFT_CUDA_TRY(cudaMemsetAsync(W.x, 0, npix * d.c_x * sizeof(float), c.stream));
    copy_channels_kernel<<<grid_for(npix * d.ctx), 256, 0, c.stream>>>(inp, d.ctx, 0, W.x, d.c_x, 0, d.ctx, npix);
    RAFT_COUNT_LAUNCH();
  }
  return raft_launch_status();
}

static int make_ctx(UpdateCtx& c, int variant, const void* prepared, int B, int h, int w, void* ws, size_t ws_bytes,
                    int precision, void* stream) {
  if (variant != RAFT_VARIANT_BASIC && variant != RAFT_VARIANT_SMALL) return RAFT_ERR_BAD_ARG;
  if (precision != RAFT_PREC_FP32 && precision != RAFT_PREC_F16X2) return RAFT_ERR_BAD_ARG;
  if (!prepared || !ws) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  c.variant = variant; c.precision = precision; c.B = B; c.h = h; c.w = w;
  c.prepared = reinterpret_cast<const uint8_t*>(prepared);
  c.PL = prepared_layout(variant, precision);
  c.W = workspace_layout(ws, variant, B, h, w, precision);
  if (c.W.total > ws_bytes) return RAFT_ERR_WORKSPACE;
  c.stream = reinterpret_cast<cudaStream_t>(stream);
  c.plan = nullptr;
  c.fim_ready = false;
  return 0;
}

// One update_mega_kernel launch for all tensor-core layers of an update-block application (default), or one launch per
// layer (RAFT_B200_MEGA=0: A/B timing and bisecting).
static bool mega_enabled() {
  static const int v = [] { const char* e = getenv("RAFT_B200_MEGA"); return e ? atoi(e) : 1; }();
  return v != 0;
}
// CTA pairs (update_mega_kernel<true>) whenever the number of pixel tiles is even; RAFT_B200_PAIR=0 keeps single CTAs (A/B).
static bool pair_enabled() {
  static const int v = [] { const char* e = getenv("RAFT_B200_PAIR"); return e ? atoi(e) : 1; }();
  return v != 0;
}
static int update_block_tc(UpdateCtx& c, float* h, float* delta, float* mask, float* adv_coords) {
  MegaPlan plan;
  c.plan = mega_enabled() ? &plan : nullptr;
  {
    int tw, th;
    tc_pick_tile(c.w, c.h, &tw, &th);
    const int mtiles = c.B * ceil_div(c.h, th) * ceil_div(c.w, tw);
    plan.pair = pair_enabled() && (mtiles % 2 == 0) ? 1 : 0;
  }
  const int st = update_core_tc(c, h, delta, mask, adv_coords);
  c.plan = nullptr;
  RAFT_TRY(st);
  if (!mega_enabled()) return 0;
  RAFT_COUNT_LAUNCH();
  return mega_launch(plan, c.W.mega_flags, c.W.mega_flag_words, true, c.stream);
}

static int update_once(int variant, const void* prepared, const float* net, const float* inp, const float* corr,
                       const float* flow, float* net_out, float* mask, float* delta, int B, int h, int w, void* ws,
                       size_t ws_bytes, int precision, void* stream) {
  if (!net || !inp || !corr || !flow || !net_out || !delta) return RAFT_ERR_BAD_ARG;
  UpdateCtx c;
  RAFT_TRY(make_ctx(c, variant, prepared, B, h, w, ws, ws_bytes, precision, stream));
  const VariantDims d = variant_dims(variant);
  const size_t npix = (size_t)B * h * w;
  if (net_out != net)
    RAFT_CUDA_TRY(cudaMemcpyAsync(net_out, net, npix * d.hid * sizeof(float), cudaMemcpyDeviceToDevice, c.stream));
  RAFT_CUDA_TRY(cudaMemcpyAsync(c.W.flow, flow, npix * 2 * sizeof(float), cudaMemcpyDeviceToDevice, c.stream));
  RAFT_TRY(update_begin(c, net_out, inp));
  if (precision == RAFT_PREC_F16X2) {
    split_plane_kernel<<<grid_for(npix * d.s_corr), 256, 0, c.stream>>>(corr, d.corr_ch, 0, d.corr_ch, d.s_corr,
                                                                         c.W.corr_hi, c.W.corr_lo, d.s_corr, 0, npix, 1.0f);
    RAFT_COUNT_LAUNCH();
    return update_block_tc(c, net_out, delta, mask, nullptr);
  }
  RAFT_CUDA_TRY(cudaMemcpyAsync(c.W.corr, corr, npix * d.corr_ch * sizeof(float), cudaMemcpyDeviceToDevice, c.stream));
  return update_core_fp32(c, net_out, delta, mask);
}

// im_flow != null (iteration loop, tensor-core path): the convf1 im2col planes im_hi / im_lo are produced too -- by the
// window kernel itself when it runs, else by flow_im2col_kernel.
static int lookup_launch(const float* const pyr[], const float* coords, int B, int h, int w, int levels, int radius,
                         float* out, int out_stride, __half* out_hi, __half* out_lo, int h_stride, int h_pad,
                         cudaStream_t st, const float* im_flow = nullptr, __half* im_hi = nullptr, __half* im_lo = nullptr) {
  LookupParams p;
  memset(&p, 0, sizeof(p));
  int lh = h, lw = w;
  for (int l = 0; l < levels; ++l) {
    if (lh < 1 || lw < 1) return RAFT_ERR_BAD_SHAPE;
    p.pyr[l] = pyr[l];
    p.lh[l] = lh;
    p.lw[l] = lw;
    lh /= 2;
    lw /= 2;
  }
  p.coords = coords;
  p.out = out; p.out_stride = out_stride;
  p.out_hi = out_hi; p.out_lo = out_lo; p.h_stride = h_stride; p.h_pad = h_pad;
  p.nq = B * h * w; p.levels = levels; p.radius = radius;
  p.im_flow = im_flow; p.im_hi = im_hi; p.im_lo = im_lo; p.im_B = B; p.im_h = h; p.im_w = w;
  const size_t nwork = (size_t)p.nq * levels;
  static const int gather = [] { const char* e = getenv("RAFT_B200_LOOKUP_GATHER"); return e ? atoi(e) : 0; }();   // A/B: force the generic kernel
  if (gather || !lookup_win_launch(p, levels, radius, st)) {       // window kernel for the model's (radius, levels); else generic
    corr_lookup_kernel<<<grid_for(nwork * 32, 256, kNumSMs * 32), 256, 0, st>>>(p);
    if (im_flow) {
      flow_im2col_kernel<<<grid_for((size_t)p.nq * 128), 256, 0, st>>>(im_flow, B, h, w, im_hi, im_lo);
      RAFT_COUNT_LAUNCH();
    }
  }
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

}  // namespace raft

using namespace raft;

// =================================================================================================
extern "C" {

const char* raft_b200_strerror(int status) {
  switch (status) {
    case RAFT_OK: return "ok";
    case RAFT_ERR_BAD_ARG: return "bad argument (null pointer or unknown enum)";
    case RAFT_ERR_BAD_SHAPE: return "bad shape";
    case RAFT_ERR_WORKSPACE: return "workspace or prepared-weights buffer too small";
    case RAFT_ERR_NO_DEVICE: return "no sm_100 CUDA device";
    case RAFT_ERR_DRIVER: return "cuTensorMapEncodeTiled unavailable or failed";
    case RAFT_ERR_UNSUPPORTED: return "unsupported configuration";
    default: return status > 0 ? cudaGetErrorString((cudaError_t)status) : "unknown raft_status";
  }
}

int raft_b200_abi_version(void) { return RAFT_B200_ABI_VERSION; }

int raft_b200_device_ok(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) {
    (void)cudaGetLastError();
    return RAFT_ERR_NO_DEVICE;
  }
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess) return RAFT_ERR_NO_DEVICE;
  return major == 10 ? RAFT_OK : RAFT_ERR_NO_DEVICE;
}

void raft_b200_profile_loop(int enable) { g_prof.on = enable != 0; g_prof.n = 0; }
int raft_b200_profile_read(float* lookup_ms, float* update_ms, int* iterations) {
  if (!lookup_ms || !update_ms || !iterations) return RAFT_ERR_BAD_ARG;
  *lookup_ms = 0.f; *update_ms = 0.f; *iterations = g_prof.n;
  for (int i = 0; i < g_prof.n; ++i) {
    float a = 0.f, b = 0.f;
    RAFT_CUDA_TRY(cudaEventSynchronize(g_prof.ev[i][2]));
    RAFT_CUDA_TRY(cudaEventElapsedTime(&a, g_prof.ev[i][0], g_prof.ev[i][1]));
    RAFT_CUDA_TRY(cudaEventElapsedTime(&b, g_prof.ev[i][1], g_prof.ev[i][2]));
    *lookup_ms += a;
    *update_ms += b;
  }
  return RAFT_OK;
}

long long raft_b200_launch_count(void) { return g_launches; }
void raft_b200_debug_timeline(int tc_layer, long long* device_buf_2048) {
  g_dbg_layer = tc_layer;
  g_dbg_count = 0;
  g_dbg_buf = device_buf_2048;
}
void raft_b200_launch_count_reset(void) { g_launches = 0; }

int raft_b200_corr_pyramid_sizes(int B, int h, int w, int levels, size_t bytes_per_level[]) {
  if (!bytes_per_level || levels < 1 || levels > RAFT_MAX_LEVELS) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  int lh = h, lw = w;
  for (int l = 0; l < levels; ++l) {
    if (lh < 1 || lw < 1) return RAFT_ERR_BAD_SHAPE;
    bytes_per_level[l] = (size_t)B * h * w * lh * lw * sizeof(float);
    lh /= 2;
    lw /= 2;
  }
  return RAFT_OK;
}

int raft_b200_corr_workspace_bytes(int B, int h, int w, int C, int levels, int precision, size_t* bytes) {
  if (!bytes || levels < 1 || levels > RAFT_MAX_LEVELS) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  if (C < 1) return RAFT_ERR_BAD_SHAPE;
  *bytes = corr_ws_layout(nullptr, B, h, w, C, levels, precision).total + 1024;
  return RAFT_OK;
}

int raft_b200_corr_pyramid_build(const float* fmap1, const float* fmap2, int B, int h, int w, int C, int levels,
                                 float* const pyr[], void* workspace, size_t workspace_bytes, int precision,
                                 void* stream) {
  if (!fmap1 || !fmap2 || !pyr || levels < 1 || levels > RAFT_MAX_LEVELS) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  if (C < 1 || (h >> (levels - 1)) < 1 || (w >> (levels - 1)) < 1) return RAFT_ERR_BAD_SHAPE;
  for (int l = 0; l < levels; ++l)
    if (!pyr[l]) return RAFT_ERR_BAD_ARG;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (precision == RAFT_PREC_FP32) return corr_build_fp32(fmap1, fmap2, B, h, w, C, levels, pyr, st);
  if (precision != RAFT_PREC_F16X2) return RAFT_ERR_BAD_ARG;
  if (!workspace || corr_ws_layout(nullptr, B, h, w, C, levels, precision).total > workspace_bytes)
    return RAFT_ERR_WORKSPACE;
  return corr_build_tc(fmap1, fmap2, B, h, w, C, levels, pyr, workspace, st);
}

int raft_b200_corr_lookup(const float* const pyr[], const float* coords, int B, int h, int w, int levels, int radius,
                          float* out, int out_stride, void* stream) {
  if (!pyr || !coords || !out || levels < 1 || levels > RAFT_MAX_LEVELS || radius < 0) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  const int side = 2 * radius + 1;
  if (out_stride < levels * side * side) return RAFT_ERR_BAD_SHAPE;
  return lookup_launch(pyr, coords, B, h, w, levels, radius, out, out_stride, nullptr, nullptr, 0, 0,
                       reinterpret_cast<cudaStream_t>(stream));
}

int raft_b200_corr_lookup_backward(const float* const pyr[], const float* coords, const float* grad_out, int B, int h, int w,
                                   int levels, int radius, float* grad_coords, float* const grad_pyr[], void* stream) {
  if (!pyr || !coords || !grad_out || !grad_coords || !grad_pyr || levels < 1 || levels > RAFT_MAX_LEVELS || radius < 0)
    return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  LookupBwdParams p;
  memset(&p, 0, sizeof(p));
  int lh = h, lw = w;
  for (int l = 0; l < levels; ++l) {
    if (lh < 1 || lw < 1) return RAFT_ERR_BAD_SHAPE;
    if (!pyr[l] || !grad_pyr[l]) return RAFT_ERR_BAD_ARG;
    p.pyr[l] = pyr[l]; p.gpyr[l] = grad_pyr[l]; p.lh[l] = lh; p.lw[l] = lw;
    lh /= 2;
    lw /= 2;
  }
  const int side = 2 * radius + 1;
  p.coords = coords; p.gout = grad_out; p.gout_stride = levels * side * side; p.gcoords = grad_coords;
  p.nq = B * h * w; p.levels = levels; p.radius = radius;
  const size_t nwork = (size_t)p.nq * levels;
  corr_lookup_bwd_kernel<<<grid_for(nwork * 32, 256, kNumSMs * 32), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_sumsq(const float* g, size_t n, float* partials, size_t npartials, float* out, void* stream) {
  if (!g || !partials || !out || npartials < 1) return RAFT_ERR_BAD_ARG;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int blocks = (int)std::min<size_t>(std::min<size_t>(npartials, (size_t)kNumSMs * 4), (n + 255) / 256);
  if (blocks < 1) blocks = 1;
  sumsq_partial_kernel<<<blocks, 256, 0, st>>>(g, n, partials);
  sumsq_final_kernel<<<1, 256, 0, st>>>(partials, blocks, out);
  g_launches += 2;
  return raft_launch_status();
}

int raft_b200_adamw_step(float* param, const float* grad, float* m, float* v, size_t n, const float* sumsq, float clip_norm,
                         float lr_t, float beta1, float beta2, float epsilon, float weight_decay, void* stream) {
  if (!param || !grad || !m || !v || (clip_norm > 0.0f && !sumsq)) return RAFT_ERR_BAD_ARG;
  adamw_kernel<<<grid_for(n), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(param, grad, m, v, n, sumsq, clip_norm, lr_t,
                                                                             beta1, beta2, epsilon, weight_decay);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_bilinear_sampler(const float* image, const float* coords, int M, int H, int W, int P, float* out,
                               void* stream) {
  if (!image || !coords || !out) return RAFT_ERR_BAD_ARG;
  if (M < 1 || H < 1 || W < 1 || P < 1) return RAFT_ERR_BAD_SHAPE;
  bilinear_sampler_kernel<<<grid_for((size_t)M * P), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(image, coords, M,
                                                                                                      H, W, P, out);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_coords_grid(int B, int h, int w, float* out, void* stream) {
  if (!out) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  coords_grid_kernel<<<grid_for((size_t)B * h * w), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(out, B, h, w);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_update_prepared_bytes(int variant, int corr_channels, int precision, size_t* bytes) {
  if (!bytes) return RAFT_ERR_BAD_ARG;
  if (variant != RAFT_VARIANT_BASIC && variant != RAFT_VARIANT_SMALL) return RAFT_ERR_BAD_ARG;
  if (precision != RAFT_PREC_FP32 && precision != RAFT_PREC_F16X2) return RAFT_ERR_BAD_ARG;
  if (corr_channels != variant_dims(variant).corr_ch) return RAFT_ERR_BAD_SHAPE;
  *bytes = prepared_layout(variant, precision).total;
  return RAFT_OK;
}

int raft_b200_update_prepare(int variant, const void* weights, void* prepared, size_t prepared_bytes, int precision,
                             void* stream) {
  if (!weights || !prepared) return RAFT_ERR_BAD_ARG;
  if (variant != RAFT_VARIANT_BASIC && variant != RAFT_VARIANT_SMALL) return RAFT_ERR_BAD_ARG;
  if (precision != RAFT_PREC_FP32 && precision != RAFT_PREC_F16X2) return RAFT_ERR_BAD_ARG;
  const PreparedLayout L = prepared_layout(variant, precision);
  if (L.total > prepared_bytes) return RAFT_ERR_WORKSPACE;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const raft_conv* convs = reinterpret_cast<const raft_conv*>(weights);   // both structs are arrays of raft_conv
  const ConvDim* cd = conv_dims(variant);
  uint8_t* base = reinterpret_cast<uint8_t*>(prepared);
  for (int i = 0; i < n_convs(variant); ++i) {
    const raft_conv& cv = convs[i];
    if (!cv.kernel || !cv.bias) return RAFT_ERR_BAD_ARG;
    if (cv.kh != cd[i].kh || cv.kw != cd[i].kw || cv.cin != cd[i].cin || cv.cout != cd[i].cout) return RAFT_ERR_BAD_SHAPE;
  }
  RAFT_CUDA_TRY(cudaMemsetAsync(base, 0, L.total, st));
  for (int i = 0; i < n_convs(variant); ++i) {
    const size_t nw = (size_t)cd[i].kh * cd[i].kw * cd[i].cin * cd[i].cout;
    RAFT_CUDA_TRY(cudaMemcpyAsync(base + L.raw_w[i], convs[i].kernel, nw * sizeof(float), cudaMemcpyDeviceToDevice, st));
    RAFT_CUDA_TRY(cudaMemcpyAsync(base + L.raw_b[i], convs[i].bias, cd[i].cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  if (precision == RAFT_PREC_F16X2) {
    const TcLayerSpec* tl = tc_layers(variant);
    for (int li = 0; li < n_tc_layers(variant); ++li) {
      const TcLayerSpec& T = tl[li];
      unsigned int* amax = reinterpret_cast<unsigned int*>(base + L.tc_absmax[li]);
      float* scale = reinterpret_cast<float*>(base + L.tc_scale[li]);
      for (int s = 0; s < T.nsrc; ++s) {
        const int ci = T.src[s];
        const size_t nw = (size_t)cd[ci].kh * cd[ci].kw * cd[ci].cin * cd[ci].cout;
        absmax_kernel<<<grid_for(nw), 256, 0, st>>>(convs[ci].kernel, nw, amax);
        RAFT_COUNT_LAUNCH();
      }
      weight_scale_kernel<<<1, 1, 0, st>>>(amax, scale);
      RAFT_COUNT_LAUNCH();
      int cout_off = 0;
      for (int s = 0; s < T.nsrc; ++s) {
        const int ci = T.src[s];
        PackParams pp;
        memset(&pp, 0, sizeof(pp));
        pp.w = convs[ci].kernel;
        pp.kh = cd[ci].kh; pp.kw = cd[ci].kw; pp.cin = cd[ci].cin; pp.cout = cd[ci].cout;
        if (T.flatten) { pp.cin = pp.kh * pp.kw * pp.cin; pp.kh = pp.kw = 1; }   // HWIO is already [tap*cin + c][cout]
        pp.hi = reinterpret_cast<__half*>(base + L.tc_hi[li]);
        pp.lo = reinterpret_cast<__half*>(base + L.tc_lo[li]);
        pp.cout_pad = T.cout_pad; pp.cin_pad = T.cin_pad; pp.cout_off = cout_off;
        pp.nrange = T.nrange;
        for (int r = 0; r < T.nrange; ++r) {
          pp.r_src0[r] = T.r_src0[r];
          pp.r_n[r] = T.r_n[r];
          pp.r_dst0[r] = T.r_dst0[r];
        }
        pp.scale = scale;
        const size_t nw = (size_t)cd[ci].kh * cd[ci].kw * cd[ci].cin * cd[ci].cout;
        pack_weights_kernel<<<grid_for(nw), 256, 0, st>>>(pp);
        RAFT_COUNT_LAUNCH();
        RAFT_CUDA_TRY(cudaMemcpyAsync(base + L.tc_bias[li] + cout_off * sizeof(float), convs[ci].bias,
                                      cd[ci].cout * sizeof(float), cudaMemcpyDeviceToDevice, st));
        cout_off += cd[ci].cout;
      }
    }
  }
  return raft_launch_status();
}

int raft_b200_update_workspace_bytes(int variant, int B, int h, int w, int precision, size_t* bytes) {
  if (!bytes) return RAFT_ERR_BAD_ARG;
  if (variant != RAFT_VARIANT_BASIC && variant != RAFT_VARIANT_SMALL) return RAFT_ERR_BAD_ARG;
  if (precision != RAFT_PREC_FP32 && precision != RAFT_PREC_F16X2) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  *bytes = workspace_layout(nullptr, variant, B, h, w, precision).total;
  return RAFT_OK;
}

int raft_b200_update_basic(const void* prepared, const float* net, const float* inp, const float* corr,
                           const float* flow, float* net_out, float* mask_or_null, float* delta_flow, int B, int h,
                           int w, void* workspace, size_t workspace_bytes, int precision, void* stream) {
  return update_once(RAFT_VARIANT_BASIC, prepared, net, inp, corr, flow, net_out, mask_or_null, delta_flow, B, h, w,
                     workspace, workspace_bytes, precision, stream);
}

int raft_b200_update_small(const void* prepared, const float* net, const float* inp, const float* corr,
                           const float* flow, float* net_out, float* delta_flow, int B, int h, int w, void* workspace,
                           size_t workspace_bytes, int precision, void* stream) {
  return update_once(RAFT_VARIANT_SMALL, prepared, net, inp, corr, flow, net_out, nullptr, delta_flow, B, h, w,
                     workspace, workspace_bytes, precision, stream);
}

int raft_b200_upsample_convex(const float* flow, const float* mask, int B, int h, int w, float* out, void* stream) {
  if (!flow || !mask || !out) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  const size_t npix = (size_t)B * h * w;
  upsample_convex_kernel<<<grid_for(npix, 4, kNumSMs * 32), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(flow, mask,
                                                                                                            B, h, w, out);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_upflow8(const float* flow, int B, int h, int w, float* out, void* stream) {
  if (!flow || !out) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  upflow8_kernel<<<grid_for((size_t)B * h * w * 64), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(flow, B, h, w, out);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_forward_interpolate(const float* flow, int B, int h, int w, int out_coords, float* out, void* stream) {
  if (!flow || !out) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, h, w));
  if (B > 65535 || (long long)h * w > (1ll << 30)) return RAFT_ERR_BAD_SHAPE;         // grid.y; int sample indices
  const size_t n = (size_t)B * h * w * 2;
  if (out < flow + n && flow < out + n) return RAFT_ERR_BAD_ARG;                      // out must not overlap flow
  const dim3 grid((unsigned)((h * w + kFwdInterpThreads - 1) / kFwdInterpThreads), (unsigned)B);
  forward_interpolate_kernel<<<grid, kFwdInterpThreads, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      flow, h, w, out_coords, out);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_encoder_prepared_bytes(int variant, int out_dim, size_t* bytes) {
  if (!bytes || (variant != RAFT_VARIANT_BASIC && variant != RAFT_VARIANT_SMALL)) return RAFT_ERR_BAD_ARG;
  if (out_dim < 32 || out_dim > 256 || out_dim % 32) return RAFT_ERR_BAD_SHAPE;
  *bytes = enc_layout(variant, out_dim).total;
  return RAFT_OK;
}

int raft_b200_encoder_prepare(int variant, int norm_type, int out_dim, const raft_encoder_weights* weights,
                              void* prepared, size_t prepared_bytes, void* stream) {
  if (!weights || !prepared || (variant != RAFT_VARIANT_BASIC && variant != RAFT_VARIANT_SMALL)) return RAFT_ERR_BAD_ARG;
  if (norm_type < 0 || norm_type > 2) return RAFT_ERR_BAD_ARG;
  if (out_dim < 32 || out_dim > 256 || out_dim % 32) return RAFT_ERR_BAD_SHAPE;
  return encoder_prepare(variant, norm_type, out_dim, weights, prepared, prepared_bytes, reinterpret_cast<cudaStream_t>(stream));
}

int raft_b200_encoder_workspace_bytes(int variant, int N, int H, int W, size_t* bytes) {
  if (!bytes || (variant != RAFT_VARIANT_BASIC && variant != RAFT_VARIANT_SMALL)) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(N, H, W));
  *bytes = enc_ws_layout(nullptr, variant, N, H, W).total;
  return RAFT_OK;
}

int raft_b200_encoder_forward(int variant, int norm_type, int out_dim, const void* prepared, const float* images,
                              int N, int H, int W, int training, int image_norm, float* out, void* workspace,
                              size_t workspace_bytes, void* stream) {
  if (!prepared || !images || !out || !workspace) return RAFT_ERR_BAD_ARG;
  if (variant != RAFT_VARIANT_BASIC && variant != RAFT_VARIANT_SMALL) return RAFT_ERR_BAD_ARG;
  if (norm_type < 0 || norm_type > 2) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(N, H, W));
  if (out_dim < 32 || out_dim > 256 || out_dim % 32 || H < 8 || W < 8) return RAFT_ERR_BAD_SHAPE;
  return encoder_forward(variant, norm_type, out_dim, prepared, images, N, H, W, training, image_norm, out, workspace, workspace_bytes,
                         reinterpret_cast<cudaStream_t>(stream));
}

int raft_b200_context_split(const float* cnet, int npix, int hidden, int context, float* net, float* inp,
                            void* stream) {
  if (!cnet || !net || !inp) return RAFT_ERR_BAD_ARG;
  if (npix < 1 || hidden < 1 || context < 1) return RAFT_ERR_BAD_SHAPE;
  context_split_kernel<<<grid_for((size_t)npix * (hidden + context)), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      cnet, (size_t)npix, hidden, context, net, inp);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_conv2d(const float* x, const float* kernel, const float* bias, int B, int H, int W, int cin, int kh,
                     int kw, int cout, int act, float* out, int out_stride, int out_c0, void* stream) {
  if (!x || !kernel || !out) return RAFT_ERR_BAD_ARG;
  RAFT_TRY(check_dims(B, H, W));
  if (cin < 1 || cout < 1 || kh < 1 || kw < 1 || !(kh & 1) || !(kw & 1) || act < 0 || act > 3) return RAFT_ERR_BAD_SHAPE;
  if (out_stride < out_c0 + cout) return RAFT_ERR_BAD_SHAPE;
  SimtConvParams p;
  memset(&p, 0, sizeof(p));
  p.src[0] = x; p.src_stride[0] = cin; p.src_c0[0] = 0; p.src_n[0] = cin; p.nsrc = 1;
  p.w = kernel; p.bias = bias;
  p.kh = kh; p.kw = kw; p.cin = cin; p.cout = cout;
  p.B = B; p.H = H; p.W = W;
  p.out = out; p.out_stride = out_stride; p.out_c0 = out_c0;
  p.act = act; p.out_scale = 1.0f;
  dim3 grid((unsigned)ceil_div(B * H * W, 64), (unsigned)ceil_div(cout, 64));
  conv_simt_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  RAFT_COUNT_LAUNCH();
  return raft_launch_status();
}

int raft_b200_forward_loop(int variant, const void* prepared, const float* const pyr[], int levels, int radius,
                           float* net, const float* inp, float* coords1, float* const flow_up[], int iters, int B,
                           int h, int w, void* workspace, size_t workspace_bytes, int precision, void* stream) {
  if (!pyr || !net || !inp || !coords1 || !flow_up || iters < 0) return RAFT_ERR_BAD_ARG;
  if (levels < 1 || levels > RAFT_MAX_LEVELS || radius < 0) return RAFT_ERR_BAD_ARG;
  UpdateCtx c;
  RAFT_TRY(make_ctx(c, variant, prepared, B, h, w, workspace, workspace_bytes, precision, stream));
  const VariantDims d = variant_dims(variant);
  const int side = 2 * radius + 1;
  if (levels * side * side != d.corr_ch) return RAFT_ERR_BAD_SHAPE;
  const size_t npix = (size_t)B * h * w;
  const Workspace& W = c.W;
  RAFT_TRY(update_begin(c, net, inp));
  flow_advance_kernel<<<grid_for(npix), 256, 0, c.stream>>>(coords1, nullptr, W.flow, B, h, w);   // model.py:97
  RAFT_COUNT_LAUNCH();
  const bool prof = g_prof.on && iters <= 64;
  if (prof && !g_prof.created) {
    for (int i = 0; i < 64; ++i)
      for (int k = 0; k < 3; ++k) RAFT_CUDA_TRY(cudaEventCreate(&g_prof.ev[i][k]));
    g_prof.created = true;
  }
  if (prof) g_prof.n = iters;
  for (int i = 0; i < iters; ++i) {
    float* mask = (variant == RAFT_VARIANT_BASIC && flow_up[i]) ? W.mask : nullptr;
    if (precision == RAFT_PREC_F16X2) {
      if (prof) RAFT_CUDA_TRY(cudaEventRecord(g_prof.ev[i][0], c.stream));
      RAFT_TRY(lookup_launch(pyr, coords1, B, h, w, levels, radius, nullptr, 0, W.corr_hi, W.corr_lo, d.s_corr, d.s_corr,
                             c.stream, W.flow, W.fim_hi, W.fim_lo));                                // model.py:95 (+ convf1's im2col)
      if (prof) RAFT_CUDA_TRY(cudaEventRecord(g_prof.ev[i][1], c.stream));
      c.fim_ready = true;
      RAFT_TRY(update_block_tc(c, net, W.delta, mask, coords1));                                    // :99, :102 (fused advance)
      c.fim_ready = false;
      if (prof) RAFT_CUDA_TRY(cudaEventRecord(g_prof.ev[i][2], c.stream));
    } else {
      RAFT_TRY(lookup_launch(pyr, coords1, B, h, w, levels, radius, W.corr, d.corr_ch, nullptr, nullptr, 0, 0, c.stream));
      RAFT_TRY(update_core_fp32(c, net, W.delta, mask));
      flow_advance_kernel<<<grid_for(npix), 256, 0, c.stream>>>(coords1, W.delta, W.flow, B, h, w);  // :102
      RAFT_COUNT_LAUNCH();
    }
    if (flow_up[i]) {                                                                               // :105 / :223
      if (variant == RAFT_VARIANT_BASIC)
        RAFT_TRY(raft_b200_upsample_convex(W.flow, W.mask, B, h, w, flow_up[i], stream));
      else
        RAFT_TRY(raft_b200_upflow8(W.flow, B, h, w, flow_up[i], stream));
    }
  }
  return raft_launch_status();
}

}  // extern "C"
