// tcr_api.cu — C ABI of libtcr_b200 (include/tcr_b200.h): handle, constant tables, layer plan,
// workspace and the per-call launch sequences.  No torch types; the caller owns tensors and the stream.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <random>

#include "tcr_net.h"
#include "tcr_plan.h"

using namespace tcr;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define TCR_CUDA(call)                                                                         \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) return fail(TCR_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

extern "C" int tcr_abi_version(void) { return TCR_ABI_VERSION; }
extern "C" const char* tcr_last_error(void) { return g_err; }

extern "C" int tcr_config_default(tcr_config* cfg) {
  if (!cfg) return fail(TCR_ERR_INVALID, "cfg is NULL");
  memset(cfg, 0, sizeof(*cfg));
  cfg->model = TCR_MODEL_TCRESNET8;
  cfg->width_multiplier = 1.0f;
  cfg->num_classes = 12;
  cfg->sample_rate = 16000;
  cfg->clip_samples = 16000;
  cfg->window_size_samples = 640;
  cfg->window_stride_samples = 320;
  cfg->num_mel_bins = 64;
  cfg->num_mfccs = 40;
  cfg->lower_edge_hertz = 80.0f;
  cfg->upper_edge_hertz = 7600.0f;
  cfg->feature_kind = TCR_FEATURE_MFCC;
  cfg->max_batch = 512;
  cfg->bn_decay = 0.997f;
  cfg->bn_epsilon = 0.001f;
  cfg->dropout_keep_prob = 0.5f;
  cfg->label_smoothing = 0.0f;
  cfg->device = 0;
  return TCR_OK;
}

// ------------------------------------------------------------------------------------------------
// device allocation helpers
// ------------------------------------------------------------------------------------------------
template <class T>
static int dev_alloc(tcr_handle* h, T** p, size_t count) {
  void* q = nullptr;
  size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
  bytes = (bytes + 255) & ~(size_t)255;
  if (cudaMalloc(&q, bytes) != cudaSuccess) return fail(TCR_ERR_CUDA, "cudaMalloc(%zu bytes) failed", bytes);
  h->allocs.push_back(q);
  h->workspace_bytes += (int64_t)bytes;
  *p = (T*)q;
  return TCR_OK;
}
template <class T>
static int dev_upload(tcr_handle* h, T** p, const std::vector<T>& v) {
  int rc = dev_alloc(h, p, v.size());
  if (rc) return rc;
  if (!v.empty()) TCR_CUDA(cudaMemcpy(*p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
  return TCR_OK;
}
#define TCR_TRY(x)            \
  do {                        \
    int rc_ = (x);            \
    if (rc_) return rc_;      \
  } while (0)

// ------------------------------------------------------------------------------------------------
// front-end tables (datasets/preprocessors.py:64-96, 183-194; TF r1.13 op semantics, SURVEY.md 8c)
// ------------------------------------------------------------------------------------------------
static int next_pow2(int n) {
  int p = 1;
  while (p < n) p <<= 1;
  return p;
}

static int build_frontend_tables(tcr_handle* h) {
  const tcr_config& c = h->cfg;
  const int W = c.window_size_samples, fft = h->fft, nf2 = fft / 2, bins = nf2 + 1;
  // tf.contrib.signal.hann_window(periodic=True): n = W + even - 1, w = 0.5 - 0.5 cos(2 pi i / n)
  std::vector<float> win(W);
  const int even = 1 - W % 2;
  const double nn = (double)(W + even - 1);
  for (int i = 0; i < W; ++i) win[i] = (float)(0.5 - 0.5 * cos(2.0 * M_PI * i / nn));
  std::vector<float2> tw(nf2), tw2(bins);
  for (int i = 0; i < nf2; ++i) {
    const double a = -2.0 * M_PI * i / nf2;
    tw[i] = make_float2((float)cos(a), (float)sin(a));
  }
  for (int k = 0; k < bins; ++k) {
    const double a = -2.0 * M_PI * k / fft;
    tw2[k] = make_float2((float)cos(a), (float)sin(a));
  }
  // linear_to_mel_weight_matrix(num_mel_bins, bins, sample_rate, lower, upper): HTK mel, DC bin zeroed.
  const int M = c.num_mel_bins;
  auto mel = [](double f) { return 1127.0 * log(1.0 + f / 700.0); };
  std::vector<double> edges(M + 2);
  const double mlo = mel(c.lower_edge_hertz), mhi = mel(c.upper_edge_hertz);
  for (int i = 0; i < M + 2; ++i) edges[i] = mlo + (mhi - mlo) * i / (M + 1);
  std::vector<int> start(M, 0), len(M, 0), off(M, 0);
  std::vector<float> wts;
  const double nyq = c.sample_rate / 2.0;
  for (int m = 0; m < M; ++m) {
    const double lo = edges[m], ce = edges[m + 1], up = edges[m + 2];
    int first = -1, last = -1;
    std::vector<float> row;
    for (int k = 1; k < bins; ++k) {
      const double fm = mel(nyq * k / (bins - 1));
      const double w = std::max(0.0, std::min((fm - lo) / (ce - lo), (up - fm) / (up - ce)));
      if (w > 0.0) {
        if (first < 0) first = k;
        last = k;
      }
    }
    // packed for the kernel's 4-wide walk: the band starts on a multiple of four bins and covers whole groups of four, the
    // extra leading / trailing weights are zero (start = first bin of the walk, len = groups of four, off = multiple of four)
    off[m] = (int)wts.size();
    if (first >= 0) {
      const int first4 = first & ~3;
      const int groups = (last - first4) / 4 + 1;
      start[m] = first4;
      len[m] = groups;
      for (int k = first4; k < first4 + 4 * groups; ++k) {
        const double fm = mel(nyq * k / (bins - 1));
        const double w = (k >= first && k <= last) ? std::max(0.0, std::min((fm - lo) / (ce - lo), (up - fm) / (up - ce))) : 0.0;
        wts.push_back((float)w);
      }
    }
  }
  // mfccs_from_log_mel_spectrograms: DCT-II (unnormalised, x2) * rsqrt(2 M), first F coefficients.
  const int F = h->features;
  std::vector<float> dct((size_t)M * F);
  for (int m = 0; m < M; ++m)
    for (int k = 0; k < F; ++k)
      dct[(size_t)m * F + k] = (float)(2.0 * cos(M_PI * k * (2.0 * m + 1.0) / (2.0 * M)) / sqrt(2.0 * M));
  // constant block of the front-end kernel (tcr_mfcc.h): tw | mel weights | tw2 | window, sections padded to 16 bytes
  {
    std::vector<float> blk;
    auto pad4 = [&]() { while (blk.size() % 4) blk.push_back(0.f); };
    for (auto& v : tw) { blk.push_back(v.x); blk.push_back(v.y); }
    pad4();
    h->c_melw = (int)blk.size();
    blk.insert(blk.end(), wts.begin(), wts.end());
    pad4();
    h->c_smem = (int)blk.size();                   // everything above is staged in shared memory
    h->c_tw2 = (int)blk.size();
    for (auto& v : tw2) { blk.push_back(v.x); blk.push_back(v.y); }
    pad4();
    h->c_win = (int)blk.size();
    blk.insert(blk.end(), win.begin(), win.end());
    pad4();
    if (fft == 1024 && M == 64) {
      // frame-pair kernel (tcr_mfcc_pair.cu), one contiguous section staged by a single TMA copy:
      //   W_512^(n2 k1), k1 < 16 rows of n2 < 32 | segment weights | DCT entries in lane order
      h->c_twa = (int)blk.size();
      for (int k1 = 0; k1 < 16; ++k1)
        for (int n2 = 0; n2 < 32; ++n2) {
          const double a = -2.0 * M_PI * (double)(n2 * k1) / 512.0;
          blk.push_back((float)cos(a));
          blk.push_back((float)sin(a));
        }
      // Mel by SEGMENTS: the band edges cut the bins into M + 1 runs; a bin of run j rises in band j with weight
      // u = (mel - edge_j) / (edge_j+1 - edge_j) and falls in band j - 1 with 1 - u, so with R_j = sum u P and S_j = sum P over
      // the run, band_m = R_m + (S_m+1 - R_m+1): every bin and one weight are read once (167 groups of four instead of 282).
      // A run is walked in aligned groups of four; bins of the groups that belong to a neighbouring run carry the marker -1.
      std::vector<int> seg_of(bins, -1);
      std::vector<double> up(bins, 0.0);
      for (int k = 1; k < bins; ++k) {
        const double fm = mel(nyq * k / (bins - 1));
        for (int j = 0; j <= M; ++j)
          if (fm >= edges[j] && fm < edges[j + 1]) {
            seg_of[k] = j;
            up[k] = (fm - edges[j]) / (edges[j + 1] - edges[j]);
            break;
          }
      }
      const int segw0 = (int)blk.size();
      std::vector<int> seg_meta(3 * 32, 0);           // [pass][lane]: start/4 | groups << 8 | (offset/4 from the section start) << 16
      for (int j = 0; j <= M; ++j) {
        int first = -1, last = -1;
        for (int k = 1; k < bins; ++k)
          if (seg_of[k] == j) {
            if (first < 0) first = k;
            last = k;
          }
        if (first < 0) continue;
        const int first4 = first & ~3, groups = (last - first4) / 4 + 1;
        const int off4 = ((int)blk.size() - segw0) / 4;
        for (int k = first4; k < first4 + 4 * groups; ++k) blk.push_back((k < bins && seg_of[k] == j) ? (float)up[k] : -1.0f);
        // pass 0: lane i walks run i (i < 32); pass 1: lane i walks run 64 - i; pass 2: lane 0 walks run 32
        const int slot = j < 32 ? j : (j > 32 ? 32 + (64 - j) : 64);
        seg_meta[slot] = (first4 >> 2) | (groups << 8) | (off4 << 16);
      }
      h->pair_segw_len = (int)blk.size() - segw0;
      // DCT entries in the order the kernel's lanes use them: lane (q, g) = (lane / 8, lane % 8), rows q + 4 i, columns g + 8 j
      if (F == 40) {
        for (int i = 0; i < 8; ++i)
          for (int j = 0; j < 5; ++j)
            for (int lane = 0; lane < 32; ++lane) blk.push_back(dct[(size_t)((lane >> 3) + 4 * i) * F + (lane & 7) + 8 * j]);
        h->pair_dct_len = 8 * 5 * 32;
      }
      pad4();
      TCR_TRY(dev_upload(h, &h->d_seg_meta, seg_meta));
    }
    TCR_TRY(dev_upload(h, &h->d_fe_consts, blk));
  }
  TCR_TRY(dev_upload(h, &h->d_mel_start, start));
  TCR_TRY(dev_upload(h, &h->d_mel_len, len));
  TCR_TRY(dev_upload(h, &h->d_mel_off, off));
  TCR_TRY(dev_upload(h, &h->d_dct, dct));
  return TCR_OK;
}

static MfccArgs mfcc_args(const tcr_handle* h, const void* wav, int pcm16, float* feat) {
  MfccArgs a;
  a.wav = wav;
  a.pcm16 = pcm16;
  a.feat = feat;
  a.clip = h->cfg.clip_samples;
  a.window = h->cfg.window_size_samples;
  a.stride = h->cfg.window_stride_samples;
  a.frames = h->frames;
  a.features = h->features;
  a.mel_bins = h->cfg.num_mel_bins;
  a.fpb = h->fpb;
  a.warps = h->fwarps;
  a.magnitude = h->cfg.feature_kind == TCR_FEATURE_LOG_MEL;
  a.use_dct = h->cfg.feature_kind == TCR_FEATURE_MFCC;
  a.consts = h->d_fe_consts;
  a.c_tw2 = h->c_tw2; a.c_melw = h->c_melw; a.c_win = h->c_win; a.c_smem = h->c_smem;
  a.c_twa = h->c_twa;
  a.seg_meta = h->d_seg_meta; a.segw_len = h->pair_segw_len; a.dct_len = h->pair_dct_len;
  a.n_utts = 0;
  a.mel_start = h->d_mel_start;
  a.mel_len = h->d_mel_len;
  a.mel_off = h->d_mel_off;
  a.dct = h->d_dct;
  return a;
}

// ------------------------------------------------------------------------------------------------
// layer plan (audio_nets/tc_resnet.py:6-70) and variable table (tf.trainable_variables() order)
// ------------------------------------------------------------------------------------------------
static void same_padding(int len, int k, int s, int* out, int* left) {
  *out = (len + s - 1) / s;
  int total = std::max((*out - 1) * s + k - len, 0);
  *left = total / 2;
}

static void add_desc(tcr_handle* h, const std::string& name, int kind, int rank, const int* shape, int64_t off, int64_t numel) {
  tcr_param_desc d;
  memset(&d, 0, sizeof(d));
  snprintf(d.name, sizeof(d.name), "%s", name.c_str());
  d.kind = kind;
  d.rank = rank;
  for (int i = 0; i < rank; ++i) d.shape[i] = shape[i];
  d.offset = off;
  d.numel = numel;
  h->table.push_back(d);
}

static int build_plan(tcr_handle* h) {
  const tcr_config& c = h->cfg;
  std::vector<int> plan;
  if (c.model == TCR_MODEL_TCRESNET8) {
    h->scope = "TCResNet8";
    plan = {16, 24, 32, 48};
  } else if (c.model == TCR_MODEL_TCRESNET14) {
    h->scope = "TCResNet14";
    plan = {16, 24, 24, 32, 32, 48, 48};
  } else {
    return fail(TCR_ERR_INVALID, "unknown model %d (expected 8 or 14)", c.model);
  }
  for (int& x : plan) {
    x = (int)((double)x * (double)c.width_multiplier);   // int(x * width_multiplier), tc_resnet.py:60
    if (x <= 0 || x % 4 != 0)
      return fail(TCR_ERR_UNSUPPORTED, "channel count %d (width_multiplier %g) is not a positive multiple of 4", x,
                  c.width_multiplier);
  }
  if (h->features % 4 != 0) return fail(TCR_ERR_UNSUPPORTED, "feature count %d is not a multiple of 4", h->features);
  auto mk = [&](const std::string& name, int cin, int cout, int k, int s, int t, int relu) {
    ConvPlan cv;
    cv.name = name;
    cv.cin = cin;
    cv.cout = cout;
    cv.k = k;
    cv.stride = s;
    cv.t_in = t;
    cv.relu = relu;
    same_padding(t, k, s, &cv.t_out, &cv.pad_left);
    h->convs.push_back(cv);
    return (int)h->convs.size() - 1;
  };
  mk("conv0", h->features, plan[0], 3, 1, h->frames, 1);
  int ch = plan[0], t = h->convs[0].t_out;
  for (size_t i = 1; i < plan.size(); ++i) {
    const int n = plan[i];
    const std::string b = "block" + std::to_string(i - 1);
    BlockPlan bp;
    int stride = 1;
    if (n != ch) {
      stride = 2;
      bp.down = mk(b + "/down", ch, n, 1, 2, t, 1);
    }
    bp.a = mk(b + "/conv" + std::to_string(i - 1) + "_0", ch, n, 9, stride, t, 1);
    bp.b = mk(b + "/conv" + std::to_string(i - 1) + "_1", n, n, 9, 1, h->convs[bp.a].t_out, 0);
    ch = n;
    t = h->convs[bp.b].t_out;
    bp.c = ch;
    bp.t = t;
    h->blocks.push_back(bp);
  }
  if ((int)h->convs.size() > kMaxConvs) return fail(TCR_ERR_UNSUPPORTED, "too many conv layers");
  h->c_last = ch;
  h->t_last = t;
  // variable table: per conv weights, beta, gamma (creation order of slim.conv2d + slim.batch_norm), then fc, fc2
  int64_t off = 0, moff = 0;
  for (auto& cv : h->convs) {
    const std::string p = h->scope + "/" + cv.name;
    int shp[4] = {cv.k, 1, cv.cin, cv.cout};
    cv.w_off = off;
    add_desc(h, p + "/weights", TCR_KIND_WEIGHT, 4, shp, off, cv.wnumel());
    off += cv.wnumel();
    int s1[1] = {cv.cout};
    cv.beta_off = off;
    add_desc(h, p + "/BatchNorm/beta", TCR_KIND_BETA, 1, s1, off, cv.cout);
    off += cv.cout;
    cv.gamma_off = off;
    add_desc(h, p + "/BatchNorm/gamma", TCR_KIND_GAMMA, 1, s1, off, cv.cout);
    off += cv.cout;
  }
  {
    int shp[4] = {1, 1, h->c_last, c.num_classes};
    h->fc_off = off;
    add_desc(h, h->scope + "/fc/weights", TCR_KIND_WEIGHT, 4, shp, off, (int64_t)h->c_last * c.num_classes);
    off += (int64_t)h->c_last * c.num_classes;
    int shp2[4] = {1, 1, h->c_last, 2};
    h->fc2_off = off;
    add_desc(h, h->scope + "/fc2/weights", TCR_KIND_WEIGHT, 4, shp2, off, (int64_t)h->c_last * 2);
    off += (int64_t)h->c_last * 2;
  }
  h->n_train = off;
  for (auto& cv : h->convs) {
    const std::string p = h->scope + "/" + cv.name + "/BatchNorm/";
    int s1[1] = {cv.cout};
    cv.mm_off = moff;
    add_desc(h, p + "moving_mean", TCR_KIND_MOVING_MEAN, 1, s1, moff, cv.cout);
    moff += cv.cout;
    cv.mv_off = moff;
    add_desc(h, p + "moving_variance", TCR_KIND_MOVING_VAR, 1, s1, moff, cv.cout);
    moff += cv.cout;
  }
  h->n_moving = moff;
  return TCR_OK;
}

extern "C" int tcr_create(const tcr_config* cfg, tcr_handle** out) {
  if (!cfg || !out) return fail(TCR_ERR_INVALID, "cfg/out is NULL");
  *out = nullptr;
  if (cfg->max_batch <= 0) return fail(TCR_ERR_INVALID, "max_batch must be positive");
  if (cfg->window_size_samples <= 0 || cfg->window_stride_samples <= 0 || cfg->clip_samples < cfg->window_size_samples)
    return fail(TCR_ERR_INVALID, "bad window/stride/clip (%d/%d/%d)", cfg->window_size_samples,
                cfg->window_stride_samples, cfg->clip_samples);
  if (cfg->window_size_samples % 4 || cfg->window_stride_samples % 4 || cfg->clip_samples % 4)
    return fail(TCR_ERR_UNSUPPORTED, "window, stride and clip lengths must be multiples of 4 samples (16-byte TMA rows)");
  if (cfg->num_mel_bins <= 0 || cfg->num_mel_bins > 128 || cfg->num_mfccs <= 0 || cfg->num_mfccs > cfg->num_mel_bins)
    return fail(TCR_ERR_INVALID, "bad num_mel_bins/num_mfccs (%d/%d)", cfg->num_mel_bins, cfg->num_mfccs);
  if (cfg->feature_kind != TCR_FEATURE_MFCC && cfg->feature_kind != TCR_FEATURE_LOG_MEL)
    return fail(TCR_ERR_INVALID, "bad feature_kind %d", cfg->feature_kind);
  if (!(cfg->dropout_keep_prob > 0.f && cfg->dropout_keep_prob <= 1.f))
    return fail(TCR_ERR_INVALID, "dropout_keep_prob must be in (0,1]");
  if (cfg->num_classes <= 0 || cfg->num_classes > kMaxClasses)
    return fail(TCR_ERR_UNSUPPORTED, "num_classes must be in [1,%d]", kMaxClasses);
  tcr_handle* h = new tcr_handle();
  h->cfg = *cfg;
  auto bail = [&](int rc) {
    tcr_destroy(h);
    return rc;
  };
  if (cudaSetDevice(cfg->device) != cudaSuccess) return bail(fail(TCR_ERR_CUDA, "cudaSetDevice(%d) failed", cfg->device));
#ifndef TCR_EMU
  if (cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, cfg->device) != cudaSuccess || h->sms < 1) h->sms = 1;
#endif
  h->frames = 1 + (cfg->clip_samples - cfg->window_size_samples) / cfg->window_stride_samples;
  h->features = cfg->feature_kind == TCR_FEATURE_MFCC ? cfg->num_mfccs : cfg->num_mel_bins;
  h->fft = next_pow2(cfg->window_size_samples);
  if (h->fft < 128 || h->fft > 2048) return bail(fail(TCR_ERR_UNSUPPORTED, "fft length %d outside [128, 2048]", h->fft));
  // frames per CTA: a divisor-ish of T in [4, 8] so that chunks are balanced (49 -> 7, 98 -> 7)
  h->fpb = 8;
  {
    int best = 8, best_waste = 1 << 30;
    for (int f = 8; f >= 4; --f) {
      const int chunks = (h->frames + f - 1) / f;
      const int waste = chunks * f - h->frames;
      if (waste < best_waste) {
        best_waste = waste;
        best = f;
      }
    }
    h->fpb = std::min(best, h->frames);
  }
  h->fwarps = std::min(h->fpb, 7);
  if (const char* e = getenv("TCR_MFCC_FPB")) {                  // tuning knob: frames per CTA[,warps per CTA]
    int f = 0, w = 0;
    const int got = sscanf(e, "%d,%d", &f, &w);
    if (got >= 1 && f >= 1) { h->fpb = std::min(f, h->frames); h->fwarps = std::min(h->fpb, 7); }
    if (got >= 2 && w >= 1) h->fwarps = std::min(std::min(w, 7), h->fpb);
  }
  if (const char* e = getenv("TCR_MFCC_PAIR")) {                 // frame-pair kernel: 0 | 1 | frames per work item (even, <= 10)
    int f = 0, w = 0;
    const int got = sscanf(e, "%d,%d", &f, &w);
    h->mfcc_pair = got >= 1 && f >= 1;
    if (got >= 1 && f >= 2) { h->pair_fpb = std::min(f & ~1, 10); h->pair_warps = h->pair_fpb / 2; }   // one warp per frame pair
    (void)w;
  }
  int rc = build_frontend_tables(h);
  if (rc) return bail(rc);
  rc = build_plan(h);
  if (rc) return bail(rc);
  rc = net_alloc_workspace(h);
  if (rc) return bail(fail(rc, "workspace allocation failed: %s", g_err));
  *out = h;
  return TCR_OK;
}

static void hostfeed_destroy(tcr_handle* h);
static void frontend_ahead_destroy(tcr_handle* h);

extern "C" int tcr_destroy(tcr_handle* h) {
  if (!h) return TCR_OK;
  hostfeed_destroy(h);
  frontend_ahead_destroy(h);
  resident_destroy(h);
  comm_destroy(h);
  for (void* p : h->allocs) cudaFree(p);
  if (h->h_hyper) cudaFreeHost(h->h_hyper);
  delete h;
  return TCR_OK;
}

extern "C" int tcr_get_info(const tcr_handle* h, tcr_info* out) {
  if (!h || !out) return fail(TCR_ERR_INVALID, "NULL argument");
  memset(out, 0, sizeof(*out));
  out->abi_version = TCR_ABI_VERSION;
  out->frames = h->frames;
  out->features = h->features;
  out->fft_length = h->fft;
  out->num_conv_layers = (int)h->convs.size();
  out->num_blocks = (int)h->blocks.size();
  out->last_channels = h->c_last;
  out->last_frames = h->t_last;
  out->num_trainable = h->n_train;
  out->num_moving = h->n_moving;
  int64_t fl = 0;
  for (const auto& cv : h->convs) fl += 2ll * cv.t_out * cv.k * cv.cin * cv.cout;
  fl += 2ll * h->c_last * h->cfg.num_classes + 2ll * h->c_last * 2;
  out->forward_flops_per_utt = fl;
  out->workspace_bytes = h->workspace_bytes;
  return TCR_OK;
}

extern "C" int tcr_param_table(const tcr_handle* h, const tcr_param_desc** descs, int32_t* count) {
  if (!h || !descs || !count) return fail(TCR_ERR_INVALID, "NULL argument");
  *descs = h->table.data();
  *count = (int32_t)h->table.size();
  return TCR_OK;
}

extern "C" int tcr_init_variables(tcr_handle* h, float* params, float* slots, float* moving, uint64_t seed, tcr_stream stream) {
  if (!h) return fail(TCR_ERR_INVALID, "NULL handle");
  std::mt19937_64 rng(seed);
  std::vector<float> p((size_t)h->n_train, 0.f), mv((size_t)h->n_moving, 0.f);
  for (const auto& d : h->table) {
    if (d.kind == TCR_KIND_WEIGHT) {
      const double fan_in = (double)d.shape[0] * d.shape[1] * d.shape[2], fan_out = (double)d.shape[0] * d.shape[1] * d.shape[3];
      const double lim = sqrt(6.0 / (fan_in + fan_out));   // slim xavier_initializer(uniform=True)
      std::uniform_real_distribution<double> u(-lim, lim);
      for (int64_t i = 0; i < d.numel; ++i) p[(size_t)(d.offset + i)] = (float)u(rng);
    } else if (d.kind == TCR_KIND_GAMMA) {
      for (int64_t i = 0; i < d.numel; ++i) p[(size_t)(d.offset + i)] = 1.f;
    } else if (d.kind == TCR_KIND_MOVING_VAR) {
      for (int64_t i = 0; i < d.numel; ++i) mv[(size_t)(d.offset + i)] = 1.f;
    }
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (params) TCR_CUDA(cudaMemcpyAsync(params, p.data(), p.size() * 4, cudaMemcpyHostToDevice, s));
  if (moving) TCR_CUDA(cudaMemcpyAsync(moving, mv.data(), mv.size() * 4, cudaMemcpyHostToDevice, s));
  if (slots) TCR_CUDA(cudaMemsetAsync(slots, 0, (size_t)h->n_train * 4, s));
  TCR_CUDA(cudaStreamSynchronize(s));   // host staging buffers go out of scope
  return TCR_OK;
}

static int check_n(const tcr_handle* h, int n) {
  if (n <= 0) return fail(TCR_ERR_INVALID, "n must be positive (got %d)", n);
  if (n > h->cfg.max_batch) return fail(TCR_ERR_INVALID, "n=%d exceeds max_batch=%d", n, h->cfg.max_batch);
  return TCR_OK;
}

static int mfcc_run(tcr_handle* h, const void* wav, int pcm16, float* features, int32_t n, tcr_stream stream) {
  if (!h || !wav || !features) return fail(TCR_ERR_INVALID, "NULL argument");
  TCR_TRY(check_n(h, n));
  if (((uintptr_t)wav & 15) != 0) return fail(TCR_ERR_INVALID, "wav must be 16-byte aligned (TMA bulk copy)");
  if (pcm16 && (h->cfg.window_size_samples % 8 || h->cfg.window_stride_samples % 8 || h->cfg.clip_samples % 8))
    return fail(TCR_ERR_UNSUPPORTED, "int16 input needs window, stride and clip lengths that are multiples of 8 samples");
  MfccArgs a = mfcc_args(h, wav, pcm16, features);
  bool launched = false;
  if (h->mfcc_pair) {                                             // two frames per warp (tcr_mfcc_pair.cu) where the shape allows
    MfccArgs b = a;
    b.fpb = h->pair_fpb;
    b.warps = h->pair_warps;
    if (mfcc_pair_supported(b, h->fft)) {
      if (mfcc_pair_launch(b, n, 3 * h->sms, (cudaStream_t)stream) != 0) return fail(TCR_ERR_CUDA, "mfcc (frame pairs) launch configuration failed");
      launched = true;
    }
  }
  if (!launched && mfcc_launch(a, n, h->fft, (cudaStream_t)stream) != 0) return fail(TCR_ERR_CUDA, "mfcc launch configuration failed");
  TCR_CUDA(cudaGetLastError());
  return TCR_OK;
}
extern "C" int tcr_mfcc_forward(tcr_handle* h, const float* wav, float* features, int32_t n, tcr_stream stream) {
  pdl_chain_reset();
  return mfcc_run(h, wav, 0, features, n, stream);
}
extern "C" int tcr_mfcc_forward_pcm16(tcr_handle* h, const int16_t* pcm, float* features, int32_t n, tcr_stream stream) {
  pdl_chain_reset();
  return mfcc_run(h, pcm, 1, features, n, stream);
}

extern "C" int tcr_augment_pcm16(tcr_handle* h, const int16_t* pcm, int64_t pcm_stride, const tcr_augment_clip* clips,
                                 const float* background, float* wav_out, int32_t n, tcr_stream stream) {
  pdl_chain_reset();
  if (!h || !pcm || !clips || !wav_out) return fail(TCR_ERR_INVALID, "NULL argument");
  TCR_TRY(check_n(h, n));
  if (pcm_stride < 1) return fail(TCR_ERR_INVALID, "pcm_stride must be positive");
  if (((uintptr_t)wav_out & 15) != 0) return fail(TCR_ERR_INVALID, "wav_out must be 16-byte aligned");
  augment_launch(pcm, pcm_stride, clips, background, h->background_samples, wav_out, h->cfg.clip_samples, n, (cudaStream_t)stream);
  TCR_CUDA(cudaGetLastError());
  return TCR_OK;
}

extern "C" int tcr_set_background_samples(tcr_handle* h, int64_t samples) {
  if (!h || samples < 0) return fail(TCR_ERR_INVALID, "bad background length");
  h->background_samples = samples;
  return TCR_OK;
}

extern "C" int tcr_forward(tcr_handle* h, const float* input, int32_t input_is_features, const float* params,
                           const float* moving, int32_t n, int32_t is_training, uint64_t dropout_seed,
                           const float* dropout_mask, const float* onehot, float weight_decay, float* logits,
                           float* probs, float* losses, tcr_stream stream) {
  pdl_chain_reset();
  if (!h || !input || !params) return fail(TCR_ERR_INVALID, "NULL argument");
  if (!is_training && !moving) return fail(TCR_ERR_INVALID, "eval-mode forward needs the moving statistics");
  TCR_TRY(check_n(h, n));
  cudaStream_t s = (cudaStream_t)stream;
  const float* feat = input;
  if (input_is_features != TCR_INPUT_FEATURES) {
    if (input_is_features != TCR_INPUT_WAV_F32 && input_is_features != TCR_INPUT_WAV_PCM16) return fail(TCR_ERR_INVALID, "unknown input kind %d", input_is_features);
    TCR_TRY(mfcc_run(h, input, input_is_features == TCR_INPUT_WAV_PCM16, h->d_feat, n, stream));
    feat = h->d_feat;
    h->feat_last = h->d_feat;
  }
  int rc = net_forward(h, feat, params, moving, n, is_training != 0, dropout_seed, dropout_mask, onehot, weight_decay,
                       logits, probs, losses, /*backward=*/false, s);
  if (rc) return fail(rc, "forward launch failed: %s", g_err);
  TCR_CUDA(cudaGetLastError());
  h->last_n = n;
  return TCR_OK;
}

extern "C" int tcr_eval_accumulate(tcr_handle* h, const float* scores, const float* onehot, int32_t n, int32_t topk, int64_t* counts,
                                   tcr_stream stream) {
  if (!h || !scores || !onehot || !counts) return fail(TCR_ERR_INVALID, "NULL argument");
  if (n <= 0) return fail(TCR_ERR_INVALID, "n must be positive (got %d)", n);
  if (topk < 1) return fail(TCR_ERR_INVALID, "topk must be at least 1");
  eval_accumulate_launch(scores, onehot, n, h->cfg.num_classes, topk, counts, (cudaStream_t)stream);
  TCR_CUDA(cudaGetLastError());
  return TCR_OK;
}

// Front-end running ahead (tcr_step_args::input_resident): lazily created low-priority stream, second feature buffer, events.
static int frontend_ahead_get(tcr_handle* h) {
  if (h->fe_stream) return TCR_OK;
#ifndef TCR_EMU
  int lo = 0, hi = 0;
  TCR_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));          // lo = numerically greatest = lowest priority
  cudaStream_t st = nullptr;
  TCR_CUDA(cudaStreamCreateWithPriority(&st, cudaStreamNonBlocking, lo));
  for (int b = 0; b < 2; ++b) {      // its own two feature buffers: h->d_feat stays with the calls that are ordered on their stream
    void* p = nullptr;
    TCR_CUDA(cudaMalloc(&p, (size_t)h->cfg.max_batch * h->frames * h->features * sizeof(float)));
    h->allocs.push_back(p);
    h->workspace_bytes += (int64_t)h->cfg.max_batch * h->frames * h->features * (int64_t)sizeof(float);
    h->fe_feat[b] = (float*)p;
  }
  for (int b = 0; b < 2; ++b) {
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    TCR_CUDA(cudaEventCreateWithFlags(&e0, cudaEventDisableTiming));
    TCR_CUDA(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
    h->fe_ready[b] = e0;
    h->fe_free[b] = e1;
  }
  {
    cudaEvent_t g = nullptr;
    TCR_CUDA(cudaEventCreateWithFlags(&g, cudaEventDisableTiming));
    h->fe_gate = g;
  }
  h->fe_stream = st;
#endif
  return TCR_OK;
}
static void frontend_ahead_destroy(tcr_handle* h) {
#ifndef TCR_EMU
  if (!h->fe_stream) return;
  cudaStreamSynchronize((cudaStream_t)h->fe_stream);
  for (int b = 0; b < 2; ++b) {
    if (h->fe_ready[b]) cudaEventDestroy((cudaEvent_t)h->fe_ready[b]);
    if (h->fe_free[b]) cudaEventDestroy((cudaEvent_t)h->fe_free[b]);
  }
  if (h->fe_gate) cudaEventDestroy((cudaEvent_t)h->fe_gate);
  cudaStreamDestroy((cudaStream_t)h->fe_stream);
  h->fe_stream = nullptr;
#else
  (void)h;
#endif
}

// The state buffers each update rule reads and writes (tcr_step_args::optimizer).
static int check_optimizer(const tcr_step_args* a) {
  switch (a->optimizer) {
    case TCR_OPT_MOMENTUM: break;
    case TCR_OPT_ADAM:
      if (a->apply_update && (!a->slots2 || !a->opt_scalars)) return fail(TCR_ERR_INVALID, "TCR_OPT_ADAM needs slots2 (v) and opt_scalars (beta powers)");
      break;
    case TCR_OPT_RMSPROP:
      if (a->apply_update && !a->slots2) return fail(TCR_ERR_INVALID, "TCR_OPT_RMSPROP needs slots2 (mom)");
      break;
    default: return fail(TCR_ERR_INVALID, "unknown optimizer %d", a->optimizer);
  }
  return TCR_OK;
}

// input_event: what the front-end has to wait for when it runs ahead (the host feed's H2D copy), or null
static int train_step_impl(tcr_handle* h, const tcr_step_args* a, tcr_stream stream, void* input_event) {
  pdl_chain_reset();
  if (!h || !a || !a->input || !a->onehot || !a->params) return fail(TCR_ERR_INVALID, "NULL argument");
  if (a->apply_update && (!a->slots || !a->moving)) return fail(TCR_ERR_INVALID, "apply_update needs slots and moving");
  TCR_TRY(check_optimizer(a));
  TCR_TRY(check_n(h, a->n));
  cudaStream_t s = (cudaStream_t)stream;
  const float* feat = a->input;
  int fe_buf = -1;                   // feature buffer of a front-end that ran ahead
  if (a->input_is_features != TCR_INPUT_FEATURES) {
    if (a->input_is_features != TCR_INPUT_WAV_F32 && a->input_is_features != TCR_INPUT_WAV_PCM16) return fail(TCR_ERR_INVALID, "unknown input kind %d", a->input_is_features);
    tcr_stream fs = stream;          // stream of the front-end kernels
    float* featbuf = h->d_feat;
#ifndef TCR_EMU
    if (a->input_resident) {
      TCR_TRY(frontend_ahead_get(h));
      fe_buf = (int)(h->fe_count++ & 1);
      cudaStream_t f = (cudaStream_t)h->fe_stream;
      if (input_event) TCR_CUDA(cudaStreamWaitEvent(f, (cudaEvent_t)input_event, 0));
      if (h->fe_count > 2) TCR_CUDA(cudaStreamWaitEvent(f, (cudaEvent_t)h->fe_free[fe_buf], 0));   // the step two calls back has read it
      // not before the previous step's weight gradients are launched-and-done: the front-end then shares the GPU with the small,
      // latency-bound tail kernels (grad_finalize, update and its cross-GPU arrival wait) instead of time-slicing with the FMA-bound ones
      if (h->fe_gate_valid) TCR_CUDA(cudaStreamWaitEvent(f, (cudaEvent_t)h->fe_gate, 0));
      fs = (tcr_stream)f;
      featbuf = h->fe_feat[fe_buf];
    }
#endif
    h->feat_last = featbuf;
    if (a->clips) {                  // device input stage first: int16 clips + per-clip draws -> fp32 wav (tcr_augment.cu)
      if (a->input_is_features != TCR_INPUT_WAV_PCM16) return fail(TCR_ERR_INVALID, "clips need TCR_INPUT_WAV_PCM16 input");
      const int64_t stride = a->pcm_stride > 0 ? a->pcm_stride : h->cfg.clip_samples;
      float*& aug = fe_buf >= 0 ? h->fe_aug : h->d_aug;       // the ahead path decodes into its own buffer
      if (!aug) {
        void* p = nullptr;
        TCR_CUDA(cudaMalloc(&p, (size_t)h->cfg.max_batch * h->cfg.clip_samples * sizeof(float)));
        h->allocs.push_back(p);
        aug = (float*)p;
      }
      augment_launch((const int16_t*)a->input, stride, a->clips, a->background, h->background_samples, aug, h->cfg.clip_samples, a->n,
                     (cudaStream_t)fs);
      TCR_TRY(mfcc_run(h, aug, 0, featbuf, a->n, fs));
    } else {
      TCR_TRY(mfcc_run(h, a->input, a->input_is_features == TCR_INPUT_WAV_PCM16, featbuf, a->n, fs));
    }
    feat = featbuf;
#ifndef TCR_EMU
    if (fe_buf >= 0) {
      TCR_CUDA(cudaEventRecord((cudaEvent_t)h->fe_ready[fe_buf], (cudaStream_t)h->fe_stream));
      TCR_CUDA(cudaStreamWaitEvent(s, (cudaEvent_t)h->fe_ready[fe_buf], 0));
      pdl_chain_reset();             // the next launch is the first one of this call on `stream`
    }
#endif
  }
  const int resident = resident_mode(h);
  if (resident < 1) net_weight_transpose(h, a->params, s);      // the resident forward kernel writes the transposed banks itself
  int rc = resident >= 1 ? resident_forward(h, feat, a, s)
                               : net_forward(h, feat, a->params, nullptr, a->n, true, a->dropout_seed, a->dropout_mask, a->onehot,
                                             a->weight_decay, a->logits, a->probs, nullptr, /*backward=*/true, s);
  if (rc) return fail(rc, "forward launch failed: %s", g_err);
  if (resident < 2) {               // mode 2: net_update runs the resident backward kernel instead
    rc = net_backward(h, feat, a->params, a->n, s);
    if (rc) return fail(rc, "backward launch failed: %s", g_err);
  } else if (resident == 3) {       // backward-data chain as one resident kernel, then the grouped weight-gradient launch
    rc = resident_backward_data(h, feat, a, s);
    if (!rc) rc = net_weight_gradients(h, feat, a->n, s);
    if (rc) return fail(rc, "backward launch failed: %s", g_err);
  }
#ifndef TCR_EMU
  if (h->fe_gate) {                   // the gate of the NEXT step's front-end (see above)
    TCR_CUDA(cudaEventRecord((cudaEvent_t)h->fe_gate, s));
    h->fe_gate_valid = 1;
  }
#endif
  rc = net_update(h, feat, a, s);
  if (rc) return fail(rc, "update launch failed: %s", g_err);
  TCR_CUDA(cudaGetLastError());
#ifndef TCR_EMU
  if (fe_buf >= 0) TCR_CUDA(cudaEventRecord((cudaEvent_t)h->fe_free[fe_buf], s));
#endif
  h->last_n = a->n;
  return TCR_OK;
}

extern "C" int tcr_train_step(tcr_handle* h, const tcr_step_args* a, tcr_stream stream) { return train_step_impl(h, a, stream, nullptr); }

// ------------------------------------------------------------------------------------------------
// Host-buffer training step: the `feed_dict` / input-pipeline side of session.run(train_op)
// (helper/trainer.py:312-321, datasets/data_wrapper_base.py:100-108 prefetch).  Pinned host batch -> H2D on a private
// copy stream into one of kFeedDepth staging slots -> the step on the caller's stream -> D2H of the two losses.
// Submission never waits for the step it submits: the losses handed back are those of the step `lag` calls earlier,
// so the copy of batch i+1 overlaps the compute of batch i and kernel launches run ahead of the GPU.
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int kFeedDepth = 3;
struct HostSlot {
  void* d_in = nullptr; float* d_hot = nullptr; float* d_loss = nullptr; float* h_loss = nullptr;
  tcr_augment_clip* d_clips = nullptr;
  cudaEvent_t ready = nullptr, consumed = nullptr, done = nullptr;
};
struct HostFeedState {
  HostSlot slot[kFeedDepth];
  cudaStream_t copy = nullptr;
  int64_t submitted = 0, collected = 0;
};
}  // namespace

static void hostfeed_destroy(tcr_handle* h) {
  HostFeedState* f = (HostFeedState*)h->hostfeed;
  if (!f) return;
  for (auto& s : f->slot) {
    if (s.d_in) cudaFree(s.d_in);
    if (s.d_hot) cudaFree(s.d_hot);
    if (s.d_clips) cudaFree(s.d_clips);
    if (s.d_loss) cudaFree(s.d_loss);
    if (s.h_loss) cudaFreeHost(s.h_loss);
    if (s.ready) cudaEventDestroy(s.ready);
    if (s.consumed) cudaEventDestroy(s.consumed);
    if (s.done) cudaEventDestroy(s.done);
  }
  if (f->copy) cudaStreamDestroy(f->copy);
  delete f;
  h->hostfeed = nullptr;
}

static int hostfeed_get(tcr_handle* h, HostFeedState** out) {
  if (!h->hostfeed) {
    HostFeedState* f = new HostFeedState();
    h->hostfeed = f;
    TCR_CUDA(cudaStreamCreateWithFlags(&f->copy, cudaStreamNonBlocking));
    const size_t in_bytes = (size_t)h->cfg.max_batch * std::max((size_t)h->cfg.clip_samples, (size_t)h->frames * h->features) * 4;
    for (auto& s : f->slot) {
      TCR_CUDA(cudaMalloc(&s.d_in, in_bytes));
      TCR_CUDA(cudaMalloc((void**)&s.d_hot, (size_t)h->cfg.max_batch * h->cfg.num_classes * 4));
      TCR_CUDA(cudaMalloc((void**)&s.d_clips, (size_t)h->cfg.max_batch * sizeof(tcr_augment_clip)));
      TCR_CUDA(cudaMalloc((void**)&s.d_loss, 2 * sizeof(float)));
      TCR_CUDA(cudaMallocHost((void**)&s.h_loss, 2 * sizeof(float)));
      TCR_CUDA(cudaEventCreateWithFlags(&s.ready, cudaEventDisableTiming));
      TCR_CUDA(cudaEventCreateWithFlags(&s.consumed, cudaEventDisableTiming));
      TCR_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
    }
  }
  *out = (HostFeedState*)h->hostfeed;
  return TCR_OK;
}

static int hostfeed_collect(HostFeedState* f, float* losses_out, int64_t* losses_step) {
  HostSlot& s = f->slot[f->collected % kFeedDepth];
  TCR_CUDA(cudaEventSynchronize(s.done));
  if (losses_out) { losses_out[0] = s.h_loss[0]; losses_out[1] = s.h_loss[1]; }
  if (losses_step) *losses_step = f->collected;
  ++f->collected;
  return TCR_OK;
}

extern "C" int tcr_train_step_host(tcr_handle* h, const tcr_step_args* a, int32_t lag, tcr_stream stream, float* losses_out,
                                   int64_t* losses_step) {
  if (!h || !a || !a->input || !a->onehot || !a->params) return fail(TCR_ERR_INVALID, "NULL argument");
  if (lag < 0 || lag >= kFeedDepth) return fail(TCR_ERR_INVALID, "lag must be in [0, %d]", kFeedDepth - 1);
  TCR_TRY(check_optimizer(a));       // before anything is queued; the struct copy below carries the optimizer fields to the step
  TCR_TRY(check_n(h, a->n));
  HostFeedState* f = nullptr;
  TCR_TRY(hostfeed_get(h, &f));
  if (losses_step) *losses_step = -1;
  cudaStream_t s = (cudaStream_t)stream;
  HostSlot& sl = f->slot[f->submitted % kFeedDepth];
  size_t in_bytes;
  switch (a->input_is_features) {
    case TCR_INPUT_WAV_F32: in_bytes = (size_t)a->n * h->cfg.clip_samples * 4; break;
    case TCR_INPUT_WAV_PCM16: {
      const int64_t stride = (a->clips && a->pcm_stride > 0) ? a->pcm_stride : h->cfg.clip_samples;
      if (stride > 2 * (int64_t)h->cfg.clip_samples) return fail(TCR_ERR_INVALID, "pcm_stride %lld exceeds 2 x clip_samples", (long long)stride);
      in_bytes = (size_t)a->n * stride * 2;
    } break;
    case TCR_INPUT_FEATURES: in_bytes = (size_t)a->n * h->frames * h->features * 4; break;
    default: return fail(TCR_ERR_INVALID, "unknown input kind %d", a->input_is_features);
  }
  if (f->submitted >= kFeedDepth) TCR_CUDA(cudaStreamWaitEvent(f->copy, sl.consumed, 0));   // the slot's previous step has read it
  TCR_CUDA(cudaMemcpyAsync(sl.d_in, a->input, in_bytes, cudaMemcpyHostToDevice, f->copy));
  TCR_CUDA(cudaMemcpyAsync(sl.d_hot, a->onehot, (size_t)a->n * h->cfg.num_classes * 4, cudaMemcpyHostToDevice, f->copy));
  if (a->clips) TCR_CUDA(cudaMemcpyAsync(sl.d_clips, a->clips, (size_t)a->n * sizeof(tcr_augment_clip), cudaMemcpyHostToDevice, f->copy));
  TCR_CUDA(cudaEventRecord(sl.ready, f->copy));
  TCR_CUDA(cudaStreamWaitEvent(s, sl.ready, 0));                   // labels (and features) for the step proper
  tcr_step_args d = *a;
  d.input = (const float*)sl.d_in;
  d.onehot = sl.d_hot;
  d.losses = sl.d_loss;
  if (a->clips) d.clips = sl.d_clips;          // the draws travel with the batch; the background bank is already on the device
  d.input_resident = 1;                        // the front-end waits for the copy only, not for the previous step on `stream`
  TCR_TRY(train_step_impl(h, &d, stream, sl.ready));
  TCR_CUDA(cudaEventRecord(sl.consumed, s));
  TCR_CUDA(cudaMemcpyAsync(sl.h_loss, sl.d_loss, 2 * sizeof(float), cudaMemcpyDeviceToHost, s));
  TCR_CUDA(cudaEventRecord(sl.done, s));
  ++f->submitted;
  if (f->submitted - f->collected > lag) TCR_TRY(hostfeed_collect(f, losses_out, losses_step));
  return TCR_OK;
}

extern "C" int tcr_host_flush(tcr_handle* h, float* losses_out, int64_t* losses_step) {
  if (!h) return fail(TCR_ERR_INVALID, "NULL argument");
  if (losses_step) *losses_step = -1;
  HostFeedState* f = (HostFeedState*)h->hostfeed;
  if (!f || f->collected >= f->submitted) return TCR_OK;
  return hostfeed_collect(f, losses_out, losses_step);
}

extern "C" int tcr_workspace_tensor(tcr_handle* h, const char* name, float** ptr, int64_t* numel) {
  if (!h || !name || !ptr || !numel) return fail(TCR_ERR_INVALID, "NULL argument");
  const int64_t n = h->last_n > 0 ? h->last_n : h->cfg.max_batch;
  const std::string s(name);
  auto ret = [&](float* p, int64_t k) {
    *ptr = p;
    *numel = k;
    return TCR_OK;
  };
  if (s == "timeline" && h->d_timeline) return ret((float*)h->d_timeline, 2 * 16 * 8192);   // int64 viewed as float pairs
  if (s == "features") return ret(h->feat_last ? h->feat_last : h->d_feat, n * h->frames * h->features);
  if (s == "grads") return ret(h->p2p.attached && h->world > 1 ? h->p2p.grads + (size_t)(h->p2p.step & 1u) * h->n_train : h->d_grads, h->n_train);
  if (s == "logits") return ret(h->d_logits, n * h->cfg.num_classes);
  if (s == "probs") return ret(h->d_probs, n * h->cfg.num_classes);
  const size_t colon = s.find(':');
  if (colon != std::string::npos) {
    const std::string kind = s.substr(0, colon), layer = s.substr(colon + 1);
    for (size_t i = 0; i < h->blocks.size(); ++i) {
      const std::string b = "block" + std::to_string(i);
      if (layer == b) {
        if (kind == "out") return ret(h->blocks[i].out, n * h->blocks[i].t * h->blocks[i].c);
        if (kind == "g") return ret(h->blocks[i].gblk, n * h->blocks[i].t * h->blocks[i].c);
      }
    }
    for (auto& cv : h->convs) {
      if (cv.name != layer) continue;
      if (kind == "y") return ret(cv.y, n * cv.t_out * cv.cout);
      if (kind == "g" && cv.g) return ret(cv.g, n * cv.t_out * cv.cout);
      if (kind == "bnf") return ret(cv.bnf, 4 * cv.cout);
      if (kind == "var") return ret(cv.var, cv.cout);
      if (kind == "bsum") return ret(cv.bsum, 2 * cv.cout);
    }
  }
  return fail(TCR_ERR_INVALID, "unknown workspace tensor '%s'", name);
}

extern "C" int tcr_comm_unique_id(void* id128) {
  int rc = comm_unique_id(id128);
  return rc ? fail(rc, "ncclGetUniqueId unavailable: %s", comm_error()) : TCR_OK;
}
extern "C" int tcr_comm_init(tcr_handle* h, const void* id128, int32_t rank, int32_t world_size) {
  if (!h || !id128 || world_size < 1 || rank < 0 || rank >= world_size) return fail(TCR_ERR_INVALID, "bad comm arguments");
  int rc = comm_init(h, id128, rank, world_size);
  return rc ? fail(rc, "ncclCommInitRank failed: %s", comm_error()) : TCR_OK;
}
extern "C" int tcr_comm_set_sync_bn(tcr_handle* h, int32_t enable) {
  if (!h) return fail(TCR_ERR_INVALID, "NULL argument");
  if (enable && (!h->comm || h->world < 2)) return fail(TCR_ERR_INVALID, "SyncBN needs an initialised communicator (tcr_comm_init, world > 1)");
  if (enable) {
    for (auto& cv : h->convs) {
      if (cv.fsync) continue;
      void* p = nullptr;
      TCR_CUDA(cudaMalloc(&p, (size_t)4 * cv.cout * sizeof(float)));
      h->allocs.push_back(p);
      cv.fsync = (float*)p;
      cv.bsync = cv.fsync + 2 * cv.cout;
    }
  }
  h->sync_bn = enable ? 1 : 0;
  resident_destroy(h);               // the mode is decided again on the next step (SyncBN: per-layer kernels)
  return TCR_OK;
}
extern "C" int tcr_comm_p2p_export(tcr_handle* h, void* handles128) {
  if (!h || !handles128) return fail(TCR_ERR_INVALID, "NULL argument");
  int rc = comm_p2p_export(h, handles128);
  return rc ? fail(rc, "peer-memory export failed: %s", comm_error()) : TCR_OK;
}
extern "C" int tcr_comm_p2p_attach(tcr_handle* h, const void* all_handles, int32_t rank, int32_t world_size) {
  if (!h || !all_handles || world_size < 1 || rank < 0 || rank >= world_size) return fail(TCR_ERR_INVALID, "bad comm arguments");
  int rc = comm_p2p_attach(h, all_handles, rank, world_size);
  return rc ? fail(rc, "peer-memory attach failed: %s", comm_error()) : TCR_OK;
}
extern "C" int tcr_comm_p2p_detach(tcr_handle* h) {
  if (!h) return TCR_OK;
  comm_p2p_destroy(h);
  return TCR_OK;
}
extern "C" int tcr_comm_destroy(tcr_handle* h) {
  if (!h) return TCR_OK;
  comm_destroy(h);
  return TCR_OK;
}

extern "C" int tcr_measure_fp32_peak(tcr_handle* h, double* tflops, tcr_stream stream) {
  pdl_chain_reset();
  if (!h || !tflops) return fail(TCR_ERR_INVALID, "NULL argument");
  int rc = measure_fp32_peak(h, tflops, (cudaStream_t)stream);
  return rc ? fail(rc, "fp32 peak measurement failed") : TCR_OK;
}

namespace tcr {
void set_error(const char* msg) { snprintf(g_err, sizeof(g_err), "%s", msg); }
}  // namespace tcr
