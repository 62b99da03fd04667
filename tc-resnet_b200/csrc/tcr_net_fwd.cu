// tcr_net_fwd.cu — TC-ResNet forward kernels for sm_100a (fp32 CUDA-core FMA; see DESIGN.md for why the
// 9x1 temporal convolutions stay on the FMA pipe: TF32/BF16 tensor-core products break the 1e-4 logit bound).
//
// Replaces tc_resnet() (audio_nets/tc_resnet.py:6-54) under TCResNet_arg_scope (:102-123):
//   conv_fwd_kernel<K>  : [k,1] temporal conv (+ the block's 1x1/stride-2 shortcut conv from the same staged
//                         input tile), BN+ReLU(+residual) of the PRODUCER applied while staging the tile,
//                         BatchNorm partial sums in the epilogue, reduced over the 8 CTAs of a thread-block cluster through
//                         distributed shared memory; the CONSUMER kernel turns the records into the table (tcr_bn.cuh).
//   head_kernel         : residual + ReLU + global average pool + dropout + fc + softmax + cross-entropy and,
//                         for training, dlogits -> gradient of the last block + fc weight-gradient partials.
// A CTA owns U whole utterances, so SAME padding is a few zero rows of the shared-memory tile.
#include <stdlib.h>

#include "tcr_bn.cuh"
#include "tcr_net.h"

namespace tcr {

constexpr int TM = 4;   // output rows per thread task

// ------------------------------------------------------------------------------------------------
// conv forward
// ------------------------------------------------------------------------------------------------
template <int K, bool WSMEM>
__device__ __forceinline__ void conv_fwd_body(const FwdArgs& a, const int vb, const int nvb, unsigned char* smem_raw, MbarCtx& mb) {
  float* smem = reinterpret_cast<float*>(smem_raw);
  const int tid = threadIdx.x;
  const int u0 = vb * a.U;
  const int Ue = imax(0, imin(a.U, a.n - u0));        // 0: a CTA that only pads the grid to whole clusters
  (void)nvb;
  const int CS = chan_stride(a.cin);
  const int pad_right = imax((a.t_out - 1) * a.stride + K - a.pad_left - a.t_in, 0);
  const int TP = a.pad_left + a.t_in + pad_right;
  const int Rmax = a.U * a.t_out;
  // shared memory: [mbarrier | W (TMA bulk destination) | W_down | x tile | y tiles | scratch]
  uint64_t* bar = mb.bar;
  float* ws = smem + 4;                               // [K][cin][cout]   (only when a.w_smem)
  const int wn = WSMEM ? K * a.cin * a.cout : 0;
  const int wdn = (WSMEM && a.wd) ? a.cin * a.coutd : 0;
  float* wsd = ws + wn;                               // [cin][coutd]
  float* xs = wsd + wdn;                              // [U][TP][CS]
  float* ys = xs + (size_t)a.U * TP * CS;             // [KS][Rmax][cout]
  float* ysd = ys + (size_t)a.KS * Rmax * a.cout;     // [Rmax][coutd]
  float* red = ysd + (a.wd ? (size_t)Rmax * a.coutd : 0);   // [2 * kThreads] scratch
  float* tbl_in = red + 2 * kThreads;                 // [4][cin] BN table of the input layer
  float* tbl_sh = tbl_in + 4 * a.cin;                 // [4][cin] BN table of the shortcut (down conv of the previous block)
  float* spart = tbl_sh + 4 * a.cin;                  // [2*cout + 2*coutd] this CTA's (sum y, sum y^2)
  const int ws_off = (int)(ws - smem), wsd_off = (int)(wsd - smem), xs_off = (int)(xs - smem);

  tl_stamp(a.tl, vb, 0);
  // ---- one TMA bulk copy brings the whole filter bank into shared memory while the tile is staged ----
  if (WSMEM) {
    if (!mb.ready) {
      if (tid == 0) mbar_init(bar, 1);
      __syncthreads();
      mb.ready = true;
    }
    if (tid == 0) {
      fence_proxy_async();          // earlier generic-proxy reads of this buffer are ordered before the async write
      mbar_expect_tx(bar, (uint32_t)(wn + wdn) * 4u);
      tma_load_1d(ws, a.w, (uint32_t)wn * 4u, bar);
      if (wdn) tma_load_1d(wsd, a.wd, (uint32_t)wdn * 4u, bar);
    }
  }

  // ---- stage the input tile (producer's BN/ReLU/residual applied here) ----
  const int c4n = a.cin >> 2;
  const int npad = a.pad_left + pad_right;
  for (int idx = tid; idx < Ue * npad * c4n; idx += kThreads) {
    const int c4 = idx % c4n, pr = (idx / c4n) % npad, u = idx / (c4n * npad);
    const int row = pr < a.pad_left ? pr : a.t_in + pr;
    st4(xs + ((size_t)(u * TP + row) * CS + 4 * c4), make_float4(0.f, 0.f, 0.f, 0.f));
  }
  pdl_wait();                       // everything above is independent of the producer kernel (filters: caller-owned params)
  tl_stamp(a.tl, vb, 7);
  {
    // c4 fixed per thread (per-channel constants in registers), rows advance incrementally: no div/mod per element.
    // The raw rows are requested BEFORE the BN tables are built, so the two global round trips (records, tile) overlap.
    const RowWalk w = row_walk(tid, kThreads, c4n);
    const int rows = Ue * a.t_in;
    const size_t grow = (size_t)u0 * a.t_in;
    constexpr int PF = 4;             // rows per thread kept in flight (a thread owns at most ~4 rows at the tile sizes in use)
    const bool res = a.in_kind == 2;
    float4 pin[PF], psh[PF];
#pragma unroll
    for (int i = 0; i < PF; ++i) {
      const int row = w.row + i * w.rstep;
      pin[i] = psh[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row < rows) {
        const size_t gofs = (grow + row) * a.cin + 4 * w.c4;
        pin[i] = ld4(a.in.data + gofs);
        if (res) psh[i] = ld4(a.shortcut.data + gofs);
      }
    }
    // BN tables of the layers this tile reads, summed from the producers' per-cluster records (tcr_bn.cuh)
    if (res && a.shortcut.kind == 1) bn_table_build2(a.in.st, a.in.bnf, tbl_in, a.shortcut.st, a.shortcut.bnf, tbl_sh, a.cin, red, vb == 0);
    else if (a.in_kind != 0) bn_table_build(a.in.st, a.in.bnf, a.cin, tbl_in, red, vb == 0);
    if (w.row < rows) {
      int u = w.row / a.t_in, t = w.row - u * a.t_in;
      Chan4 kin, ksh;
      kin.mean = kin.rstd = kin.scale = kin.beta = ksh.mean = ksh.rstd = ksh.scale = ksh.beta = make_float4(0.f, 0.f, 0.f, 0.f);
      if (a.in_kind != 0) kin = chan4_load_s(tbl_in, a.cin, 4 * w.c4);
      const bool sh_bn = res && a.shortcut.kind == 1;
      if (sh_bn) ksh = chan4_load_s(tbl_sh, a.cin, 4 * w.c4);
      auto place = [&](int row, float4 vin, float4 vsh) {
        float4 v = vin;
        if (a.in_kind == 1) {
          v = relu4(chan4_bn(kin, vin));
        } else if (res) {
          if (sh_bn) vsh = relu4(chan4_bn(ksh, vsh));
          v = relu4(add4(chan4_bn(kin, vin), vsh));
          if (a.out_write) st4(a.out_write + (grow + row) * a.cin + 4 * w.c4, v);
        }
        st4(xs + ((size_t)(u * TP + a.pad_left + t) * CS + 4 * w.c4), v);
        t += w.rstep;
        while (t >= a.t_in) { t -= a.t_in; ++u; }
      };
#pragma unroll
      for (int i = 0; i < PF; ++i) {
        const int row = w.row + i * w.rstep;
        if (row < rows) place(row, pin[i], psh[i]);
      }
      for (int row = w.row + PF * w.rstep; row < rows; row += w.rstep) {
        const size_t gofs = (grow + row) * a.cin + 4 * w.c4;
        place(row, ld4(a.in.data + gofs), res ? ld4(a.shortcut.data + gofs) : make_float4(0.f, 0.f, 0.f, 0.f));
      }
    }
  }
  tl_stamp(a.tl, vb, 1);
  if (WSMEM) { mbar_wait(bar, mb.parity); mb.parity ^= 1u; }
  __syncthreads();
  tl_stamp(a.tl, vb, 2);

  // ---- register-tiled conv: task = (k-slice, row tile of TM, 4 output channels) ----
  const int R = Ue * a.t_out;
  const int NRT = (R + TM - 1) / TM;
  const int NCG = a.cout >> 2;
  const int KPS = K / a.KS;
  const int ntasks = NRT * NCG * a.KS;
  const int NCGD = a.wd ? (a.coutd >> 2) : 0;
  const int ntasks_all = ntasks + NRT * NCGD;
  for (int task = tid; task < ntasks_all; task += kThreads) {
    const bool is_down = task >= ntasks;
    const int tk = is_down ? task - ntasks : task;
    const int ncg = is_down ? NCGD : NCG;
    const int cg = tk % ncg;
    const int rt = (tk / ncg) % NRT;
    const int ks = is_down ? 0 : tk / (ncg * NRT);
    // 32-bit float offsets from the shared-memory base: the inner loop is LDS.128 + FFMA with integer adds only
    int xo[TM];
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int r = imin(rt + i * NRT, R - 1);      // rows of a task are NRT apart: adjacent lanes -> adjacent rows
      const int u = r / a.t_out, t = r - u * a.t_out;
      xo[i] = xs_off + (is_down ? (u * TP + a.pad_left + 2 * t) : (u * TP + t * a.stride)) * CS;
    }
    float4 acc[TM];
#pragma unroll
    for (int i = 0; i < TM; ++i) acc[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    const int k_lo = is_down ? 0 : ks * KPS, k_hi = is_down ? 1 : k_lo + KPS;
    const int co_n = is_down ? a.coutd : a.cout;
    if (WSMEM) {
      const int wb = (is_down ? wsd_off : ws_off) + 4 * cg;
      for (int k = k_lo; k < k_hi; ++k) {
        int wk = wb + k * a.cin * co_n;
        const int xk = k * CS;
#pragma unroll 2
        for (int ci = 0; ci < a.cin; ci += 4, wk += 4 * co_n) {
          const float4 w0 = ld4(smem + wk), w1 = ld4(smem + wk + co_n), w2 = ld4(smem + wk + 2 * co_n), w3 = ld4(smem + wk + 3 * co_n);
#pragma unroll
          for (int i = 0; i < TM; ++i) {
            const float4 x = ld4(smem + xo[i] + xk + ci);
            acc[i].x = fmaf(x.x, w0.x, acc[i].x); acc[i].y = fmaf(x.x, w0.y, acc[i].y);
            acc[i].z = fmaf(x.x, w0.z, acc[i].z); acc[i].w = fmaf(x.x, w0.w, acc[i].w);
            acc[i].x = fmaf(x.y, w1.x, acc[i].x); acc[i].y = fmaf(x.y, w1.y, acc[i].y);
            acc[i].z = fmaf(x.y, w1.z, acc[i].z); acc[i].w = fmaf(x.y, w1.w, acc[i].w);
            acc[i].x = fmaf(x.z, w2.x, acc[i].x); acc[i].y = fmaf(x.z, w2.y, acc[i].y);
            acc[i].z = fmaf(x.z, w2.z, acc[i].z); acc[i].w = fmaf(x.z, w2.w, acc[i].w);
            acc[i].x = fmaf(x.w, w3.x, acc[i].x); acc[i].y = fmaf(x.w, w3.y, acc[i].y);
            acc[i].z = fmaf(x.w, w3.z, acc[i].z); acc[i].w = fmaf(x.w, w3.w, acc[i].w);
          }
        }
      }
    } else {
      const float* wbase = (is_down ? a.wd : a.w) + 4 * cg;
      for (int k = k_lo; k < k_hi; ++k) {
        const float* wk = wbase + (size_t)k * a.cin * co_n;
        const int xk = k * CS;
#pragma unroll 2
        for (int ci = 0; ci < a.cin; ci += 4, wk += 4 * co_n) {
          const float4 w0 = ldg4(wk), w1 = ldg4(wk + co_n), w2 = ldg4(wk + 2 * co_n), w3 = ldg4(wk + 3 * co_n);
#pragma unroll
          for (int i = 0; i < TM; ++i) {
            const float4 x = ld4(smem + xo[i] + xk + ci);
            acc[i].x = fmaf(x.x, w0.x, acc[i].x); acc[i].y = fmaf(x.x, w0.y, acc[i].y);
            acc[i].z = fmaf(x.x, w0.z, acc[i].z); acc[i].w = fmaf(x.x, w0.w, acc[i].w);
            acc[i].x = fmaf(x.y, w1.x, acc[i].x); acc[i].y = fmaf(x.y, w1.y, acc[i].y);
            acc[i].z = fmaf(x.y, w1.z, acc[i].z); acc[i].w = fmaf(x.y, w1.w, acc[i].w);
            acc[i].x = fmaf(x.z, w2.x, acc[i].x); acc[i].y = fmaf(x.z, w2.y, acc[i].y);
            acc[i].z = fmaf(x.z, w2.z, acc[i].z); acc[i].w = fmaf(x.z, w2.w, acc[i].w);
            acc[i].x = fmaf(x.w, w3.x, acc[i].x); acc[i].y = fmaf(x.w, w3.y, acc[i].y);
            acc[i].z = fmaf(x.w, w3.z, acc[i].z); acc[i].w = fmaf(x.w, w3.w, acc[i].w);
          }
        }
      }
    }
    float* dst = is_down ? ysd : ys + (size_t)ks * Rmax * a.cout;
#pragma unroll
    for (int i = 0; i < TM; ++i) {
      const int r = rt + i * NRT;
      if (r < R) st4(dst + (size_t)r * co_n + 4 * cg, acc[i]);
    }
  }
  __syncthreads();
  tl_stamp(a.tl, vb, 3);

  // ---- epilogue: sum k-slices in fixed order, coalesced store of the pre-BN output ----
  const size_t grow0 = (size_t)u0 * a.t_out;
  for (int idx = tid; idx < R * NCG; idx += kThreads) {
    float4 v = ld4(ys + (size_t)idx * 4);
    for (int ks = 1; ks < a.KS; ++ks) v = add4(v, ld4(ys + (size_t)ks * Rmax * a.cout + (size_t)idx * 4));
    st4(ys + (size_t)idx * 4, v);
    st4(a.y + grow0 * a.cout + (size_t)idx * 4, v);
  }
  if (a.wd)
    for (int idx = tid; idx < R * NCGD; idx += kThreads) st4(a.yd + grow0 * a.coutd + (size_t)idx * 4, ld4(ysd + (size_t)idx * 4));
  if (!a.train) return;
  __syncthreads();
  tl_stamp(a.tl, vb, 4);
  tile_stats(ys, R, a.cout, red, nullptr, spart);
  if (a.wd) tile_stats(ysd, R, a.coutd, red, nullptr, spart + 2 * a.cout);
  tl_stamp(a.tl, vb, 5);
  const PubSeg segs[2] = {{spart, 2 * a.cout, a.fpart}, {spart + 2 * a.cout, a.wd ? 2 * a.coutd : 0, a.fpartd}};
  cluster_publish(segs, vb);
  tl_stamp(a.tl, vb, 6);
}

template <int K, bool WSMEM>
__global__ void __launch_bounds__(kThreads) conv_fwd_kernel(FwdArgs a) {
  TCR_DYNAMIC_SMEM(smem_raw);
  MbarCtx mb{reinterpret_cast<uint64_t*>(smem_raw), 0u, false};
  pdl_trigger();                    // grid <= resident CTA slots: the next kernel's CTAs may take slots as ours retire
  conv_fwd_body<K, WSMEM>(a, blockIdx.x, a.nvb, smem_raw, mb);
}

// Eval mode: BN tables from the moving statistics (bn_forward with is_training=False).
struct EvalBnArgs {
  int nlayers;
  const float* params;
  const float* moving;
  float eps;
  int c[kMaxConvs];
  int64_t gamma_off[kMaxConvs], beta_off[kMaxConvs], mm_off[kMaxConvs], mv_off[kMaxConvs];
  float* bnf[kMaxConvs];
};
__global__ void bn_table_eval_kernel(EvalBnArgs a) {
  pdl_wait();
  const int l = blockIdx.x;
  const int C = a.c[l];
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float mean = a.moving[a.mm_off[l] + c], var = a.moving[a.mv_off[l] + c];
    const double rstd = 1.0 / sqrt((double)var + (double)a.eps);
    a.bnf[l][c] = mean;
    a.bnf[l][C + c] = (float)rstd;
    a.bnf[l][2 * C + c] = (float)((double)a.params[a.gamma_off[l] + c] * rstd);
    a.bnf[l][3 * C + c] = a.params[a.beta_off[l] + c];
  }
}

// ------------------------------------------------------------------------------------------------
// head: kHeadU utterances per CTA.  residual add + ReLU, average pool, dropout, fc, softmax cross-entropy and, for
// training, the head backward (gradient at the block output, BN-backward partial sums, fc dW partials).
// Every stage is a short loop over a flat index, so the code that each CTA runs exactly once stays small.
// ------------------------------------------------------------------------------------------------
constexpr int kHeadU = 4;
constexpr int kHeadThreads = 256;

// Shared-memory layout (floats): tb[4][C] td[4][C] wfc[C][NC] | so, syb, ssh [U*T*C] each | drop, mk, dnet [U*C] each |
// logit, dl [U*NC] each | loss [U] (+pad) | red [4][SEG][C] (<= 4 * 256)
__host__ __device__ inline size_t head_smem_floats(int T, int C, int NC) {
  return (size_t)8 * C + (size_t)C * NC + 4 + (size_t)3 * kHeadU * T * C + 4 + (size_t)3 * kHeadU * C + (size_t)2 * kHeadU * NC +
         kHeadU + 8 + 4 * kHeadThreads + 4 * C + 4;
}

__device__ __forceinline__ void head_body(const HeadArgs& a, const int vb, const int nvb, unsigned char* smem_raw) {
  (void)nvb;
  float* smem = reinterpret_cast<float*>(smem_raw) + 4;          // first 16 bytes: the persistent kernel's mbarrier
  const int C = a.c, T = a.t, NC = a.classes, TC = T * C;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int u0 = vb * kHeadU, nu = imax(0, imin(kHeadU, a.n - u0)), rows = nu * T;   // nu == 0: cluster padding CTA
  float* tb = smem;
  float* td = tb + 4 * C;
  float* s_wfc = td + 4 * C;
  float* so = s_wfc + ((C * NC + 3) & ~3);
  float* syb = so + ((kHeadU * TC + 3) & ~3);
  float* ssh = syb + ((kHeadU * TC + 3) & ~3);
  float* s_drop = ssh + ((kHeadU * TC + 3) & ~3);
  float* s_mk = s_drop + kHeadU * C;
  float* s_dnet = s_mk + kHeadU * C;
  float* s_logit = s_dnet + kHeadU * C;
  float* s_dl = s_logit + kHeadU * NC;
  float* s_loss = s_dl + kHeadU * NC;
  float* red = s_loss + kHeadU;                           // [4 * kHeadThreads]: scratch, then the CTA's partial sums
  const bool sh_bn = a.shortcut.kind == 1;
  const size_t base = (size_t)u0 * TC;

  // the CTA's utterances are one contiguous span; its first rows are requested before the tables are summed
  constexpr int PF = 2;
  float4 pyb[PF], psh[PF];
#pragma unroll
  for (int i = 0; i < PF; ++i) {
    const int e = 4 * (tid + i * kHeadThreads);
    pyb[i] = psh[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (e < nu * TC) { pyb[i] = ld4(a.in.data + base + e); psh[i] = ld4(a.shortcut.data + base + e); }
  }
  if (sh_bn) bn_table_build2(a.in.st, a.in.bnf, tb, a.shortcut.st, a.shortcut.bnf, td, C, red, vb == 0);
  else bn_table_build(a.in.st, a.in.bnf, C, tb, red, vb == 0);
#pragma unroll 1
  for (int i = tid; i < C * NC; i += kHeadThreads) s_wfc[i] = __ldg(a.wfc + i);
#pragma unroll
  for (int i = 0; i < PF; ++i) {
    const int e = 4 * (tid + i * kHeadThreads);
    if (e < nu * TC) { st4(syb + e, pyb[i]); st4(ssh + e, psh[i]); }
  }
#pragma unroll 1
  for (int e = 4 * (tid + PF * kHeadThreads); e < nu * TC; e += 4 * kHeadThreads) {
    st4(syb + e, ld4(a.in.data + base + e));
    st4(ssh + e, ld4(a.shortcut.data + base + e));
  }
  __syncthreads();

  // block output o = relu(bn(y_b) + shortcut): thread (seg, c) walks rows seg, seg + SEG, ...
  const int SEG = kHeadThreads / C;
  const int seg = tid / C, c = tid - seg * C;
  if (seg < SEG) {
    const float mb_ = tb[c], sb_ = tb[2 * C + c], bb_ = tb[3 * C + c];
    const float md_ = td[c], sd_ = td[2 * C + c], bd_ = td[3 * C + c];
#pragma unroll 1
    for (int r = seg; r < rows; r += SEG) {
      const float zb = fmaf(syb[r * C + c] - mb_, sb_, bb_);
      float sh = ssh[r * C + c];
      if (sh_bn) sh = fmaxf(fmaf(sh - md_, sd_, bd_), 0.f);
      const float o = fmaxf(zb + sh, 0.f);
      so[r * C + c] = o;
      if (a.out_write) a.out_write[base + r * C + c] = o;
    }
  }
  __syncthreads();
  // average pool + dropout
#pragma unroll 1
  for (int i = tid; i < nu * C; i += kHeadThreads) {
    const int u = i / C, cc = i - u * C;
    float acc = 0.f;
    for (int t = 0; t < T; ++t) acc += so[(u * T + t) * C + cc];
    const float pooled = acc / (float)T;
    float mk = 1.f, dropped = pooled;
    if (a.use_dropout) {
      const size_t gi = (size_t)(u0 + u) * C + cc;
      mk = a.mask ? a.mask[gi] : floorf(a.keep + uniform01(a.seed, (uint64_t)gi));
      dropped = pooled / a.keep * mk;                       // tf.nn.dropout: x / keep_prob * floor(keep_prob + U)
    }
    s_drop[i] = dropped;
    s_mk[i] = mk;
  }
  __syncthreads();
  // fc (no bias): one warp per (utterance, class)
#pragma unroll 1
  for (int o = warp; o < nu * NC; o += kHeadThreads / 32) {
    const int u = o / NC, k = o - u * NC;
    float p = 0.f;
    for (int cc = lane; cc < C; cc += 32) p = fmaf(s_drop[u * C + cc], s_wfc[cc * NC + k], p);
    p = warp_sum(p);
    if (lane == 0) s_logit[o] = p;
  }
  __syncthreads();
  // softmax cross-entropy: one warp per utterance, lane k keeps class k (NC <= 32)
#pragma unroll 1
  for (int u = warp; u < nu; u += kHeadThreads / 32) {
    const bool act = lane < NC;
    const float logit = act ? s_logit[u * NC + lane] : 0.f;
    const float mx = warp_max(act ? logit : -3.0e38f);
    const float e = act ? expf(logit - mx) : 0.f;
    const float se = warp_sum(e);
    const float prob = e / se;
    const float logp = (logit - mx) - logf(se);
    const size_t gi = (size_t)(u0 + u) * NC + lane;
    if (act) {
      if (a.logits) a.logits[gi] = logit;
      if (a.probs) a.probs[gi] = prob;
    }
    float loss_n = 0.f, dl = 0.f;
    if (a.onehot) {
      float lab = act ? a.onehot[gi] : 0.f;
      if (a.label_smoothing > 0.f && act) lab = lab * (1.f - a.label_smoothing) + a.label_smoothing / (float)NC;
      const float labsum = warp_sum(lab);
      loss_n = -warp_sum(act ? lab * logp : 0.f);
      dl = act ? (prob * labsum - lab) * a.inv_n : 0.f;
    }
    if (act) s_dl[u * NC + lane] = dl;
    if (lane == 0) s_loss[u] = loss_n;
  }
  __syncthreads();
  if (!a.backward) {
    if (a.onehot) {
      if (tid == 0) {
        float s = 0.f;
        for (int u = 0; u < nu; ++u) s += s_loss[u];
        red[0] = s;
      }
      const PubSeg segs[1] = {{red, 1, a.loss_part}};
      cluster_publish(segs, vb);                          // one CE record per cluster; the loss kernel adds them
    }
    return;
  }

  // ---- head backward: d logits -> d pooled (fc^T, dropout, AvgPoolGrad) ----
#pragma unroll 1
  for (int i = tid; i < nu * C; i += kHeadThreads) {
    const int u = i / C, cc = i - u * C;
    float d = 0.f;
    for (int k = 0; k < NC; ++k) d = fmaf(s_dl[u * NC + k], s_wfc[cc * NC + k], d);
    if (a.use_dropout) d = d / a.keep * s_mk[i];
    s_dnet[i] = d / (float)T;
  }
  __syncthreads();
  // gradient at the block output and the BN-backward partial sums of conv_b (and of the down conv)
  {
    float sb1 = 0.f, sb2 = 0.f, sd1 = 0.f, sd2 = 0.f;
    if (seg < SEG) {
      const float mb_ = tb[c], rb_ = tb[C + c];
      const float md_ = td[c], rd_ = td[C + c], sd_ = td[2 * C + c], bd_ = td[3 * C + c];
#pragma unroll 1
      for (int r = seg; r < rows; r += SEG) {
        const int u = r / T;
        const float g = so[r * C + c] > 0.f ? s_dnet[u * C + c] : 0.f;
        a.gout[base + r * C + c] = g;
        sb1 += g;
        sb2 = fmaf(g, (syb[r * C + c] - mb_) * rb_, sb2);
        if (a.ydn) {
          const float yd = ssh[r * C + c];
          const float gs = fmaf(yd - md_, sd_, bd_) > 0.f ? g : 0.f;
          sd1 += gs;
          sd2 = fmaf(gs, (yd - md_) * rd_, sd2);
        }
      }
      red[(0 * SEG + seg) * C + c] = sb1;
      red[(1 * SEG + seg) * C + c] = sb2;
      red[(2 * SEG + seg) * C + c] = sd1;
      red[(3 * SEG + seg) * C + c] = sd2;
    }
  }
  __syncthreads();
  float* sp = red + 4 * SEG * C;                          // [4C + 1] this CTA's sums: conv_b (c*2+q), down (c*2+q), CE
#pragma unroll 1
  for (int i = tid; i < 4 * C; i += kHeadThreads) {
    const int q = i / C, cc = i - q * C;
    float s = 0.f;
    for (int k = 0; k < SEG; ++k) s += red[(q * SEG + k) * C + cc];
    sp[(q >> 1) * 2 * C + cc * 2 + (q & 1)] = s;
  }
  if (tid == 0) {
    float s = 0.f;
    for (int u = 0; u < nu; ++u) s += s_loss[u];
    sp[4 * C] = s;
  }
#pragma unroll 1
  for (int i = tid; i < C * NC; i += kHeadThreads) {
    const int cc = i / NC, k = i - cc * NC;
    float s = 0.f;
    for (int u = 0; u < nu; ++u) s = fmaf(s_drop[u * C + cc], s_dl[u * NC + k], s);
    if (nu > 0) a.dwfc_part[(size_t)vb * C * NC + i] = s;     // cluster-padding CTAs own no record
  }
  const PubSeg segs[3] = {{sp, 2 * C, a.bpartb}, {sp + 2 * C, a.ydn ? 2 * C : 0, a.bpartd}, {sp + 4 * C, 1, a.loss_part}};
  cluster_publish(segs, vb);
}

__global__ void __launch_bounds__(kHeadThreads) head_kernel(HeadArgs a) {
  TCR_DYNAMIC_SMEM(smem_raw);
  pdl_trigger();
  pdl_wait();
  head_body(a, blockIdx.x, a.nvb, smem_raw);
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static constexpr size_t kSmemBudget = 110 * 1024;   // two CTAs per SM: 2 x (110 + 1 static + 1 reserved) KB <= 227 KB

int head_groups(int n) { return (n + kHeadU - 1) / kHeadU; }

static size_t fwd_weight_floats(const ConvPlan& cv, const ConvPlan* dn) {
  return (size_t)cv.wnumel() + (dn ? (size_t)dn->wnumel() : 0);
}

static size_t fwd_smem_bytes(const ConvPlan& cv, const ConvPlan* dn, int U, int KS, bool w_smem) {
  const int CS = chan_stride(cv.cin);
  const int pad_right = std::max((cv.t_out - 1) * cv.stride + cv.k - cv.pad_left - cv.t_in, 0);
  const int TP = cv.pad_left + cv.t_in + pad_right;
  size_t f = (size_t)U * TP * CS + (size_t)KS * U * cv.t_out * cv.cout + (dn ? (size_t)U * cv.t_out * dn->cout : 0);
  f += 2 * kThreads + 8 * (size_t)cv.cin + 2 * (size_t)cv.cout + (dn ? 2 * (size_t)dn->cout : 0);   // scratch, 2 BN tables, partial sums
  f += 4 + (w_smem ? fwd_weight_floats(cv, dn) : 0);
  return f * 4;
}

// Utterances per CTA, k-slices and whether the filter bank is staged in shared memory.
// Goals: >= 2 resident CTAs per SM when the batch allows (latency hiding), all 148 SMs busy, balanced thread tasks.
static constexpr size_t kSmemMax = 200 * 1024;      // opt-in limit we are willing to use for one CTA

// Candidate tilings are compared by a small cost model: waves x (U x (co-residency slowdown) + fixed part), where a wave is one
// round of CTAs over the 148 SMs at the residency the shared-memory footprint allows.  (Measured on TCResNet14-1.5, N=1024: a tile
// that fits only one CTA per SM must cover the batch in ONE wave of <= 148 CTAs; two waves of 128 cost 2x the fixed part.)
static constexpr int kSMs = 148;
double tile_cost(int n, int U, int occ, bool wsm) {
  const int groups = (n + U - 1) / U;
  const int waves = (groups + kSMs * occ - 1) / (kSMs * occ);
  // unit = FMA time of one utterance on an otherwise idle SM.  Measured on TCResNet14-1.5 (profiles/r01_v11_*): a lone 8-warp CTA
  // per SM cannot hide its latencies (76-89 us at 152 CTAs vs 47-54 us at 256 CTAs, two per SM), and reading the filter bank
  // through L1/L2 costs about the same as staging it in shared memory (48 us), so residency decides, not the filter path.
  // The per-wave fixed part (launch, filter TMA, staging latency, statistics, cluster publish) is ~4 such units.
  return waves * (U * (occ == 2 ? 1.7 : 1.8) * (wsm ? 1.0 : 1.1) + 4.0);
}

static void pick_fwd_tile(const ConvPlan& cv, const ConvPlan* dn, int n, int* U_out, int* KS_out, int* wsm_out) {
  const size_t wbytes = fwd_weight_floats(cv, dn) * 4;
  double best = 1e30;
  *U_out = 1; *KS_out = 1; *wsm_out = 0;
  for (int pass = 0; pass < 4; ++pass) {
    // passes 0/1: filter bank in shared memory, two / one CTA per SM; passes 2/3: filters through L1/L2 (bank too large)
    const bool wsm = pass < 2;
    const int occ = (pass & 1) ? 1 : 2;
    const size_t budget = occ == 2 ? kSmemBudget : kSmemMax;
    if (wsm && wbytes + 16 * 1024 > budget) continue;
    for (int U = std::min(16, std::max(1, (n + kSMs * occ - 1) / (kSMs * occ))); U >= 1; --U) {
      int best_ks = 0;
      double best_cost = 1e30;
      for (int KS = 1; KS <= cv.k; ++KS) {
        if (cv.k % KS) continue;
        const int nrt = (U * cv.t_out + TM - 1) / TM;
        const long tasks = (long)nrt * (cv.cout / 4) * KS + (dn ? (long)nrt * (dn->cout / 4) : 0);
        const double cost = (double)((tasks + kThreads - 1) / kThreads) * (cv.k / KS);
        if (cost < best_cost - 1e-9 && fwd_smem_bytes(cv, dn, U, KS, wsm) <= budget) {
          best_cost = cost;
          best_ks = KS;
        }
      }
      if (!best_ks) continue;
      const double c = tile_cost(n, U, occ, wsm);
      if (c < best - 1e-9) { best = c; *U_out = U; *KS_out = best_ks; *wsm_out = wsm ? 1 : 0; }
      break;                        // the largest U that fits is the candidate of this pass
    }
  }
}

template <class T>
static int ws_alloc(tcr_handle* h, T** p, size_t count) {
  void* q = nullptr;
  size_t bytes = std::max<size_t>(count, 1) * sizeof(T);
  bytes = (bytes + 255) & ~(size_t)255;
  if (cudaMalloc(&q, bytes) != cudaSuccess) {
    set_error("cudaMalloc failed while sizing the workspace");
    return TCR_ERR_CUDA;
  }
  h->allocs.push_back(q);
  h->workspace_bytes += (int64_t)bytes;
  *p = (T*)q;
  return 0;
}
#define WS(x)             \
  do {                    \
    int rc_ = (x);        \
    if (rc_) return rc_;  \
  } while (0)

void plan_bwd_weight(tcr_handle* h);   // tcr_net_bwd.cu
int build_opt_segments(tcr_handle* h); // tcr_optim.cu
int build_dw_table(tcr_handle* h);     // tcr_net_bwd.cu

int net_alloc_workspace(tcr_handle* h) {
  const size_t N = (size_t)h->cfg.max_batch;
  h->g_max = h->cfg.max_batch;                       // U >= 1 -> at most max_batch CTA groups
  h->head_groups_max = head_groups(h->cfg.max_batch);
  plan_bwd_weight(h);
  WS(ws_alloc(h, &h->d_feat, N * h->frames * h->features));
  WS(ws_alloc(h, &h->d_logits, N * h->cfg.num_classes));
  WS(ws_alloc(h, &h->d_probs, N * h->cfg.num_classes));
  for (auto& cv : h->convs) {
    const size_t act = N * cv.t_out * cv.cout;
    WS(ws_alloc(h, &cv.y, act));
    WS(ws_alloc(h, &cv.bnf, 4 * (size_t)cv.cout));
    WS(ws_alloc(h, &cv.var, (size_t)cv.cout));
    WS(ws_alloc(h, &cv.fpart, (size_t)std::max(h->g_max, 256) * cv.cout * 2));
    WS(ws_alloc(h, &cv.bpart, (size_t)std::max(std::max(h->g_max, h->head_groups_max), 256) * cv.cout * 2));
    WS(ws_alloc(h, &cv.bsum, 2 * (size_t)cv.cout));
    WS(ws_alloc(h, &cv.dwpart, (size_t)cv.dw_R * cv.wnumel()));
    WS(ws_alloc(h, &cv.wT, (size_t)cv.wnumel()));
  }
  WS(ws_alloc(h, &h->convs[0].g, N * h->convs[0].t_out * h->convs[0].cout));
  for (auto& b : h->blocks) {
    WS(ws_alloc(h, &b.out, N * b.t * b.c));
    WS(ws_alloc(h, &b.gblk, N * b.t * b.c));
    ConvPlan& ca = h->convs[b.a];
    WS(ws_alloc(h, &ca.g, N * ca.t_out * ca.cout));
    h->convs[b.b].g = b.gblk;
    if (b.down >= 0) h->convs[b.down].g = b.gblk;
  }
  const size_t rec_max = (size_t)std::max(h->head_groups_max, 256);   // head records: per cluster, per 4 utterances, or per SM (resident kernel)
  WS(ws_alloc(h, &h->d_loss_part, rec_max));
  WS(ws_alloc(h, &h->d_loss, 4));
  WS(ws_alloc(h, &h->d_dwfc_part, rec_max * h->c_last * h->cfg.num_classes));
  WS(ws_alloc(h, &h->d_grads, (size_t)h->n_train));
  WS(ws_alloc(h, &h->d_l2part, 4096));
  WS(ws_alloc(h, &h->d_hyper, 1));
  WS(ws_alloc(h, &h->d_gridbar, 64));
  cudaMemset(h->d_gridbar, 0, 64 * sizeof(unsigned));
  h->d_opt_ticket = h->d_gridbar + 32;     // the resident grid barrier uses word 0; the ticket gets its own 128-byte line
  if (getenv("TCR_DEBUG_TIMELINE")) {
    WS(ws_alloc(h, &h->d_timeline, (size_t)16 * 8192));
    cudaMemset(h->d_timeline, 0, sizeof(long long) * 16 * 8192);
  }
  if (cudaMallocHost((void**)&h->h_hyper, sizeof(Hyper)) != cudaSuccess) return TCR_ERR_CUDA;
  int rc = build_dw_table(h);
  if (rc) return rc;
  return build_opt_segments(h);
}

// Thread-block cluster size of the conv / head launches: 8 CTAs add their BatchNorm partial sums through distributed shared
// memory (tcr_bn.cuh).  TCR_CLUSTER=1 falls back to one record per CTA.
int cluster_size(tcr_handle* h) {
  if (h->cluster == 0) {
    const char* e = getenv("TCR_CLUSTER");
    int c = e ? atoi(e) : 8;
    if (c != 1 && c != 2 && c != 4 && c != 8) c = 8;
    h->cluster = c;
  }
  return h->cluster;
}
StatSrc stat_src(const tcr_handle* h, const ConvPlan& cv, const float* params, int n) {
  if (sync_bn_on(h) && cv.f_gc)     // SyncBN: one "record" holding the sums over all ranks, count = global rows
    return StatSrc{cv.fsync, 1, params + cv.gamma_off, params + cv.beta_off, cv.bnf, cv.var, bn_inv(h, n, cv.t_out), h->cfg.bn_epsilon};
  return StatSrc{cv.f_gc ? cv.fpart : nullptr, cv.f_gc, params + cv.gamma_off, params + cv.beta_off, cv.bnf, cv.var,
                 1.0f / ((float)n * (float)cv.t_out), h->cfg.bn_epsilon};
}

// SyncBN (parity tests only): out[c] = sum over this rank's records, then summed over the ranks by NCCL.
__global__ void __launch_bounds__(256) records_sum_kernel(const float* __restrict__ part, int gc, int cols, float* __restrict__ out) {
  pdl_wait();
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    float s = 0.f;
    for (int g = 0; g < gc; ++g) s += part[(size_t)g * cols + c];
    out[c] = s;
  }
}
int sync_records(tcr_handle* h, const float* part, int gc, int cols, float* out, cudaStream_t s) {
  TCR_LAUNCH("records_sum", records_sum_kernel, dim3(1), dim3(256), 0, s, part, gc, cols, out);
  return comm_allreduce_sum(h, out, cols, s);
}
static ActSrc act_of(const tcr_handle* h, const ConvPlan& cv, int kind, const float* params, int n) {
  return ActSrc{cv.y, cv.bnf, kind, stat_src(h, cv, params, n)};
}

template <int K, bool WSMEM>
static int launch_conv_fwd(const char* name, const FwdArgs& a, int groups, size_t smem, cudaStream_t s, int cluster) {
  auto kfn = conv_fwd_kernel<K, WSMEM>;
#ifndef TCR_EMU
  static SmemOptIn optin;           // one per template instantiation
  if (optin.ensure(kfn, smem) != cudaSuccess) return TCR_ERR_CUDA;
#endif
  TCR_LAUNCH_CLUSTER(name, kfn, dim3(groups), dim3(kThreads), smem, s, cluster, a);
  return 0;
}

static int conv_fwd(tcr_handle* h, ConvPlan& cv, ConvPlan* dn, FwdArgs a, const float* params, int n, bool training,
                    cudaStream_t s) {
  int U, KS, wsm;
  pick_fwd_tile(cv, dn, n, &U, &KS, &wsm);
  a.n = n; a.U = U; a.t_in = cv.t_in; a.cin = cv.cin; a.w_smem = wsm;
  a.w = params + cv.w_off; a.y = cv.y; a.fpart = cv.fpart;
  a.cout = cv.cout; a.stride = cv.stride; a.t_out = cv.t_out; a.pad_left = cv.pad_left; a.KS = KS;
  a.wd = nullptr; a.yd = nullptr; a.fpartd = nullptr; a.coutd = 0;
  a.train = training ? 1 : 0;
  a.tl = (h->d_timeline && cv.name == "block2/conv2_0") ? h->d_timeline : nullptr;
  if (h->d_timeline && cv.name == "block1/conv1_1") a.tl = h->d_timeline + 2048 * 8;   // its producer, rows 2048..
  a.eps = h->cfg.bn_epsilon;
  if (dn) {
    a.wd = params + dn->w_off; a.yd = dn->y; a.fpartd = dn->fpart; a.coutd = dn->cout;
  }
  const int groups = (n + U - 1) / U;
  a.nvb = groups;
  const size_t smem = fwd_smem_bytes(cv, dn, U, KS, wsm != 0);
  cv.f_gc = 0;
  if (dn) dn->f_gc = 0;
  const int CL = cluster_size(h);
  const int grid = (groups + CL - 1) / CL * CL;
  if (training) {                   // the consumers of this layer's statistics sum grid / CL records
    cv.f_gc = grid / CL;
    if (dn) dn->f_gc = grid / CL;
  }
  int rc;
  switch (cv.k) {
    case 3: rc = wsm ? launch_conv_fwd<3, true>(("fwd:" + cv.name).c_str(), a, grid, smem, s, CL)
                     : launch_conv_fwd<3, false>(("fwd:" + cv.name).c_str(), a, grid, smem, s, CL);
      break;
    case 9: rc = wsm ? launch_conv_fwd<9, true>(("fwd:" + cv.name).c_str(), a, grid, smem, s, CL)
                     : launch_conv_fwd<9, false>(("fwd:" + cv.name).c_str(), a, grid, smem, s, CL);
      break;
    default: set_error("unsupported kernel width"); return TCR_ERR_UNSUPPORTED;
  }
  if (!rc && training && sync_bn_on(h)) {
    rc = sync_records(h, cv.fpart, cv.f_gc, 2 * cv.cout, cv.fsync, s);
    if (!rc && dn) rc = sync_records(h, dn->fpart, dn->f_gc, 2 * dn->cout, dn->fsync, s);
  }
  return rc;
}

int net_forward(tcr_handle* h, const float* feat, const float* params, const float* moving, int n, bool training,
                uint64_t seed, const float* mask, const float* onehot, float weight_decay, float* logits,
                float* probs, float* losses, bool backward, cudaStream_t s) {
  (void)weight_decay;
  if (h->c_last > kHeadThreads) { set_error("last_channels > 256 unsupported by the head kernel"); return TCR_ERR_UNSUPPORTED; }
  if (!training) {
    EvalBnArgs e;
    e.nlayers = (int)h->convs.size();
    e.params = params; e.moving = moving; e.eps = h->cfg.bn_epsilon;
    for (int l = 0; l < e.nlayers; ++l) {
      const ConvPlan& cv = h->convs[l];
      e.c[l] = cv.cout; e.gamma_off[l] = cv.gamma_off; e.beta_off[l] = cv.beta_off;
      e.mm_off[l] = cv.mm_off; e.mv_off[l] = cv.mv_off; e.bnf[l] = cv.bnf;
    }
    TCR_LAUNCH("bn_table_eval", bn_table_eval_kernel, dim3(e.nlayers), dim3(128), 0, s, e);
  }
  // conv0 on raw features
  {
    FwdArgs a;
    memset(&a, 0, sizeof(a));
    a.in_kind = 0;
    a.in = ActSrc{feat, nullptr, 0, StatSrc{}};
    int rc = conv_fwd(h, h->convs[0], nullptr, a, params, n, training, s);
    if (rc) return rc;
  }
  ActSrc prev = act_of(h, h->convs[0], 1, params, n);   // activation feeding the next block
  for (size_t i = 0; i < h->blocks.size(); ++i) {
    BlockPlan& b = h->blocks[i];
    ConvPlan& ca = h->convs[b.a];
    ConvPlan& cb = h->convs[b.b];
    ConvPlan* dn = b.down >= 0 ? &h->convs[b.down] : nullptr;
    FwdArgs a;
    memset(&a, 0, sizeof(a));
    if (i == 0) {
      a.in_kind = 1;
      a.in = prev;
    } else {
      // input = output of block i-1 = relu(bn(y_b) + shortcut); materialised here for the backward pass
      BlockPlan& pb = h->blocks[i - 1];
      a.in_kind = 2;
      a.in = act_of(h, h->convs[pb.b], 0, params, n);
      a.shortcut = pb.down >= 0 ? act_of(h, h->convs[pb.down], 1, params, n) : prev;
      a.out_write = pb.out;
    }
    int rc = conv_fwd(h, ca, dn, a, params, n, training, s);
    if (rc) return rc;
    if (i > 0) prev = ActSrc{h->blocks[i - 1].out, nullptr, 0, StatSrc{}};   // materialised by the launch above
    FwdArgs a2;
    memset(&a2, 0, sizeof(a2));
    a2.in_kind = 1;
    a2.in = act_of(h, ca, 1, params, n);
    rc = conv_fwd(h, cb, nullptr, a2, params, n, training, s);
    if (rc) return rc;
    if (i + 1 == h->blocks.size()) {
      BlockPlan& lb = b;
      HeadArgs ha;
      memset(&ha, 0, sizeof(ha));
      ha.in = act_of(h, cb, 0, params, n);
      ha.shortcut = dn ? act_of(h, *dn, 1, params, n) : prev;
      ha.out_write = lb.out;
      ha.n = n; ha.t = lb.t; ha.c = lb.c; ha.classes = h->cfg.num_classes;
      ha.wfc = params + h->fc_off;
      ha.onehot = onehot;
      ha.mask = mask; ha.seed = seed; ha.keep = h->cfg.dropout_keep_prob;
      ha.use_dropout = (training && h->cfg.dropout_keep_prob < 1.0f) ? 1 : 0;
      ha.label_smoothing = h->cfg.label_smoothing;
      ha.logits = logits ? logits : h->d_logits;
      ha.probs = probs ? probs : h->d_probs;
      ha.loss_part = h->d_loss_part;
      ha.backward = backward ? 1 : 0;
      ha.inv_n = 1.0f / (float)n;
      ha.gout = lb.gblk;
      ha.yb = cb.y; ha.bnfb = cb.bnf; ha.bpartb = cb.bpart;
      ha.ydn = dn ? dn->y : nullptr; ha.bnfd = dn ? dn->bnf : nullptr; ha.bpartd = dn ? dn->bpart : nullptr;
      ha.dwfc_part = h->d_dwfc_part;
      const int groups = head_groups(n);
      ha.nvb = groups;
      const int CL = cluster_size(h);
      const int grid = (groups + CL - 1) / CL * CL;
      h->loss_gc = grid / CL;
      h->fc_records = groups;           // CE records the loss / update kernel adds
      cb.b_gc = backward ? grid / CL : 0;
      if (dn) dn->b_gc = cb.b_gc;
      const size_t smem = (head_smem_floats(lb.t, lb.c, ha.classes) + 8) * 4;
      if (smem > kSmemBudget || lb.c > kHeadThreads) { set_error("head tile does not fit in shared memory"); return TCR_ERR_UNSUPPORTED; }
      {
#ifndef TCR_EMU
        static SmemOptIn optin;
        if (optin.ensure(head_kernel, smem) != cudaSuccess) return TCR_ERR_CUDA;
#endif
        TCR_LAUNCH_CLUSTER("head", head_kernel, dim3(grid), dim3(kHeadThreads), smem, s, CL, ha);
      }
      if (backward && sync_bn_on(h)) {
        int rcs = sync_records(h, cb.bpart, cb.b_gc, 2 * cb.cout, cb.bsync, s);
        if (!rcs && dn) rcs = sync_records(h, dn->bpart, dn->b_gc, 2 * dn->cout, dn->bsync, s);
        if (rcs) return rcs;
      }
    }
    // the identity shortcut of the NEXT block is this block's materialised output; it is written by the next
    // block's first kernel, so `prev` is updated at the top of the next iteration.
  }
  if (losses && onehot && !backward) {
    int rc = launch_loss_only(h, params, weight_decay, n, losses, s);
    if (rc) return rc;
  }
  return 0;
}

}  // namespace tcr
