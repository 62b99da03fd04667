// tcr_plan.h — host-side layer plan and handle of libtcr_b200.
#pragma once
#include <string>
#include <vector>

#include "tcr_device.cuh"
#include "tcr_internal.h"
#include "tcr_mfcc.h"

namespace tcr {

struct ConvPlan {
  std::string name;            // TF scope under <Net>/, e.g. "block0/conv0_0"
  int cin = 0, cout = 0, k = 0, stride = 1, t_in = 0, t_out = 0, pad_left = 0, relu = 1;
  int64_t w_off = 0, beta_off = 0, gamma_off = 0;   // offsets into the flat trainable buffer
  int64_t mm_off = 0, mv_off = 0;                    // offsets into the flat moving-statistics buffer
  // workspace (device)
  float* y = nullptr;          // [N, t_out, cout] pre-BN
  float* g = nullptr;          // [N, t_out, cout] dL/dz (conv_a / conv0 own one; conv_b and down alias gblk)
  float* bnf = nullptr;        // [4][cout]
  float* var = nullptr;        // [cout]
  float* fpart = nullptr;      // [records][cout][2] (sum y, sum y^2) per cluster (per CTA in the persistent kernel)
  float* bpart = nullptr;      // [records][cout][2] (sum dz, sum dz*xhat)
  float* bsum = nullptr;       // [2][cout]
  float* dwpart = nullptr;     // [R][k*cin*cout]
  float* wT = nullptr;         // [k][cout][cin] transposed filter bank (refreshed per backward pass)
  int dw_R = 1, dw_cot = 0, dw_RG = 1, dw_UB = 1;
  // per call: how many per-cluster records the producer launch of this step left in fpart / bpart (0: the global table /
  // sums are final: persistent kernel, evaluation tables)
  int f_gc = 0, b_gc = 0;
  float* fsync = nullptr; float* bsync = nullptr;   // [2*cout] sums over ALL ranks (tcr_comm_set_sync_bn, parity tests only)
  int64_t wnumel() const { return (int64_t)k * cin * cout; }
};

struct BlockPlan {
  int down = -1, a = -1, b = -1;   // indices into convs
  int c = 0, t = 0;
  float* out = nullptr;            // [N, t, c]
  float* gblk = nullptr;           // [N, t, c]
};

}  // namespace tcr

struct tcr_handle {
  tcr_config cfg;
  int frames = 0, features = 0, fft = 0, fpb = 1, fwarps = 1;
  int mfcc_pair = 1, pair_fpb = 10, pair_warps = 5, c_twa = -1, sms = 1, pair_segw_len = 0, pair_dct_len = 0;
  int* d_seg_meta = nullptr;   // frame-pair front-end kernel (tcr_mfcc_pair.cu)
  std::string scope;
  std::vector<tcr::ConvPlan> convs;
  std::vector<tcr::BlockPlan> blocks;
  int c_last = 0, t_last = 0;
  int64_t n_train = 0, n_moving = 0, fc_off = 0, fc2_off = 0;
  std::vector<tcr_param_desc> table;
  int g_max = 0;                 // max CTA groups of any producer kernel (partials are sized for it)
  int head_groups_max = 0;
  // front-end tables
  float* d_fe_consts = nullptr; int c_tw2 = 0, c_melw = 0, c_win = 0, c_smem = 0;   // front-end constant block (tcr_mfcc.h)
  int* d_mel_start = nullptr; int* d_mel_len = nullptr; int* d_mel_off = nullptr;
  float* d_dct = nullptr;
  // workspace
  float* d_feat = nullptr;
  // front-end running ahead on its own stream (tcr_step_args::input_resident, tcr_train_step_host): two feature buffers, the
  // events "features of buffer b are ready" / "the step that read buffer b has finished"
  void* fe_stream = nullptr; float* fe_feat[2] = {nullptr, nullptr}; void* fe_ready[2] = {nullptr, nullptr};
  void* fe_free[2] = {nullptr, nullptr}; long long fe_count = 0;
  float* fe_aug = nullptr;           // the ahead path's own decoded-wav buffer (device input stage)
  void* fe_gate = nullptr; int fe_gate_valid = 0;   // recorded on the step's stream once the weight gradients are launched: the next
                                     // step's front-end starts behind it, i.e. next to grad_finalize / update, not next to the FMA-bound kernels
  float* feat_last = nullptr;
  int sync_bn = 0;                   // BatchNorm statistics over the global batch (per-layer kernels + NCCL; tcr_comm_set_sync_bn)        // feature buffer the library filled last ("features" of tcr_workspace_tensor)
  float* d_logits = nullptr; float* d_probs = nullptr;
  float* d_loss_part = nullptr; float* d_loss = nullptr; float* d_dwfc_part = nullptr;
  float* d_grads = nullptr;
  float* d_l2part = nullptr;
  tcr::Hyper* d_hyper = nullptr; tcr::Hyper* h_hyper = nullptr;
  tcr::OptSegment* d_segs = nullptr; int n_segs = 0;
  tcr::MovingSegment* d_msegs = nullptr; int n_msegs = 0;
  tcr::DwLayer* d_dw_layers = nullptr; int n_dw_layers = 0; int dw_ctas = 0; size_t dw_smem = 0;
  std::vector<void*> allocs;
  int64_t workspace_bytes = 0;
  // data-parallel
  void* comm = nullptr; int rank = 0, world = 1;
  // peer-memory gradient exchange (csrc/tcr_comm.cu): own double-buffered flat gradient + arrival flags, and every rank's
  // mappings of them (CUDA IPC).  When attached, the update kernel sums the ranks' gradients itself and NCCL is not used.
  struct P2P {
    int attached = 0;
    float* grads = nullptr;          // [2][n_train] this rank's flat gradient, buffer = step parity
    unsigned* flags = nullptr;       // [kMaxPeers] flags[r] = last step whose gradient rank r has finished
    float* peer_grads[8] = {};       // every rank's `grads` as mapped here (own entry = own pointer)
    unsigned* peer_flags[8] = {};
    unsigned step = 0;
  } p2p;
  int last_n = 0;
  int loss_gc = 0;            // cross-entropy records left by the head launch of this call
  int cluster = 0;            // CTAs per thread-block cluster of the conv / head launches (env TCR_CLUSTER, default 8)
  int64_t background_samples = 0;   // floats in the background bank (tcr_set_background_samples); 0: offsets are trusted
  float* d_aug = nullptr;      // [max_batch][clip_samples] fp32 output of the device input stage inside a step (lazy)
  void* hostfeed = nullptr;   // HostFeedState (tcr_api.cu): staging slots of tcr_train_step_host
  void* resident = nullptr;          // ResidentState (tcr_resident.cu): layout + program of the resident forward kernel
  int fc_records = 0;                // per-CTA records of the fc weight gradient left by the last head launch
  unsigned* d_gridbar = nullptr;    // arrival counter of the resident kernel's grid barrier (monotonic, never reset)
  unsigned* d_opt_ticket = nullptr; // retirement counter of the Adam update launch (0 between launches; the last CTA resets it)
  long long* d_timeline = nullptr;   // TCR_DEBUG_TIMELINE=1: per-CTA phase stamps (fwd kernels: 8 slots per CTA; dw: after)
};
