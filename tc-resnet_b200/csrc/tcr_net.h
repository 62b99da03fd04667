// tcr_net.h — host-side launch sequences implemented in tcr_net_fwd.cu / tcr_net_bwd.cu /
// tcr_optim.cu / tcr_comm.cu.  All return 0 or a TCR_ERR_* code (message via tcr::set_error).
#pragma once
#include "tcr_plan.h"

namespace tcr {

void set_error(const char* msg);

int net_alloc_workspace(tcr_handle* h);

// Forward pass on features [n, T, F].  training: batch-statistics BN (+ dropout); otherwise the BN tables are
// built from `moving`.  backward: the head additionally emits dlogits-derived tensors for net_backward.
int net_forward(tcr_handle* h, const float* feat, const float* params, const float* moving, int n, bool training,
                uint64_t seed, const float* mask, const float* onehot, float weight_decay, float* logits,
                float* probs, float* losses, bool backward, cudaStream_t s);

// Backward-data chain + all weight-gradient kernels; leaves per-layer partial sums in the workspace.
int cluster_size(tcr_handle* h);
StatSrc stat_src(const tcr_handle* h, const ConvPlan& cv, const float* params, int n);
int augment_launch(const int16_t* pcm, int64_t pcm_stride, const tcr_augment_clip* clips, const float* background, int64_t background_samples,
                   float* out, int clip, int n, cudaStream_t s);
int eval_accumulate_launch(const float* scores, const float* onehot, int n, int classes, int topk, int64_t* counts, cudaStream_t s);
int net_weight_transpose(tcr_handle* h, const float* params, cudaStream_t s);
// Resident forward (tcr_resident.cu): the training forward + head as one cooperative kernel with SM-resident activations.
int sync_records(tcr_handle* h, const float* part, int gc, int cols, float* out, cudaStream_t s);   // SyncBN: sum records, all-reduce
inline bool sync_bn_on(const tcr_handle* h) { return h->sync_bn && h->world > 1 && h->comm; }
inline float bn_inv(const tcr_handle* h, int n, int t) { return 1.0f / ((float)n * (float)t * (sync_bn_on(h) ? (float)h->world : 1.0f)); }
int resident_mode(tcr_handle* h);      // 0: per-layer kernels, 1: resident forward, 2: resident forward + backward (dW inside), 3: resident forward + backward-data
int resident_forward(tcr_handle* h, const float* feat, const tcr_step_args* a, cudaStream_t s);
int resident_backward(tcr_handle* h, const float* feat, const tcr_step_args* a, float* grads, int* l2_records, cudaStream_t s);
int resident_backward_data(tcr_handle* h, const float* feat, const tcr_step_args* a, cudaStream_t s);   // mode 3
int net_weight_gradients(tcr_handle* h, const float* feat, int n, cudaStream_t s);                      // the grouped launch alone
void resident_destroy(tcr_handle* h);
int net_backward(tcr_handle* h, const float* feat, const float* params, int n, cudaStream_t s);

// Gradient finalisation (+ weight decay), optional NCCL all-reduce, optimizer update (tcr_step_args::optimizer, + EMA), BN moving
// averages, losses.
int net_update(tcr_handle* h, const float* feat, const tcr_step_args* a, cudaStream_t s);

int launch_loss_only(tcr_handle* h, const float* params, float weight_decay, int n, float* losses, cudaStream_t s);
int head_groups(int n);


int measure_fp32_peak(tcr_handle* h, double* tflops, cudaStream_t s);

// NCCL through dlopen (tcr_comm.cu): no link-time dependency, the torch-bundled libnccl is reused when loaded.
int comm_unique_id(void* id128);
int comm_init(tcr_handle* h, const void* id128, int rank, int world);
void comm_destroy(tcr_handle* h);
int comm_allreduce_sum(tcr_handle* h, float* buf, int64_t count, cudaStream_t s);
int comm_p2p_export(tcr_handle* h, void* handles128);
int comm_p2p_attach(tcr_handle* h, const void* all_handles, int rank, int world);
void comm_p2p_destroy(tcr_handle* h);
const char* comm_error();

}  // namespace tcr
