// Backward of the masked-AR stack / fused IAF step: internal interface used by iaf_capi.cu.
#pragma once
#include <algorithm>
#include <cstring>
#include <new>

#include "iaf_common.h"

struct IafBwdPlan;

struct IafBwdArgs {
  int mode;  // IAF_MODE_STEP | IAF_MODE_MULTICONV | IAF_MODE_LAYER
  int B;
  const float* z;
  const float* ctx;
  // packed (masked, normalised) weights of the plan, one entry per stage (iaf_pack.cu layout)
  const float* w_packed[IAF_MAX_STAGES];
  const float* bias_packed[IAF_MAX_STAGES];
  const float* padw_packed[IAF_MAX_STAGES];
  // raw parameters, one entry per layer (hidden layers first, then heads), reference layouts
  const float* const* w_raw;
  const float* const* scale_raw;
  // upstream gradients
  const float* g_zout;   // step: [B,n_z,H,W]
  const float* g_logsd;  // step: [B,n_z,H,W] or nullptr
  const float* g_logdet; // step: [B] or nullptr
  const float* g_heads[IAF_MAX_HEADS];  // multiconv: gradient of each head output
  // activations kept by the training forward (iaf_step_fwd_train): when have_saved the recompute is skipped
  int have_saved;
  const float* z_out_saved;              // z'
  const float* logsd_saved;              // arw_logsd
  const float* h_saved[IAF_MAX_HIDDEN];  // h_{j+1} = output of hidden layer j
  // fused-layer mode (IAF_MODE_LAYER): z is eps; the posterior / prior statistics and the KL gradients
  const float* post_mean; const float* post_logsd; const float* prior_mean; const float* prior_logsd;
  const float* g_kl;       // [B,C,H,W] or nullptr
  const float* g_kl_bc;    // [B,C] or nullptr
  const float* g_kl_cost;  // [B] or nullptr
  float* g_post_mean; float* g_post_logsd; float* g_prior_mean; float* g_prior_logsd;
  float* g_eps;            // nullable
  // results
  float* g_z;
  float* g_ctx;          // nullable
  float* const* g_w;     // nullable (as arrays): raw-parameter gradients in the reference layouts
  float* const* g_scale;
  float* const* g_bias;
};

// Data-dependent initialisation (iaf_multiconv_init): the stack run once, stage by stage, on the exact-fp32 layer conv;
// each layer's per-channel statistics become its new (g|s, b) and its normalised output feeds the next layer.
struct IafInitArgs {
  int B;
  const float* z;
  const float* ctx;
  // every stage packed with TF: zero gain and bias | Theano: the current s and b (iaf_pack.cu layout)
  const float* w_packed[IAF_MAX_STAGES];
  const float* bias_packed[IAF_MAX_STAGES];
  const float* padw_packed[IAF_MAX_STAGES];
  const float* const* scale_in;  // Theano: copied to the outputs of a skipped layer; unused for TF
  const float* const* bias_in;
  float* const* scale_out;       // one entry per layer (hidden layers first, then heads)
  float* const* bias_out;
  float* const* outs;            // head outputs of the pass, nullable
  int* skipped;                  // [n_layers]: channels with zero std (Theano skips the layer when > 0), nullable
};
int iaf_init_run(IafBwdPlan* p, const IafInitArgs* a, cudaStream_t stream, int* n_launches);

// allow_tc: the plan's forward runs on the tensor-core path, so its backward may too (data gradient as a layered-kernel stage,
// weight gradient as MN-major MMAs over the slot stream); a plan pinned to the exact-fp32 SIMT path keeps the SIMT backward
int iaf_bwd_plan_create(IafBwdPlan** out, const iaf_desc_t* d, const int* cin, const int* cout, const int* cout_pad,
                        int head_pad, int allow_tc);
int iaf_bwd_plan_uses_tc(const IafBwdPlan* p);  // 0: SIMT, 1: data gradient on tensor cores, 2: data and weight gradient
void iaf_bwd_plan_destroy(IafBwdPlan* p);
int iaf_bwd_run(IafBwdPlan* p, const IafBwdArgs* a, cudaStream_t stream, int* n_launches);
