/*
 * iaf_b200 -- C ABI of the B200-native IAF posterior step.
 *
 * The reference (openai/iaf) has no FFI layer: its boundary for this path is a python
 * callable.  These entry points are what a python (ctypes/cffi) binding of that callable
 * binds; each comment names the reference interface the function replaces
 * (paths relative to the reference repo).  Plain pointers and sizes only -- no torch,
 * no CUDA types in the signatures (streams travel as void*; NULL = default stream).
 *
 * All tensors are fp32, NCHW, contiguous.  Device pointers unless a name ends in _host.
 * Every function returns IAF_OK (0) or a negative iaf_status; nothing here ever falls
 * back to a CPU path.
 */
#ifndef IAF_B200_H
#define IAF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IAF_MAX_HIDDEN 4
#define IAF_MAX_HEADS 2

typedef enum {
  IAF_OK = 0,
  IAF_ERR_BAD_ARG = -1,     /* NULL pointer, non-positive size                               */
  IAF_ERR_BAD_SHAPE = -2,   /* the asserts of ar.py:225-257 / layers.py:116 (divisibility)    */
  IAF_ERR_UNSUPPORTED = -3, /* valid in the reference but outside what the kernels cover       */
  IAF_ERR_CUDA = -4,        /* a CUDA runtime call failed; see iaf_last_cuda_error()           */
  IAF_ERR_NOT_PACKED = -5,  /* iaf_step_* called before iaf_pack_weights                       */
  IAF_ERR_NO_DEVICE = -6    /* no sm_100 device                                                */
} iaf_status;

/* which of the reference's two implementations the numerics follow (SURVEY F2) */
typedef enum {
  IAF_VARIANT_TF = 0,    /* tf_utils/layers.py: SAME zero pad, cross-correlation, exp(g)*rsqrt(max(ss,1e-12)) */
  IAF_VARIANT_THEANO = 1 /* graphy/nodes/ar.py: pad channel, true convolution, exp(3s)/(sqrt(ss)+1e-8)        */
} iaf_variant;

/* graphy/nodes/__init__.py:158-177 (parameter-free entries); tf.nn.elu */
typedef enum { IAF_NL_NONE = 0, IAF_NL_ELU = 1, IAF_NL_SOFTPLUS = 2, IAF_NL_RELU = 3, IAF_NL_TANH = 4, IAF_NL_LEAKYRELU = 5 } iaf_nl;

typedef enum {
  IAF_PATH_AUTO = 0, /* tensor cores when the shape qualifies, else SIMT            */
  IAF_PATH_SIMT = 1, /* exact-fp32 FMA kernel (parity anchor, any shape)            */
  IAF_PATH_TC = 2    /* tcgen05 implicit-GEMM kernel, bf16x3 split operands         */
} iaf_path;

/*
 * Static description of one masked-AR conv stack; the arguments of
 *   multiconv2d(name, n_in, n_h, n_out, size_kernel, flipmask, nl, w)   graphy/nodes/ar.py:378
 *   ar_multiconv2d(name, x, context, n_h, n_out, nl)                     tf_utils/layers.py:159
 * size_kernel is fixed to 3x3 (the only size either caller uses: train.py:63, layers.py:145)
 * and flipmask to False (models.py:92).
 */
typedef struct iaf_desc {
  int variant;                /* iaf_variant                                               */
  int n_z;                    /* n_in: channels of z                                        */
  int n_hidden;               /* len(n_h): 0..IAF_MAX_HIDDEN (0 only meaningful for Theano, F8) */
  int hidden[IAF_MAX_HIDDEN]; /* n_h                                                        */
  int n_heads;                /* len(n_out): 1 or 2                                         */
  int head[IAF_MAX_HEADS];    /* n_out; two heads must have equal size                     */
  int H, W;                   /* feature-map size                                           */
  int nl;                     /* iaf_nl                                                     */
  int path;                   /* iaf_path                                                   */
} iaf_desc_t;

/* opaque: packed weights, scratch, launch geometry.  A plan is NOT re-entrant: its scratch serves one call at a time.
 * Calls on the same stream are ordered by the stream; when consecutive calls use different streams the library makes the
 * later stream wait for the earlier one (one event), so results stay correct -- but two streams never run the same plan
 * concurrently.  Use one plan per concurrent stream. */
typedef struct iaf_plan iaf_plan_t;

/* Validate the description and allocate the plan (replaces the graph-construction half of
 * ar.multiconv2d, ar.py:378-394, incl. its asserts).  */
int iaf_plan_create(iaf_plan_t** plan, const iaf_desc_t* desc);
void iaf_plan_destroy(iaf_plan_t* plan);

/*
 * Weight preparation, one fused kernel (replaces the per-call graph ops of
 * layers.py:53-60 and ar.py:312-321 + 267-281 + the mask constants of layers.py:134-141 /
 * ar.py:241-264).  Arrays have n_hidden + n_heads entries, hidden layers first, in the
 * reference's own layouts and names:
 *   TF:     w[i] = V [3,3,Cin,Cout], scale[i] = g [Cout], bias[i] = b [Cout]
 *   Theano: w[i] = {name}_w [Cout,Cin+1,3,3], scale[i] = {name}_s [Cout], bias[i] = {name}_b [Cout]
 * Raw (un-masked, un-normalised) parameters go in; masking is applied here, which also
 * makes the postup() re-masking of ar.py:369-373 unnecessary for the forward pass.
 */
int iaf_pack_weights(iaf_plan_t* plan, const float* const* w, const float* const* scale,
                     const float* const* bias, void* stream);

/*
 * The un-fused operator: outs[k] = head k of the masked-AR stack, i.e. exactly what
 *   posterior_conv1(z, context, w)            models.py:170,281 (ar.py:396-416)
 *   ar_multiconv2d(name, z, context, ...)     tf_train.py:69    (layers.py:158-166)
 * return (before the caller's *0.1).  z [B,n_z,H,W], context [B,hidden[0],H,W]
 * (ignored when n_hidden == 0), outs[k] [B,head[k],H,W].
 */
int iaf_multiconv_fwd(iaf_plan_t* plan, const float* z, const float* context, float* const* outs,
                      int B, void* stream);

/*
 * The fused IAF step (the hot path): stack + the caller's three lines
 *   arw_mean*=.1; arw_logsd*=.1; z=(z-arw_mean)/exp(arw_logsd); logqs+=arw_logsd
 *   models.py:282-285, models.py:171-175, tf_train.py:70-72
 * z_out [B,n_z,H,W]; logsd_out [B,n_z,H,W] = arw_logsd (the per-element term the ELBO
 * consumes, F7; may be NULL); logdet_out [B] = -sum_{c,h,w} arw_logsd (may be NULL).
 * Needs n_heads == 2 and head[0] == head[1] == n_z.
 */
int iaf_step_fwd(iaf_plan_t* plan, const float* z, const float* context, float* z_out,
                 float* logsd_out, float* logdet_out, int B, void* stream);

/*
 * Same step, host buffers: copies z/context H2D, runs iaf_step_fwd, copies the results
 * D2H and synchronises.  Buffers may be pageable or pinned (pinned for speed); device
 * staging belongs to the plan and grows on demand.  This is the end-to-end entry
 * bench.py's "e2e" times.
 */
int iaf_step_fwd_host(iaf_plan_t* plan, const float* z_host, const float* context_host,
                      float* z_out_host, float* logsd_out_host, float* logdet_out_host, int B,
                      void* stream);

/*
 * Pipelined form of the host entry for back-to-back batches: enqueues copy-in, the step and
 * copy-out of one batch on three internal streams (three device staging slots, so the H2D of batch
 * i+1, the kernel of batch i and the D2H of batch i-1 overlap: PCIe is full duplex) and returns
 * immediately.  Host buffers must be pinned and stay valid until iaf_host_wait() returns.
 */
int iaf_step_submit_host(iaf_plan_t* plan, const float* z_host, const float* context_host,
                         float* z_out_host, float* logsd_out_host, float* logdet_out_host, int B);
int iaf_host_wait(iaf_plan_t* plan);

/*
 * The stochastic-layer block around the step, fused (SURVEY 8f-1):
 *   tf_train.py:56-85 / models.py:273-298: posterior sample from the given noise, logqs,
 *   the IAF step, prior logps at z', kl = logqs - logps and its reductions.
 * post_mean/post_logsd: the posterior's mean and log-sd (rz+qz, already summed by the
 * caller: one add each, tf_train.py:57); eps: N(0,1) noise; prior_mean/prior_logsd.
 * Outputs: z_out [B,n_z,H,W]; kl_out [B,n_z,H,W] (may be NULL); kl_bc_out [B,n_z]
 * = sum_{h,w} kl (what the free-bits term consumes, may be NULL); kl_cost_out [B]
 * = sum_{c,h,w} kl (may be NULL).
 */
int iaf_layer_fwd(iaf_plan_t* plan, const float* eps, const float* post_mean, const float* post_logsd,
                  const float* prior_mean, const float* prior_logsd, const float* context,
                  float* z_out, float* kl_out, float* kl_bc_out, float* kl_cost_out, int B, void* stream);

/*
 * Backward of the fused step (SURVEY 8f-4): what theano.grad / tf.gradients derive for
 *   models.py:281-285 + ar.py:396-416   |   tf_train.py:69-72 + layers.py:158-166
 * including the gradient through the in-graph weight normalisation and the mask, so masked
 * taps receive exactly zero gradient (the contract postup() re-imposes, ar.py:369-373).
 * Inputs: the forward's z and context (activations are recomputed, nothing is saved by
 * iaf_step_fwd), the raw parameters w/scale as given to iaf_pack_weights (which must have
 * been called with them), and the upstream gradients g_z_out [B,n_z,H,W], g_logsd
 * [B,n_z,H,W] (may be NULL), g_logdet [B] (may be NULL).
 * Outputs: g_z [B,n_z,H,W]; g_context [B,hidden[0],H,W] (may be NULL; untouched when
 * n_hidden == 0); g_w/g_scale/g_bias: arrays of n_hidden + n_heads pointers in the
 * reference layouts of the parameters (each array may be NULL: all three NULL skips the
 * weight-gradient kernels).  Reductions are fixed-order: results are deterministic.
 */
int iaf_step_bwd(iaf_plan_t* plan, const float* z, const float* context, const float* const* w,
                 const float* const* scale, const float* g_z_out, const float* g_logsd,
                 const float* g_logdet, float* g_z, float* g_context, float* const* g_w,
                 float* const* g_scale, float* const* g_bias, int B, void* stream);

/*
 * Training pair: iaf_step_fwd_train is iaf_step_fwd that ALSO writes the hidden activations
 * (hidden_out[j] [B,hidden[j],H,W], j < n_hidden; the output of nl in ar.py:404 /
 * layers.py:164) from inside the same kernels, and iaf_step_bwd_saved is iaf_step_bwd fed
 * with them plus the forward's z_out / logsd_out instead of recomputing the stack (the
 * context is not needed then: it only enters the forward).  This is what the python
 * operator's autograd node uses.
 */
int iaf_step_fwd_train(iaf_plan_t* plan, const float* z, const float* context, float* z_out,
                       float* logsd_out, float* logdet_out, float* const* hidden_out, int B,
                       void* stream);
int iaf_step_bwd_saved(iaf_plan_t* plan, const float* z, const float* z_out, const float* logsd,
                       const float* const* hidden, const float* const* w,
                       const float* const* scale, const float* g_z_out, const float* g_logsd,
                       const float* g_logdet, float* g_z, float* g_context, float* const* g_w,
                       float* const* g_scale, float* const* g_bias, int B, void* stream);

/* The same pair for the un-fused operator (the reference's own drop-in signatures train through it). */
int iaf_multiconv_fwd_train(iaf_plan_t* plan, const float* z, const float* context,
                            float* const* outs, float* const* hidden_out, int B, void* stream);
int iaf_multiconv_bwd_saved(iaf_plan_t* plan, const float* z, const float* const* hidden,
                            const float* const* w, const float* const* scale,
                            const float* const* g_outs, float* g_z, float* g_context,
                            float* const* g_w, float* const* g_scale, float* const* g_bias, int B,
                            void* stream);

/*
 * Backward of the fused stochastic-layer block iaf_layer_fwd (tf_train.py:56-85 / models.py:273-298): upstream gradients
 * of z_out (may be NULL), of the per-element kl (may be NULL), of kl_bc [B,n_z] (may be NULL) and of kl_cost [B] (may be
 * NULL); results: the gradients of the posterior / prior statistics, of the noise (g_eps, may be NULL), of the context
 * and of the raw parameters.  Activations are recomputed.
 */
int iaf_layer_bwd(iaf_plan_t* plan, const float* eps, const float* post_mean, const float* post_logsd,
                  const float* prior_mean, const float* prior_logsd, const float* context,
                  const float* const* w, const float* const* scale, const float* g_z_out,
                  const float* g_kl, const float* g_kl_bc, const float* g_kl_cost, float* g_post_mean,
                  float* g_post_logsd, float* g_prior_mean, float* g_prior_logsd, float* g_eps,
                  float* g_context, float* const* g_w, float* const* g_scale, float* const* g_bias, int B,
                  void* stream);

/* Backward of the un-fused operator iaf_multiconv_fwd: g_outs[k] [B,head[k],H,W] is the
 * gradient at head k.  Same outputs as iaf_step_bwd. */
int iaf_multiconv_bwd(iaf_plan_t* plan, const float* z, const float* context, const float* const* w,
                      const float* const* scale, const float* const* g_outs, float* g_z,
                      float* g_context, float* const* g_w, float* const* g_scale,
                      float* const* g_bias, int B, void* stream);

/*
 * Data-dependent initialisation of the stack: the pass both reference front-ends run once on the first minibatch
 * before training (tf_train.py:226-228 -> layers.py:38-51 with init_scale = 1; models.py:541-544 -> ar.py:331-353),
 * layer by layer, each layer's returned tensor feeding the next (context added after hidden layer 0, nl after every
 * hidden layer).  Statistics are per output channel over (batch, H, W), population variance.
 *   TF:     x = xcorr(x_in, l2_normalize(mask o V)) (no gain, no bias; the current g, b are not read);
 *           scale = 1/sqrt(var + 1e-10); g := log(scale)/3; b := -mean*scale; returns scale*(x - mean).
 *           A zero-variance channel gets scale 1e5.  The forward uses exp(g), not exp(3g) (layers.py:60): a forward with
 *           the new parameters does NOT reproduce this pass's output -- the reference's behaviour, kept.
 *   Theano: h = the normal forward of the layer with the CURRENT s and b; if any channel has std 0 the layer keeps s, b
 *           and returns h (the reference prints a warning); else s := -log(std)/3, h /= std, b := -mean(h), h -= mean(h).
 *           s and b are overwritten, not composed with their current values.
 * w/scale/bias: n_hidden + n_heads entries in the layouts of iaf_pack_weights (TF: scale and bias may be NULL, they are
 * not read).  scale_out/bias_out: the new parameters, same layouts; they must not alias any input.  outs[k]
 * [B,head[k],H,W]: the pass's head outputs (outs may be NULL).  skipped [n_hidden + n_heads] int32 (may be NULL): the
 * number of zero-std channels of each layer; Theano skipped the layer when it is > 0, TF always writes 0.
 * Runs on exact-fp32 kernels with fixed-order double reductions on every plan (tensor-core plans included: it runs once
 * per training run and its statistics become the parameters); results are bit-identical across runs and paths.
 * Afterwards the plan is NOT packed: forward and backward entries return IAF_ERR_NOT_PACKED until iaf_pack_weights.
 */
int iaf_multiconv_init(iaf_plan_t* plan, const float* z, const float* context, const float* const* w,
                       const float* const* scale, const float* const* bias, float* const* scale_out,
                       float* const* bias_out, float* const* outs, int* skipped, int B, void* stream);

/* introspection */
const char* iaf_strerror(int status);
const char* iaf_last_cuda_error(void);          /* message of the last failing CUDA call (thread-local) */
int iaf_version(void);                          /* 10000*major + 100*minor + patch                      */
int iaf_plan_path(const iaf_plan_t* plan);      /* iaf_path actually selected (SIMT or TC)              */
/* The path ONE entry point runs on this plan.  A plan created with IAF_PATH_AUTO serves an entry the tensor-core kernels
 * cannot take for this shape (e.g. the fused layer's per-(sample, channel) scratch does not fit next to the resident
 * weights) on the exact-fp32 SIMT kernel -- 10-40x slower -- and says so here; a plan created with IAF_PATH_TC never
 * downgrades: that entry returns IAF_ERR_UNSUPPORTED, and so does this function. */
typedef enum { IAF_ENTRY_MULTICONV = 0, IAF_ENTRY_STEP = 1, IAF_ENTRY_LAYER = 2 } iaf_entry;
int iaf_plan_path_for_entry(const iaf_plan_t* plan, int entry);
/* Which kernels the plan's BACKWARD entries run (creates the backward plan on first use): 0 = exact-fp32 SIMT kernels,
 * 1 = data gradient on the tensor cores, 2 = data and weight gradient on the tensor cores (plans whose forward is on the
 * tensor-core path, channel counts in multiples of 16; IAF_BWD_TC=0 / IAF_BWD_WG_TC=0 in the environment switch them off).
 * The reference differentiates the same graph it runs forward (graphy/nodes/ar.py:304-329 through theano.grad). */
int iaf_plan_bwd_path(iaf_plan_t* plan);
uint64_t iaf_plan_launch_count(const iaf_plan_t* plan); /* kernels launched through this plan so far    */
size_t iaf_plan_algorithmic_bytes(const iaf_plan_t* plan, int B); /* SURVEY 8d bytes of one iaf_step_fwd */
double iaf_plan_algorithmic_flops(const iaf_plan_t* plan, int B); /* 2*B*H*W*sum nnz(mask)              */

#ifdef __cplusplus
}
#endif
#endif /* IAF_B200_H */
