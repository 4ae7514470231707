// C ABI of libiaf_b200.so (declared in include/iaf_b200.h): plan management, weight
// packing, path selection and the launchers.  No torch, no CPU fallback.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include "iaf_common.h"
#include "iaf_tc.h"
#include "iaf_bwd.h"

namespace {

thread_local char g_cuda_err[512] = "";

int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
  return IAF_ERR_CUDA;
}
#define CK(call)                                   \
  do {                                             \
    cudaError_t e_ = (call);                       \
    if (e_ != cudaSuccess) return cuda_fail(e_, #call); \
  } while (0)

int round_up(int a, int b) { return (a + b - 1) / b * b; }

long long centre_nnz(int cin, int cout, int zd) {
  long long n = 0;
  for (int co = 0; co < cout; ++co)
    for (int ci = 0; ci < cin; ++ci) {
      bool vis;
      if (cout >= cin) {
        int k = cout / cin, i = co / k;
        vis = zd ? ci < i : ci <= i;
      } else {
        int k = cin / cout;
        vis = zd ? ci < co * k : ci < (co + 1) * k;
      }
      n += vis;
    }
  return n;
}

}  // namespace

struct iaf_plan {
  iaf_desc_t d;
  int path;
  int device;
  int n_stages;                       // n_hidden + 1
  // SIMT packed weights, one entry per stage (last = merged heads)
  float* w[IAF_MAX_STAGES];
  float* bias[IAF_MAX_STAGES];
  float* padw[IAF_MAX_STAGES];
  int cin[IAF_MAX_STAGES], cout[IAF_MAX_STAGES], cout_pad[IAF_MAX_STAGES];
  size_t w_elems[IAF_MAX_STAGES];
  int head_pad;
  bool packed;
  bool simt_ok;
  // SIMT geometry
  int band_rows, n_bands, P;
  int bufz, bufa, bufb, tilepart;
  size_t smem;
  // scratch
  float* partial;
  unsigned* counter;
  int scratch_B;
  // host-entry staging
  float* st_z; float* st_ctx; float* st_zo; float* st_ls; float* st_ld;
  int staging_B;
  // pipelined host entry: IAF_NSLOT device staging slots, copy-in / compute / copy-out streams
  float* ps_z[3]; float* ps_ctx[3]; float* ps_zo[3]; float* ps_ls[3]; float* ps_ld[3];
  cudaStream_t s_h2d, s_cmp, s_d2h;
  cudaEvent_t ev_h2d[3], ev_cmp[3], ev_d2h[3];
  int pipe_B;
  uint64_t submit_idx;
  // tensor-core path
  IafTcPlan* tc;
  // backward (created on the first iaf_*_bwd call)
  IafBwdPlan* bwd;
  // recompute of iaf_step_bwd (the entry without kept activations) on the forward's own tensor-core kernels
  float* rc_zo; float* rc_ls; float* rc_h[IAF_MAX_HIDDEN];
  int rc_B;
  // zero gain and bias the TF data-dependent init packs with (allocated on first use)
  float* init_zeros;
  uint64_t launches;
  // a plan's scratch (partial sums, counters, packed weights, operand images) serves ONE stream at a time: when a call
  // arrives on a different stream than the previous one, the new stream first waits for the old one's work
  cudaStream_t last_stream;
  bool last_stream_valid;
  cudaEvent_t ev_handoff;
};
#define IAF_NSLOT 3

static bool simt_geometry(iaf_plan* pl, int band_rows, size_t* smem_out) {
  const iaf_desc_t& d = pl->d;
  const int nst = pl->n_stages;
  const int nseg = (d.W + 7) / 8;
  const int P = 8 * nseg + 2;
  const int rows_alloc = band_rows + nst;
  int bufz = d.n_z * rows_alloc * P;
  int ca = 0, cb = 0;
  for (int j = 0; j + 1 < nst; ++j) {
    if (j & 1) cb = std::max(cb, pl->cout[j]);
    else ca = std::max(ca, pl->cout[j]);
  }
  int bufa = ca * rows_alloc * P, bufb = cb * rows_alloc * P;
  int tilepart = band_rows * nseg * (pl->cout_pad[nst - 1] / 8) * 4;
  // keep every region 16-byte aligned
  bufz = round_up(bufz, 4); bufa = round_up(bufa, 4); bufb = round_up(bufb, 4);
  size_t smem = sizeof(float) * ((size_t)bufz + bufa + bufb + tilepart);
  if (smem_out) *smem_out = smem;
  pl->band_rows = band_rows;
  pl->n_bands = (d.H + band_rows - 1) / band_rows;
  pl->P = P;
  pl->bufz = bufz; pl->bufa = bufa; pl->bufb = bufb; pl->tilepart = tilepart;
  pl->smem = smem;
  return true;
}

// Order this call after the plan's previous call when the stream changed (see iaf_plan::last_stream).  Skipped while
// either stream is being captured into a CUDA graph: a capture only ever sees one stream of ours.
static int stream_handoff(iaf_plan* pl, cudaStream_t stream) {
#ifndef IAF_EMU
  if (pl->last_stream_valid && pl->last_stream != stream) {
    cudaStreamCaptureStatus c0 = cudaStreamCaptureStatusNone, c1 = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(stream, &c1);
    cudaStreamIsCapturing(pl->last_stream, &c0);
    if (c0 == cudaStreamCaptureStatusNone && c1 == cudaStreamCaptureStatusNone) {
      if (!pl->ev_handoff) CK(cudaEventCreateWithFlags(&pl->ev_handoff, cudaEventDisableTiming));
      CK(cudaEventRecord(pl->ev_handoff, pl->last_stream));
      CK(cudaStreamWaitEvent(stream, pl->ev_handoff, 0));
    }
  }
  pl->last_stream = stream;
  pl->last_stream_valid = true;
#else
  (void)pl; (void)stream;
#endif
  return IAF_OK;
}

static int ensure_scratch(iaf_plan* pl, int B) {
  if (B <= pl->scratch_B) return IAF_OK;
  if (pl->partial) cudaFree(pl->partial);
  if (pl->counter) cudaFree(pl->counter);
  pl->partial = nullptr; pl->counter = nullptr; pl->scratch_B = 0;
  const int maxbands = pl->d.H;  // worst case band_rows = 1
  CK(cudaMalloc(&pl->partial, sizeof(float) * (size_t)B * maxbands * std::max(1, pl->d.head[0])));
  CK(cudaMalloc(&pl->counter, sizeof(unsigned) * (size_t)B));
  CK(cudaMemset(pl->counter, 0, sizeof(unsigned) * (size_t)B));
  pl->scratch_B = B;
  return IAF_OK;
}

extern "C" {

int iaf_version(void) { return 100; }  // 0.1.0

const char* iaf_strerror(int status) {
  switch (status) {
    case IAF_OK: return "ok";
    case IAF_ERR_BAD_ARG: return "bad argument (null pointer or non-positive size)";
    case IAF_ERR_BAD_SHAPE: return "bad shape (channel counts must divide one another; two heads must be equal)";
    case IAF_ERR_UNSUPPORTED: return "configuration not supported by the B200 kernels";
    case IAF_ERR_CUDA: return "CUDA error (see iaf_last_cuda_error)";
    case IAF_ERR_NOT_PACKED: return "iaf_pack_weights has not been called on this plan";
    case IAF_ERR_NO_DEVICE: return "no CUDA device";
    default: return "unknown status";
  }
}

const char* iaf_last_cuda_error(void) { return g_cuda_err; }

int iaf_plan_create(iaf_plan_t** out, const iaf_desc_t* desc) {
  if (!out || !desc) return IAF_ERR_BAD_ARG;
  *out = nullptr;
  const iaf_desc_t& d = *desc;
  if (d.n_z <= 0 || d.H <= 0 || d.W <= 0) return IAF_ERR_BAD_ARG;
  if (d.variant != IAF_VARIANT_TF && d.variant != IAF_VARIANT_THEANO) return IAF_ERR_BAD_ARG;
  if (d.n_hidden < 0 || d.n_hidden > IAF_MAX_HIDDEN) return IAF_ERR_UNSUPPORTED;
  if (d.n_heads < 1 || d.n_heads > IAF_MAX_HEADS) return IAF_ERR_UNSUPPORTED;
  if (d.nl < IAF_NL_NONE || d.nl > IAF_NL_LEAKYRELU) return IAF_ERR_UNSUPPORTED;
  if (d.path < IAF_PATH_AUTO || d.path > IAF_PATH_TC) return IAF_ERR_BAD_ARG;
  for (int i = 0; i < d.n_hidden; ++i)
    if (d.hidden[i] <= 0) return IAF_ERR_BAD_ARG;
  for (int i = 0; i < d.n_heads; ++i)
    if (d.head[i] <= 0) return IAF_ERR_BAD_ARG;
  if (d.n_heads == 2 && d.head[0] != d.head[1]) return IAF_ERR_BAD_SHAPE;
  if (d.head[0] > 256) return IAF_ERR_UNSUPPORTED;
  {  // ar.py:250,257 / layers.py:116
    int prev = d.n_z;
    for (int i = 0; i < d.n_hidden; ++i) {
      if (prev % d.hidden[i] != 0 && d.hidden[i] % prev != 0) return IAF_ERR_BAD_SHAPE;
      prev = d.hidden[i];
    }
    if (prev % d.head[0] != 0 && d.head[0] % prev != 0) return IAF_ERR_BAD_SHAPE;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return IAF_ERR_NO_DEVICE;
  }
  iaf_plan* pl = new (std::nothrow) iaf_plan();
  if (!pl) return IAF_ERR_BAD_ARG;
  memset(pl, 0, sizeof(*pl));
  pl->d = d;
  // a CUDA failure from here on releases the half-built plan (struct and device buffers) before returning
#define CKP(call)                                                    \
  do {                                                              \
    cudaError_t e_ = (call);                                        \
    if (e_ != cudaSuccess) { iaf_plan_destroy(pl); return cuda_fail(e_, #call); } \
  } while (0)
  CKP(cudaGetDevice(&pl->device));
  pl->n_stages = d.n_hidden + 1;
  int prev = d.n_z;
  for (int j = 0; j < pl->n_stages; ++j) {
    pl->cin[j] = prev;
    if (j < d.n_hidden) {
      pl->cout[j] = d.hidden[j];
      pl->cout_pad[j] = round_up(d.hidden[j], 8);
    } else if (d.n_heads == 2) {
      pl->head_pad = round_up(d.head[0], 4);
      pl->cout[j] = 2 * d.head[0];
      pl->cout_pad[j] = 2 * pl->head_pad;
    } else {
      pl->head_pad = round_up(d.head[0], 8);
      pl->cout[j] = d.head[0];
      pl->cout_pad[j] = pl->head_pad;
    }
    prev = pl->cout[j];
    pl->w_elems[j] = (size_t)IAF_NTAPS * pl->cin[j] * pl->cout_pad[j];
    CKP(cudaMalloc(&pl->w[j], sizeof(float) * pl->w_elems[j]));
    CKP(cudaMalloc(&pl->bias[j], sizeof(float) * pl->cout_pad[j]));
    CKP(cudaMalloc(&pl->padw[j], sizeof(float) * 4 * pl->cout_pad[j]));
  }
#undef CKP
  // SIMT geometry: the largest band that leaves room for two CTAs per SM, else the largest that fits at all
  const size_t kTwo = 100 * 1024, kMax = 225 * 1024;
  int chosen = 0;
  for (int pass = 0; pass < 2 && !chosen; ++pass) {
    for (int div = 1; div <= d.H; div *= 2) {
      int r = (d.H + div - 1) / div;
      size_t smem;
      simt_geometry(pl, r, &smem);
      if (smem <= (pass == 0 ? kTwo : kMax)) { chosen = r; break; }
      if (r == 1) break;
    }
  }
  bool simt_ok = chosen > 0;
  if (simt_ok) simt_geometry(pl, chosen, nullptr);
  pl->simt_ok = simt_ok;

  // tensor-core path
  pl->tc = nullptr;
  const bool tc_ok = iaf_tc_supported(&d);
  int path = d.path;
  if (path == IAF_PATH_AUTO) path = tc_ok ? IAF_PATH_TC : IAF_PATH_SIMT;
  if ((path == IAF_PATH_TC && !tc_ok) || (path == IAF_PATH_SIMT && !simt_ok)) {
    iaf_plan_destroy(pl);
    return IAF_ERR_UNSUPPORTED;
  }
  pl->path = path;
  if (path == IAF_PATH_TC) {
    int st = iaf_tc_plan_create(&pl->tc, &d);
    if (st != IAF_OK) {
      if (st == IAF_ERR_CUDA) cuda_fail(cudaGetLastError(), "iaf_tc_plan_create");
      iaf_plan_destroy(pl);
      return st;
    }
  }
  if (simt_ok) {
    cudaError_t e = iaf_simt_set_smem();
    if (e != cudaSuccess) { iaf_plan_destroy(pl); return cuda_fail(e, "cudaFuncSetAttribute(simt smem)"); }
  }
  *out = pl;
  return IAF_OK;
}

void iaf_plan_destroy(iaf_plan_t* pl) {
  if (!pl) return;
  for (int j = 0; j < IAF_MAX_STAGES; ++j) {
    if (pl->w[j]) cudaFree(pl->w[j]);
    if (pl->bias[j]) cudaFree(pl->bias[j]);
    if (pl->padw[j]) cudaFree(pl->padw[j]);
  }
  if (pl->partial) cudaFree(pl->partial);
  if (pl->counter) cudaFree(pl->counter);
  float* st[] = {pl->st_z, pl->st_ctx, pl->st_zo, pl->st_ls, pl->st_ld};
  for (float* q : st) if (q) cudaFree(q);
  for (int i = 0; i < IAF_NSLOT; ++i) {
    float* ps[] = {pl->ps_z[i], pl->ps_ctx[i], pl->ps_zo[i], pl->ps_ls[i], pl->ps_ld[i]};
    for (float* q : ps) if (q) cudaFree(q);
    if (pl->ev_h2d[i]) cudaEventDestroy(pl->ev_h2d[i]);
    if (pl->ev_cmp[i]) cudaEventDestroy(pl->ev_cmp[i]);
    if (pl->ev_d2h[i]) cudaEventDestroy(pl->ev_d2h[i]);
  }
  if (pl->ev_handoff) cudaEventDestroy(pl->ev_handoff);
  if (pl->s_h2d) cudaStreamDestroy(pl->s_h2d);
  if (pl->s_cmp) cudaStreamDestroy(pl->s_cmp);
  if (pl->s_d2h) cudaStreamDestroy(pl->s_d2h);
  if (pl->tc) iaf_tc_plan_destroy(pl->tc);
  if (pl->bwd) iaf_bwd_plan_destroy(pl->bwd);
  if (pl->rc_zo) cudaFree(pl->rc_zo);
  if (pl->rc_ls) cudaFree(pl->rc_ls);
  for (int j = 0; j < IAF_MAX_HIDDEN; ++j)
    if (pl->rc_h[j]) cudaFree(pl->rc_h[j]);
  if (pl->init_zeros) cudaFree(pl->init_zeros);
  delete pl;
}

// the SIMT packed layout of every stage (iaf_pack.cu), from raw parameters
static int pack_simt(iaf_plan* pl, const float* const* w, const float* const* scale, const float* const* bias,
                     cudaStream_t stream) {
  const iaf_desc_t& d = pl->d;
  const int n_layers = d.n_hidden + d.n_heads;
  IafPackParams pp;
  memset(&pp, 0, sizeof(pp));
  pp.n_layers = n_layers;
  pp.variant = d.variant;
  int max_cout = 0;
  for (int j = 0; j < pl->n_stages; ++j) {
    CK(cudaMemsetAsync(pl->w[j], 0, sizeof(float) * pl->w_elems[j], stream));
    CK(cudaMemsetAsync(pl->bias[j], 0, sizeof(float) * pl->cout_pad[j], stream));
    CK(cudaMemsetAsync(pl->padw[j], 0, sizeof(float) * 4 * pl->cout_pad[j], stream));
  }
  for (int i = 0; i < n_layers; ++i) {
    IafPackLayer& L = pp.layer[i];
    const bool is_head = i >= d.n_hidden;
    const int j = is_head ? d.n_hidden : i;
    L.w = w[i]; L.scale = scale[i]; L.bias = bias[i];
    L.w_out = pl->w[j]; L.bias_out = pl->bias[j]; L.padw_out = pl->padw[j];
    L.cin = pl->cin[j];
    L.cout = is_head ? d.head[i - d.n_hidden] : d.hidden[i];
    L.cout_pad = pl->cout_pad[j];
    L.zerodiag = is_head ? 1 : 0;        // ar.py:388,394 / layers.py:162,166
    L.head_pairs = (is_head && d.n_heads == 2) ? 1 : 0;
    L.head_c = d.head[0];
    L.head_pad = pl->head_pad;
    L.col0 = is_head ? 4 * (i - d.n_hidden) : 0;
    max_cout = std::max(max_cout, L.cout);
  }
  CK(iaf_launch_pack(pp, max_cout, stream));
  pl->launches += 1;
  return IAF_OK;
}

int iaf_pack_weights(iaf_plan_t* pl, const float* const* w, const float* const* scale, const float* const* bias,
                     void* stream_) {
  if (!pl || !w || !scale || !bias) return IAF_ERR_BAD_ARG;
  cudaStream_t stream = (cudaStream_t)stream_;
  const iaf_desc_t& d = pl->d;
  const int n_layers = d.n_hidden + d.n_heads;
  for (int i = 0; i < n_layers; ++i)
    if (!w[i] || !scale[i] || !bias[i]) return IAF_ERR_BAD_ARG;
  { int hs = stream_handoff(pl, stream); if (hs != IAF_OK) return hs; }
  { int st = pack_simt(pl, w, scale, bias, stream); if (st != IAF_OK) return st; }
  if (pl->tc) {
    int st = iaf_tc_pack(pl->tc, w, scale, bias, stream);
    if (st != IAF_OK) return st == IAF_ERR_CUDA ? cuda_fail(cudaGetLastError(), "iaf_tc_pack") : st;
    pl->launches += 1;
  }
  pl->packed = true;
  return IAF_OK;
}

static int run(iaf_plan* pl, int mode, const float* z, const float* ctx, const float* post_mean,
               const float* post_logsd, const float* prior_mean, const float* prior_logsd, float* z_out,
               float* elem_out, float* m_out, float* s_out, float* bc_out, float* persample_out, int B,
               cudaStream_t stream, float* const* hid_out = nullptr) {
  if (!pl->packed) return IAF_ERR_NOT_PACKED;
  if (B <= 0) return IAF_ERR_BAD_ARG;
  { int hs = stream_handoff(pl, stream); if (hs != IAF_OK) return hs; }
  const iaf_desc_t& d = pl->d;
  // a plan the caller pinned to the tensor-core path never downgrades silently (see iaf_plan_path_for_entry)
  if (pl->path == IAF_PATH_TC && pl->d.path == IAF_PATH_TC && !iaf_tc_mode_supported(pl->tc, mode)) return IAF_ERR_UNSUPPORTED;
  if (pl->path == IAF_PATH_TC && iaf_tc_mode_supported(pl->tc, mode)) {
    IafTcArgs a;
    memset(&a, 0, sizeof(a));
    a.mode = mode; a.z = z; a.ctx = ctx; a.post_mean = post_mean; a.post_logsd = post_logsd;
    a.prior_mean = prior_mean; a.prior_logsd = prior_logsd; a.z_out = z_out; a.elem_out = elem_out;
    if (mode == IAF_MODE_MULTICONV) { a.z_out = m_out; a.elem_out = s_out; }  // raw heads travel in the same slots
    a.bc_out = bc_out; a.persample_out = persample_out; a.B = B;
    for (int j = 0; j < d.n_hidden && hid_out; ++j) a.hid_out[j] = hid_out[j];
    int nl = 0;
    int st = iaf_tc_run(pl->tc, &a, stream, &nl);
    if (st == IAF_ERR_CUDA) return cuda_fail(cudaGetLastError(), "iaf_tc_run");
    pl->launches += nl;
    return st;
  }
  if (!pl->simt_ok) return IAF_ERR_UNSUPPORTED;
  int st = ensure_scratch(pl, B);
  if (st != IAF_OK) return st;
  IafSimtParams p;
  memset(&p, 0, sizeof(p));
  p.z = z; p.ctx = ctx; p.post_mean = post_mean; p.post_logsd = post_logsd;
  p.prior_mean = prior_mean; p.prior_logsd = prior_logsd;
  p.z_out = z_out; p.logsd_out = elem_out; p.m_out = m_out; p.s_out = s_out;
  p.bc_out = bc_out; p.persample_out = persample_out;
  p.partial = pl->partial; p.counter = pl->counter;
  for (int j = 0; j < d.n_hidden && hid_out; ++j) p.hid_out[j] = hid_out[j];
  for (int j = 0; j < pl->n_stages; ++j) {
    p.stage[j].w = pl->w[j];
    p.stage[j].bias = pl->bias[j];
    p.stage[j].padw = d.variant == IAF_VARIANT_THEANO ? pl->padw[j] : nullptr;
    p.stage[j].cin = pl->cin[j];
    p.stage[j].cout = pl->cout[j];
    p.stage[j].cout_pad = pl->cout_pad[j];
  }
  p.n_stages = pl->n_stages;
  p.n_heads = d.n_heads; p.head_c = d.head[0]; p.head_pad = pl->head_pad;
  p.B = B; p.C = d.n_z; p.H = d.H; p.W = d.W; p.P = pl->P;
  p.band_rows = pl->band_rows; p.n_bands = pl->n_bands;
  p.flip = d.variant == IAF_VARIANT_THEANO ? 1 : 0;
  p.nl = d.nl; p.mode = mode; p.scale = 0.1f;
  p.bufz_elems = pl->bufz; p.bufa_elems = pl->bufa; p.bufb_elems = pl->bufb;
  CK(iaf_launch_simt(p, pl->smem, stream));
  pl->launches += 1;
  return IAF_OK;
}

int iaf_multiconv_fwd(iaf_plan_t* pl, const float* z, const float* context, float* const* outs, int B,
                      void* stream) {
  if (!pl || !z || !outs || !outs[0]) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !context) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads == 2 && !outs[1]) return IAF_ERR_BAD_ARG;
  return run(pl, IAF_MODE_MULTICONV, z, context, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, outs[0],
             pl->d.n_heads == 2 ? outs[1] : nullptr, nullptr, nullptr, B, (cudaStream_t)stream);
}

int iaf_step_fwd(iaf_plan_t* pl, const float* z, const float* context, float* z_out, float* logsd_out,
                 float* logdet_out, int B, void* stream) {
  if (!pl || !z || !z_out) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !context) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads != 2 || pl->d.head[0] != pl->d.n_z) return IAF_ERR_BAD_SHAPE;
  return run(pl, IAF_MODE_STEP, z, context, nullptr, nullptr, nullptr, nullptr, z_out, logsd_out, nullptr, nullptr,
             nullptr, logdet_out, B, (cudaStream_t)stream);
}

int iaf_layer_fwd(iaf_plan_t* pl, const float* eps, const float* post_mean, const float* post_logsd,
                  const float* prior_mean, const float* prior_logsd, const float* context, float* z_out,
                  float* kl_out, float* kl_bc_out, float* kl_cost_out, int B, void* stream) {
  if (!pl || !eps || !post_mean || !post_logsd || !prior_mean || !prior_logsd || !z_out) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !context) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads != 2 || pl->d.head[0] != pl->d.n_z) return IAF_ERR_BAD_SHAPE;
  return run(pl, IAF_MODE_LAYER, eps, context, post_mean, post_logsd, prior_mean, prior_logsd, z_out, kl_out,
             nullptr, nullptr, kl_bc_out, kl_cost_out, B, (cudaStream_t)stream);
}

int iaf_step_fwd_train(iaf_plan_t* pl, const float* z, const float* context, float* z_out, float* logsd_out,
                       float* logdet_out, float* const* hidden_out, int B, void* stream) {
  if (!pl || !z || !z_out || !logsd_out) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && (!context || !hidden_out)) return IAF_ERR_BAD_ARG;
  for (int j = 0; j < pl->d.n_hidden; ++j)
    if (!hidden_out[j]) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads != 2 || pl->d.head[0] != pl->d.n_z) return IAF_ERR_BAD_SHAPE;
  return run(pl, IAF_MODE_STEP, z, context, nullptr, nullptr, nullptr, nullptr, z_out, logsd_out, nullptr, nullptr,
             nullptr, logdet_out, B, (cudaStream_t)stream, hidden_out);
}

static int run_bwd(iaf_plan* pl, int mode, const float* z, const float* ctx, const float* const* w,
                   const float* const* scale, const float* g_zout, const float* g_logsd, const float* g_logdet,
                   const float* const* g_heads, float* g_z, float* g_ctx, float* const* g_w, float* const* g_scale,
                   float* const* g_bias, int B, cudaStream_t stream, const float* z_out_saved = nullptr,
                   const float* logsd_saved = nullptr, const float* const* hidden_saved = nullptr) {
  if (!pl->packed) return IAF_ERR_NOT_PACKED;
  if (B <= 0) return IAF_ERR_BAD_ARG;
  { int hs = stream_handoff(pl, stream); if (hs != IAF_OK) return hs; }
  const iaf_desc_t& d = pl->d;
  const int n_layers = d.n_hidden + d.n_heads;
  const bool want_params = g_w || g_scale || g_bias;
  if (want_params) {
    if (!w || !scale) return IAF_ERR_BAD_ARG;
    for (int i = 0; i < n_layers; ++i)
      if (!w[i] || !scale[i]) return IAF_ERR_BAD_ARG;
  }
  if (!pl->bwd) {
    int st = iaf_bwd_plan_create(&pl->bwd, &d, pl->cin, pl->cout, pl->cout_pad, pl->head_pad, pl->path == IAF_PATH_TC);
    if (st != IAF_OK) return st == IAF_ERR_CUDA ? cuda_fail(cudaGetLastError(), "iaf_bwd_plan_create") : st;
  }
  IafBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = mode; a.B = B; a.z = z; a.ctx = ctx;
  for (int j = 0; j < pl->n_stages; ++j) {
    a.w_packed[j] = pl->w[j]; a.bias_packed[j] = pl->bias[j]; a.padw_packed[j] = pl->padw[j];
  }
  a.w_raw = w; a.scale_raw = scale;
  a.g_zout = g_zout; a.g_logsd = g_logsd; a.g_logdet = g_logdet;
  if (g_heads) { a.g_heads[0] = g_heads[0]; a.g_heads[1] = d.n_heads == 2 ? g_heads[1] : nullptr; }
  a.g_z = g_z; a.g_ctx = d.n_hidden > 0 ? g_ctx : nullptr;
  a.g_w = g_w; a.g_scale = g_scale; a.g_bias = g_bias;
  a.z_out_saved = z_out_saved; a.logsd_saved = logsd_saved;
  for (int j = 0; j < d.n_hidden && hidden_saved; ++j) a.h_saved[j] = hidden_saved[j];
  a.have_saved = z_out_saved != nullptr;
  if (mode == IAF_MODE_STEP && !z_out_saved && pl->path == IAF_PATH_TC && iaf_tc_mode_supported(pl->tc, IAF_MODE_STEP) &&
      iaf_bwd_plan_uses_tc(pl->bwd)) {
    // a tensor-core plan recomputes z', arw_logsd and the activations with its own forward (one training-forward call)
    // instead of the SIMT layer convs: what iaf_step_fwd_train would have kept
    if (B > pl->rc_B) {
      const size_t hw = (size_t)d.H * d.W;
      if (pl->rc_zo) cudaFree(pl->rc_zo);
      if (pl->rc_ls) cudaFree(pl->rc_ls);
      pl->rc_zo = pl->rc_ls = nullptr;
      for (int j = 0; j < IAF_MAX_HIDDEN; ++j) { if (pl->rc_h[j]) cudaFree(pl->rc_h[j]); pl->rc_h[j] = nullptr; }
      pl->rc_B = 0;
      if (cudaMalloc(&pl->rc_zo, sizeof(float) * B * d.n_z * hw) != cudaSuccess ||
          cudaMalloc(&pl->rc_ls, sizeof(float) * B * d.n_z * hw) != cudaSuccess)
        return cuda_fail(cudaGetLastError(), "recompute scratch");
      for (int j = 0; j < d.n_hidden; ++j)
        if (cudaMalloc(&pl->rc_h[j], sizeof(float) * B * d.hidden[j] * hw) != cudaSuccess)
          return cuda_fail(cudaGetLastError(), "recompute scratch");
      pl->rc_B = B;
    }
    int st = run(pl, IAF_MODE_STEP, z, ctx, nullptr, nullptr, nullptr, nullptr, pl->rc_zo, pl->rc_ls, nullptr, nullptr, nullptr,
                 nullptr, B, stream, pl->rc_h);
    if (st != IAF_OK) return st;
    a.z_out_saved = pl->rc_zo; a.logsd_saved = pl->rc_ls;
    for (int j = 0; j < d.n_hidden; ++j) a.h_saved[j] = pl->rc_h[j];
    a.have_saved = 1;
  }
  int nl = 0;
  int st = iaf_bwd_run(pl->bwd, &a, stream, &nl);
  if (st == IAF_ERR_CUDA) return cuda_fail(cudaGetLastError(), "iaf_bwd_run");
  pl->launches += nl;
  return st;
}

int iaf_step_bwd(iaf_plan_t* pl, const float* z, const float* context, const float* const* w,
                 const float* const* scale, const float* g_z_out, const float* g_logsd, const float* g_logdet,
                 float* g_z, float* g_context, float* const* g_w, float* const* g_scale, float* const* g_bias, int B,
                 void* stream) {
  if (!pl || !z || !g_z_out || !g_z) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !context) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads != 2 || pl->d.head[0] != pl->d.n_z) return IAF_ERR_BAD_SHAPE;
  return run_bwd(pl, IAF_MODE_STEP, z, context, w, scale, g_z_out, g_logsd, g_logdet, nullptr, g_z, g_context, g_w,
                 g_scale, g_bias, B, (cudaStream_t)stream);
}

int iaf_step_bwd_saved(iaf_plan_t* pl, const float* z, const float* z_out, const float* logsd,
                       const float* const* hidden, const float* const* w, const float* const* scale,
                       const float* g_z_out, const float* g_logsd, const float* g_logdet, float* g_z, float* g_context,
                       float* const* g_w, float* const* g_scale, float* const* g_bias, int B, void* stream) {
  if (!pl || !z || !z_out || !logsd || !g_z_out || !g_z) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !hidden) return IAF_ERR_BAD_ARG;
  for (int j = 0; j < pl->d.n_hidden; ++j)
    if (!hidden[j]) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads != 2 || pl->d.head[0] != pl->d.n_z) return IAF_ERR_BAD_SHAPE;
  return run_bwd(pl, IAF_MODE_STEP, z, nullptr, w, scale, g_z_out, g_logsd, g_logdet, nullptr, g_z, g_context, g_w,
                 g_scale, g_bias, B, (cudaStream_t)stream, z_out, logsd, hidden);
}

int iaf_layer_bwd(iaf_plan_t* pl, const float* eps, const float* post_mean, const float* post_logsd,
                  const float* prior_mean, const float* prior_logsd, const float* context, const float* const* w,
                  const float* const* scale, const float* g_z_out, const float* g_kl, const float* g_kl_bc,
                  const float* g_kl_cost, float* g_post_mean, float* g_post_logsd, float* g_prior_mean,
                  float* g_prior_logsd, float* g_eps, float* g_context, float* const* g_w, float* const* g_scale,
                  float* const* g_bias, int B, void* stream) {
  if (!pl || !eps || !post_mean || !post_logsd || !prior_mean || !prior_logsd) return IAF_ERR_BAD_ARG;
  if (!g_post_mean || !g_post_logsd || !g_prior_mean || !g_prior_logsd) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !context) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads != 2 || pl->d.head[0] != pl->d.n_z) return IAF_ERR_BAD_SHAPE;
  if (!pl->packed) return IAF_ERR_NOT_PACKED;
  if (B <= 0) return IAF_ERR_BAD_ARG;
  { int hs = stream_handoff(pl, (cudaStream_t)stream); if (hs != IAF_OK) return hs; }
  const iaf_desc_t& d = pl->d;
  const bool want_params = g_w || g_scale || g_bias;
  if (want_params) {
    if (!w || !scale) return IAF_ERR_BAD_ARG;
    for (int i = 0; i < d.n_hidden + d.n_heads; ++i)
      if (!w[i] || !scale[i]) return IAF_ERR_BAD_ARG;
  }
  if (!pl->bwd) {
    int st = iaf_bwd_plan_create(&pl->bwd, &d, pl->cin, pl->cout, pl->cout_pad, pl->head_pad, pl->path == IAF_PATH_TC);
    if (st != IAF_OK) return st == IAF_ERR_CUDA ? cuda_fail(cudaGetLastError(), "iaf_bwd_plan_create") : st;
  }
  IafBwdArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = IAF_MODE_LAYER; a.B = B; a.z = eps; a.ctx = context;
  for (int j = 0; j < pl->n_stages; ++j) {
    a.w_packed[j] = pl->w[j]; a.bias_packed[j] = pl->bias[j]; a.padw_packed[j] = pl->padw[j];
  }
  a.w_raw = w; a.scale_raw = scale;
  a.post_mean = post_mean; a.post_logsd = post_logsd; a.prior_mean = prior_mean; a.prior_logsd = prior_logsd;
  a.g_zout = g_z_out; a.g_kl = g_kl; a.g_kl_bc = g_kl_bc; a.g_kl_cost = g_kl_cost;
  a.g_post_mean = g_post_mean; a.g_post_logsd = g_post_logsd; a.g_prior_mean = g_prior_mean; a.g_prior_logsd = g_prior_logsd;
  a.g_eps = g_eps;
  a.g_z = nullptr; a.g_ctx = d.n_hidden > 0 ? g_context : nullptr;
  a.g_w = g_w; a.g_scale = g_scale; a.g_bias = g_bias;
  int nl = 0;
  int st = iaf_bwd_run(pl->bwd, &a, (cudaStream_t)stream, &nl);
  if (st == IAF_ERR_CUDA) return cuda_fail(cudaGetLastError(), "iaf_bwd_run");
  pl->launches += nl;
  return st;
}

int iaf_multiconv_fwd_train(iaf_plan_t* pl, const float* z, const float* context, float* const* outs,
                            float* const* hidden_out, int B, void* stream) {
  if (!pl || !z || !outs || !outs[0]) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && (!context || !hidden_out)) return IAF_ERR_BAD_ARG;
  for (int j = 0; j < pl->d.n_hidden; ++j)
    if (!hidden_out[j]) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads == 2 && !outs[1]) return IAF_ERR_BAD_ARG;
  return run(pl, IAF_MODE_MULTICONV, z, context, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, outs[0],
             pl->d.n_heads == 2 ? outs[1] : nullptr, nullptr, nullptr, B, (cudaStream_t)stream, hidden_out);
}

int iaf_multiconv_bwd_saved(iaf_plan_t* pl, const float* z, const float* const* hidden, const float* const* w,
                            const float* const* scale, const float* const* g_outs, float* g_z, float* g_context,
                            float* const* g_w, float* const* g_scale, float* const* g_bias, int B, void* stream) {
  if (!pl || !z || !g_outs || !g_outs[0] || !g_z) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !hidden) return IAF_ERR_BAD_ARG;
  for (int j = 0; j < pl->d.n_hidden; ++j)
    if (!hidden[j]) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads == 2 && !g_outs[1]) return IAF_ERR_BAD_ARG;
  // z_out_saved doubles as the "activations were kept" flag of run_bwd; the multiconv backward never reads it
  return run_bwd(pl, IAF_MODE_MULTICONV, z, nullptr, w, scale, nullptr, nullptr, nullptr, g_outs, g_z, g_context, g_w,
                 g_scale, g_bias, B, (cudaStream_t)stream, z, nullptr, hidden);
}

int iaf_multiconv_bwd(iaf_plan_t* pl, const float* z, const float* context, const float* const* w,
                      const float* const* scale, const float* const* g_outs, float* g_z, float* g_context,
                      float* const* g_w, float* const* g_scale, float* const* g_bias, int B, void* stream) {
  if (!pl || !z || !g_outs || !g_outs[0] || !g_z) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !context) return IAF_ERR_BAD_ARG;
  if (pl->d.n_heads == 2 && !g_outs[1]) return IAF_ERR_BAD_ARG;
  return run_bwd(pl, IAF_MODE_MULTICONV, z, context, w, scale, nullptr, nullptr, nullptr, g_outs, g_z, g_context, g_w,
                 g_scale, g_bias, B, (cudaStream_t)stream);
}

int iaf_multiconv_init(iaf_plan_t* pl, const float* z, const float* context, const float* const* w,
                       const float* const* scale, const float* const* bias, float* const* scale_out,
                       float* const* bias_out, float* const* outs, int* skipped, int B, void* stream_) {
  if (!pl || !z || !w || !scale_out || !bias_out) return IAF_ERR_BAD_ARG;
  const iaf_desc_t& d = pl->d;
  const bool theano = d.variant == IAF_VARIANT_THEANO;
  if (d.n_hidden > 0 && !context) return IAF_ERR_BAD_ARG;
  if (theano && (!scale || !bias)) return IAF_ERR_BAD_ARG;
  if (B <= 0) return IAF_ERR_BAD_ARG;
  const int n_layers = d.n_hidden + d.n_heads;
  for (int i = 0; i < n_layers; ++i) {
    if (!w[i] || !scale_out[i] || !bias_out[i] || scale_out[i] == bias_out[i]) return IAF_ERR_BAD_ARG;
    if (theano && (!scale[i] || !bias[i])) return IAF_ERR_BAD_ARG;
    if (theano && (scale_out[i] == scale[i] || bias_out[i] == bias[i])) return IAF_ERR_BAD_ARG;  // outputs never alias inputs
  }
  if (outs)
    for (int k = 0; k < d.n_heads; ++k)
      if (!outs[k]) return IAF_ERR_BAD_ARG;
  cudaStream_t stream = (cudaStream_t)stream_;
  { int hs = stream_handoff(pl, stream); if (hs != IAF_OK) return hs; }
  // the packed buffers are this pass's scratch: forward and backward entries refuse the plan until it is packed again
  pl->packed = false;
  if (!pl->bwd) {
    int st = iaf_bwd_plan_create(&pl->bwd, &d, pl->cin, pl->cout, pl->cout_pad, pl->head_pad, pl->path == IAF_PATH_TC);
    if (st != IAF_OK) return st == IAF_ERR_CUDA ? cuda_fail(cudaGetLastError(), "iaf_bwd_plan_create") : st;
  }
  // TF: the init branch convolves with l2_normalize(mask o V) alone (layers.py:44-45), i.e. gain exp(0) and bias 0
  const float* zs[IAF_MAX_HIDDEN + IAF_MAX_HEADS];
  if (!theano) {
    int mc = 0;
    for (int j = 0; j < pl->n_stages; ++j) mc = std::max(mc, pl->cout[j]);
    if (!pl->init_zeros && cudaMalloc(&pl->init_zeros, sizeof(float) * mc) != cudaSuccess) {
      pl->init_zeros = nullptr;
      return cuda_fail(cudaGetLastError(), "cudaMalloc(init zeros)");
    }
    CK(cudaMemsetAsync(pl->init_zeros, 0, sizeof(float) * mc, stream));
    for (int i = 0; i < n_layers; ++i) zs[i] = pl->init_zeros;
  }
  { int st = pack_simt(pl, w, theano ? scale : zs, theano ? bias : zs, stream); if (st != IAF_OK) return st; }
  IafInitArgs a;
  memset(&a, 0, sizeof(a));
  a.B = B; a.z = z; a.ctx = context;
  for (int j = 0; j < pl->n_stages; ++j) {
    a.w_packed[j] = pl->w[j]; a.bias_packed[j] = pl->bias[j]; a.padw_packed[j] = pl->padw[j];
  }
  a.scale_in = scale; a.bias_in = bias; a.scale_out = scale_out; a.bias_out = bias_out;
  a.outs = outs; a.skipped = skipped;
  int nl = 0;
  int st = iaf_init_run(pl->bwd, &a, stream, &nl);
  if (st == IAF_ERR_CUDA) return cuda_fail(cudaGetLastError(), "iaf_init_run");
  pl->launches += nl;
  return st;
}

int iaf_step_fwd_host(iaf_plan_t* pl, const float* z_host, const float* context_host, float* z_out_host,
                      float* logsd_out_host, float* logdet_out_host, int B, void* stream_) {
  if (!pl || !z_host || !z_out_host || B <= 0) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !context_host) return IAF_ERR_BAD_ARG;
  cudaStream_t stream = (cudaStream_t)stream_;
  const iaf_desc_t& d = pl->d;
  const size_t hw = (size_t)d.H * d.W;
  const size_t nz = (size_t)B * d.n_z * hw, nc = (size_t)B * (d.n_hidden ? d.hidden[0] : 1) * hw;
  if (B > pl->staging_B) {
    float** st[] = {&pl->st_z, &pl->st_ctx, &pl->st_zo, &pl->st_ls, &pl->st_ld};
    for (float** q : st) { if (*q) cudaFree(*q); *q = nullptr; }
    pl->staging_B = 0;
    CK(cudaMalloc(&pl->st_z, sizeof(float) * nz));
    CK(cudaMalloc(&pl->st_ctx, sizeof(float) * nc));
    CK(cudaMalloc(&pl->st_zo, sizeof(float) * nz));
    CK(cudaMalloc(&pl->st_ls, sizeof(float) * nz));
    CK(cudaMalloc(&pl->st_ld, sizeof(float) * B));
    pl->staging_B = B;
  }
  CK(cudaMemcpyAsync(pl->st_z, z_host, sizeof(float) * nz, cudaMemcpyHostToDevice, stream));
  if (d.n_hidden > 0)
    CK(cudaMemcpyAsync(pl->st_ctx, context_host, sizeof(float) * nc, cudaMemcpyHostToDevice, stream));
  int st = iaf_step_fwd(pl, pl->st_z, pl->st_ctx, pl->st_zo, logsd_out_host ? pl->st_ls : nullptr,
                        logdet_out_host ? pl->st_ld : nullptr, B, stream_);
  if (st != IAF_OK) return st;
  CK(cudaMemcpyAsync(z_out_host, pl->st_zo, sizeof(float) * nz, cudaMemcpyDeviceToHost, stream));
  if (logsd_out_host)
    CK(cudaMemcpyAsync(logsd_out_host, pl->st_ls, sizeof(float) * nz, cudaMemcpyDeviceToHost, stream));
  if (logdet_out_host)
    CK(cudaMemcpyAsync(logdet_out_host, pl->st_ld, sizeof(float) * B, cudaMemcpyDeviceToHost, stream));
  CK(cudaStreamSynchronize(stream));
  return IAF_OK;
}

int iaf_step_submit_host(iaf_plan_t* pl, const float* z_host, const float* context_host, float* z_out_host,
                         float* logsd_out_host, float* logdet_out_host, int B) {
  if (!pl || !z_host || !z_out_host || B <= 0) return IAF_ERR_BAD_ARG;
  if (pl->d.n_hidden > 0 && !context_host) return IAF_ERR_BAD_ARG;
  const iaf_desc_t& d = pl->d;
  const size_t hw = (size_t)d.H * d.W;
  const size_t nz = (size_t)B * d.n_z * hw, nc = (size_t)B * (d.n_hidden ? d.hidden[0] : 1) * hw;
  if (!pl->s_h2d) {
    CK(cudaStreamCreateWithFlags(&pl->s_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&pl->s_cmp, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&pl->s_d2h, cudaStreamNonBlocking));
    for (int i = 0; i < IAF_NSLOT; ++i) {
      CK(cudaEventCreateWithFlags(&pl->ev_h2d[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&pl->ev_cmp[i], cudaEventDisableTiming));
      CK(cudaEventCreateWithFlags(&pl->ev_d2h[i], cudaEventDisableTiming));
    }
  }
  if (B > pl->pipe_B) {
    CK(cudaDeviceSynchronize());
    for (int i = 0; i < IAF_NSLOT; ++i) {
      float** ps[] = {&pl->ps_z[i], &pl->ps_ctx[i], &pl->ps_zo[i], &pl->ps_ls[i], &pl->ps_ld[i]};
      for (float** q : ps) { if (*q) cudaFree(*q); *q = nullptr; }
      CK(cudaMalloc(&pl->ps_z[i], sizeof(float) * nz));
      CK(cudaMalloc(&pl->ps_ctx[i], sizeof(float) * nc));
      CK(cudaMalloc(&pl->ps_zo[i], sizeof(float) * nz));
      CK(cudaMalloc(&pl->ps_ls[i], sizeof(float) * nz));
      CK(cudaMalloc(&pl->ps_ld[i], sizeof(float) * B));
    }
    pl->pipe_B = B;
  }
  const int sl = (int)(pl->submit_idx % IAF_NSLOT);
  const bool reuse = pl->submit_idx >= IAF_NSLOT;
  // copy-in: the slot's previous step must have been computed
  if (reuse) CK(cudaStreamWaitEvent(pl->s_h2d, pl->ev_cmp[sl], 0));
  CK(cudaMemcpyAsync(pl->ps_z[sl], z_host, sizeof(float) * nz, cudaMemcpyHostToDevice, pl->s_h2d));
  if (d.n_hidden > 0)
    CK(cudaMemcpyAsync(pl->ps_ctx[sl], context_host, sizeof(float) * nc, cudaMemcpyHostToDevice, pl->s_h2d));
  CK(cudaEventRecord(pl->ev_h2d[sl], pl->s_h2d));
  // compute: inputs landed, the slot's previous outputs already copied out
  CK(cudaStreamWaitEvent(pl->s_cmp, pl->ev_h2d[sl], 0));
  if (reuse) CK(cudaStreamWaitEvent(pl->s_cmp, pl->ev_d2h[sl], 0));
  int st = iaf_step_fwd(pl, pl->ps_z[sl], pl->ps_ctx[sl], pl->ps_zo[sl], logsd_out_host ? pl->ps_ls[sl] : nullptr,
                        logdet_out_host ? pl->ps_ld[sl] : nullptr, B, (void*)pl->s_cmp);
  if (st != IAF_OK) return st;
  CK(cudaEventRecord(pl->ev_cmp[sl], pl->s_cmp));
  // copy-out
  CK(cudaStreamWaitEvent(pl->s_d2h, pl->ev_cmp[sl], 0));
  CK(cudaMemcpyAsync(z_out_host, pl->ps_zo[sl], sizeof(float) * nz, cudaMemcpyDeviceToHost, pl->s_d2h));
  if (logsd_out_host)
    CK(cudaMemcpyAsync(logsd_out_host, pl->ps_ls[sl], sizeof(float) * nz, cudaMemcpyDeviceToHost, pl->s_d2h));
  if (logdet_out_host)
    CK(cudaMemcpyAsync(logdet_out_host, pl->ps_ld[sl], sizeof(float) * B, cudaMemcpyDeviceToHost, pl->s_d2h));
  CK(cudaEventRecord(pl->ev_d2h[sl], pl->s_d2h));
  pl->submit_idx += 1;
  return IAF_OK;
}

int iaf_host_wait(iaf_plan_t* pl) {
  if (!pl) return IAF_ERR_BAD_ARG;
  if (pl->s_d2h) {
    CK(cudaStreamSynchronize(pl->s_h2d));
    CK(cudaStreamSynchronize(pl->s_cmp));
    CK(cudaStreamSynchronize(pl->s_d2h));
  }
  return IAF_OK;
}

int iaf_plan_path(const iaf_plan_t* pl) { return pl ? pl->path : IAF_ERR_BAD_ARG; }

int iaf_plan_path_for_entry(const iaf_plan_t* pl, int entry) {
  if (!pl || entry < IAF_MODE_MULTICONV || entry > IAF_MODE_LAYER) return IAF_ERR_BAD_ARG;
  if (pl->path == IAF_PATH_TC && iaf_tc_mode_supported(pl->tc, entry)) return IAF_PATH_TC;
  if (pl->path == IAF_PATH_TC && pl->d.path == IAF_PATH_TC) return IAF_ERR_UNSUPPORTED;
  return pl->simt_ok ? IAF_PATH_SIMT : IAF_ERR_UNSUPPORTED;
}
int iaf_plan_bwd_path(iaf_plan_t* pl) {
  if (!pl) return IAF_ERR_BAD_ARG;
  if (!pl->bwd) {
    int st = iaf_bwd_plan_create(&pl->bwd, &pl->d, pl->cin, pl->cout, pl->cout_pad, pl->head_pad, pl->path == IAF_PATH_TC);
    if (st != IAF_OK) return st == IAF_ERR_CUDA ? cuda_fail(cudaGetLastError(), "iaf_bwd_plan_create") : st;
  }
  return iaf_bwd_plan_uses_tc(pl->bwd);
}
uint64_t iaf_plan_launch_count(const iaf_plan_t* pl) { return pl ? pl->launches : 0; }

size_t iaf_plan_algorithmic_bytes(const iaf_plan_t* pl, int B) {
  if (!pl || B <= 0) return 0;
  const iaf_desc_t& d = pl->d;
  const size_t hw = (size_t)d.H * d.W;
  const size_t ctx_c = d.n_hidden ? d.hidden[0] : 0;
  // read z, read context, write z', write per-element arw_logsd, write logdet  (SURVEY 8d)
  return 4 * (size_t)B * hw * (d.n_z + ctx_c + d.n_z + d.n_z) + 4 * (size_t)B;
}

double iaf_plan_algorithmic_flops(const iaf_plan_t* pl, int B) {
  if (!pl || B <= 0) return 0.0;
  const iaf_desc_t& d = pl->d;
  long long nnz = 0;
  int prev = d.n_z;
  for (int i = 0; i < d.n_hidden; ++i) {
    nnz += 4LL * prev * d.hidden[i] + centre_nnz(prev, d.hidden[i], 0);
    prev = d.hidden[i];
  }
  for (int k = 0; k < d.n_heads; ++k) nnz += 4LL * prev * d.head[k] + centre_nnz(prev, d.head[k], 1);
  return 2.0 * B * d.H * d.W * (double)nnz;
}

}  // extern "C"
