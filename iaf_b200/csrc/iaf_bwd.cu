// Backward of the masked-AR stack and of the fused IAF step (SURVEY 8f-4): exact-fp32 SIMT kernels.
//
// What the reference gets from theano.grad / tf.gradients over
//   ar.multiconv2d (graphy/nodes/ar.py:396-416) / ar_multiconv2d (tf_utils/layers.py:158-166)
//   + the affine update (models.py:282-285, tf_train.py:70-72)
// including the gradient through the in-graph weight normalisation (ar.py:267-281,312-321; layers.py:53-60) and the
// mask (so masked taps receive exactly zero gradient: the contract ar.py:369-373 `postup` re-imposes after each
// optimiser step).
//
// Schedule (layer at a time, activations in HBM, all in the packed weight layout of iaf_pack.cu):
//   1. forward recompute  h_{j+1} = nl(conv_j(h_j) + b (+ctx))            iaf_lconv_kernel<fwd>
//   2. heads + affine backward: (g_z', g_logsd, g_logdet) -> g_m, g_s, direct g_z    iaf_bwd_affine_kernel
//   3. for j = heads .. 0:  dW_j = corr(h_j, G_j)                          iaf_bwd_wgrad_kernel (+ reduce)
//                           G_{j-1} = convT(G_j, W_j) * nl'(h_j)           iaf_lconv_kernel<bwd>
//   4. dW -> (dV, dg) through mask and weight norm                          iaf_bwd_wnorm_kernel
// Orientation: as in iaf_simt.cu everything is computed in the TF form (taps (0,0)c (0,+1) (+1,-1) (+1,0) (+1,+1));
// the Theano variant is the same computation on the point-reflected image (pixel p <-> HW-1-p on every global
// load/store), its pad channel a position-dependent bias whose gradient is a masked sum of G.
// Reductions use fixed-order partial sums (no float atomics): results are run-to-run deterministic.
// The data-dependent initialisation (iaf_multiconv_init, iaf_init_run at the end) also lives here: it runs the stack
// layer at a time on the same forward layer conv, then per-channel statistics, new parameters and normalised outputs.
#include "iaf_bwd.h"
#include "iaf_tc.h"

#define BW_THREADS 256
#define BW_PX 8
#define BW_CT 8

enum { EPI_FWD_HIDDEN = 0, EPI_FWD_HEADS = 1, EPI_BWD_HIDDEN = 2, EPI_BWD_Z = 3 };

// Division by a run-time constant in the staging / epilogue loops.  Default: the plain `/` (a ~25-instruction sequence
// per quotient, two or three per staged element).  -DBW_FASTDIV (development variant, emulation-tested in
// tests/test_emu_kernels.py, not yet timed on the GPU): multiply-high by a per-thread precomputed reciprocal.
struct BwDiv {
  int d;
  unsigned m;
};
__device__ __forceinline__ BwDiv bw_mkdiv(int d) {
  BwDiv f;
  f.d = d;
#ifdef BW_FASTDIV
  f.m = d > 1 ? (unsigned)((1ull << 32) / (unsigned)d) + 1u : 0u;  // floor(2^32 / d) + 1: quotient at most one too large
#else
  f.m = 0u;
#endif
  return f;
}
__device__ __forceinline__ int bw_div(int s, const BwDiv& f) {  // 0 <= s < 2^31
#ifdef BW_FASTDIV
  if (f.d == 1) return s;
  int q = (int)__umulhi((unsigned)s, f.m);
  if (s - q * f.d < 0) --q;
  return q;
#else
  return s / f.d;
#endif
}

// ------------------------------------------------------------------------------------------
// layer convolution, global -> global.  out[n, co, p] = epi( sum_t sum_ci in[n, ci, p +/- d_t] * w[t][ci][co] )
// ------------------------------------------------------------------------------------------
struct IafLconvParams {
  const float* in;     // [B][in_planes][HW]
  const float* w;      // [5][cin][ncol]
  const float* bias;   // fwd: [ncol]
  const float* padw;   // fwd, Theano: [4][ncol]; else nullptr
  const float* ctx;    // fwd, first hidden layer: [B][nout][HW]; else nullptr
  const float* hprev;  // EPI_BWD_HIDDEN: activations h_j [B][nout][HW] (nl' is evaluated from the output of nl)
  float* out;          // [B][out_planes][HW]
  int B, H, W, cin, in_planes, nout, ncol, out_planes;
  int bwd, epi, nl, flip;
  int RB, n_bands, nseg, P, nctb, n_cblk, CK;
};

__device__ __forceinline__ float bw_apply_nl(float v, int nl) {
  switch (nl) {
    case IAF_NL_ELU: return v < 0.f ? expm1f(v) : v;
    case IAF_NL_SOFTPLUS: return v > 0.f ? v + log1pf(expf(-v)) : log1pf(expf(v));
    case IAF_NL_RELU: return v >= 0.f ? v : 0.f;
    case IAF_NL_TANH: return tanhf(v);
    case IAF_NL_LEAKYRELU: return v < 0.f ? 0.01f * v : v;
    default: return v;
  }
}
// d nl(a) / d a as a function of h = nl(a)
__device__ __forceinline__ float bw_nl_grad(float h, int nl) {
  switch (nl) {
    case IAF_NL_ELU: return h > 0.f ? 1.f : h + 1.f;
    case IAF_NL_SOFTPLUS: return 1.f - expf(-h);
    case IAF_NL_RELU: return h > 0.f ? 1.f : 0.f;
    case IAF_NL_TANH: return 1.f - h * h;
    case IAF_NL_LEAKYRELU: return h < 0.f ? 0.01f : 1.f;
    default: return 1.f;
  }
}

#define BW_TAP(T, A, OFF)                                                                   \
  {                                                                                         \
    const float4 wa = *reinterpret_cast<const float4*>(wrow + (T) * ncolb);                 \
    const float4 wb = *reinterpret_cast<const float4*>(wrow + (T) * ncolb + 4);             \
    _Pragma("unroll") for (int j = 0; j < BW_PX; ++j) {                                     \
      const float a = A[j + (OFF)];                                                         \
      acc[j][0] = fmaf(a, wa.x, acc[j][0]); acc[j][1] = fmaf(a, wa.y, acc[j][1]);           \
      acc[j][2] = fmaf(a, wa.z, acc[j][2]); acc[j][3] = fmaf(a, wa.w, acc[j][3]);           \
      acc[j][4] = fmaf(a, wb.x, acc[j][4]); acc[j][5] = fmaf(a, wb.y, acc[j][5]);           \
      acc[j][6] = fmaf(a, wb.z, acc[j][6]); acc[j][7] = fmaf(a, wb.w, acc[j][7]);           \
    }                                                                                       \
  }

template <bool BWD>
__global__ void __launch_bounds__(BW_THREADS) iaf_lconv_kernel(const __grid_constant__ IafLconvParams p) {
  // [CK][RB+1][P] activations, then [CK][5][ncolb] weights of this CTA's column block.  (The first version read the
  // weights with __ldg inside the channel loop: ncu showed the warps waiting on those loads, long-scoreboard stalls
  // 3-5 per issued instruction and the FMA pipe 15-25 % busy; staged copies are read with broadcast LDS.128.)
  IAF_DYN_SMEM(float, sm);
  const int tid = threadIdx.x;
  const int H = p.H, W = p.W, HW = H * W, P = p.P;
  int bid = blockIdx.x;
  const int cblk = bid % p.n_cblk; bid /= p.n_cblk;
  const int band = bid % p.n_bands;
  const int n = bid / p.n_bands;
  const int r0 = band * p.RB;
  const int R = min(p.RB, H - r0);
  const int rows = p.RB + 1;
  const int plane = rows * P;

  // this thread's 8 px x 8 channel tile
  const int ctl = tid % p.nctb;
  const int t2 = tid / p.nctb;
  const int seg = t2 % p.nseg;
  const int yl = t2 / p.nseg;
  const int ct = cblk * p.nctb + ctl;
  const bool active = (yl < R) && (ct * BW_CT < p.ncol);

  float acc[BW_PX][BW_CT];
#pragma unroll
  for (int j = 0; j < BW_PX; ++j)
#pragma unroll
    for (int c = 0; c < BW_CT; ++c) acc[j][c] = 0.f;

  const int ncolb = p.nctb * BW_CT;
  float* sw = sm + (size_t)p.CK * plane;
  const BwDiv dPlane = bw_mkdiv(plane), dP = bw_mkdiv(P), dW = bw_mkdiv(W), dNb4 = bw_mkdiv(ncolb >> 2),
              dNb20 = bw_mkdiv((ncolb >> 2) * IAF_NTAPS);
  // smem row slot l holds image row r0 + l (fwd: rows y, y+1) or r0 - 1 + l (bwd: rows y-1, y); column c holds x = c - 1
  const int row_base = BWD ? r0 - 1 : r0;
  const int slotA = BWD ? yl + 1 : yl;   // row y
  const int slotB = BWD ? yl : yl + 1;   // row y +/- 1

  for (int c0 = 0; c0 < p.cin; c0 += p.CK) {
    const int ck = min(p.CK, p.cin - c0);
    __syncthreads();  // the previous chunk has been consumed
    // global loads are issued in batches of 8 before their shared-memory stores, so their latencies overlap
    for (int i0 = tid; i0 < ck * plane; i0 += BW_THREADS * 8) {
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = i0 + k * BW_THREADS;
        const int c = bw_div(i, dPlane);
        const int rem = i - c * plane;
        const int l = bw_div(rem, dP);
        const int col = rem - l * P;
        const int y = row_base + l, x = col - 1;
        v[k] = 0.f;
        if (i < ck * plane && y >= 0 && y < H && x >= 0 && x < W) {
          const int pix = y * W + x;
          v[k] = __ldg(p.in + ((size_t)n * p.in_planes + c0 + c) * HW + (p.flip ? HW - 1 - pix : pix));
        }
      }
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int i = i0 + k * BW_THREADS;
        if (i < ck * plane) sm[i] = v[k];
      }
    }
    {
      const int nb4 = ncolb >> 2;  // float4 groups per (channel, tap) row; ncol and ncolb are multiples of 8
      for (int i = tid; i < ck * IAF_NTAPS * nb4; i += BW_THREADS) {
        const int c = bw_div(i, dNb20);
        const int r2 = i - c * nb4 * IAF_NTAPS;
        const int t = bw_div(r2, dNb4);
        const int c4 = r2 - t * nb4;
        const int gcol = cblk * ncolb + c4 * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (gcol < p.ncol) v = __ldg(reinterpret_cast<const float4*>(p.w + ((size_t)t * p.cin + c0 + c) * p.ncol + gcol));
        *reinterpret_cast<float4*>(sw + ((size_t)c * IAF_NTAPS + t) * ncolb + c4 * 4) = v;
      }
    }
    __syncthreads();
    if (active) {
      const float* aAp = sm + slotA * P + seg * BW_PX;  // cols x0-1 .. x0+8
      const float* aBp = sm + slotB * P + seg * BW_PX;
      const float* wrow = sw + ctl * BW_CT;
      for (int c = 0; c < ck; ++c) {
        float a0[BW_PX + 2], a1[BW_PX + 2];
#pragma unroll
        for (int j = 0; j < BW_PX + 2; ++j) { a0[j] = aAp[j]; a1[j] = aBp[j]; }
        if (!BWD) {
          BW_TAP(0, a0, 1)  // ( 0, 0)
          BW_TAP(1, a0, 2)  // ( 0,+1)
          BW_TAP(2, a1, 0)  // (+1,-1)
          BW_TAP(3, a1, 1)  // (+1, 0)
          BW_TAP(4, a1, 2)  // (+1,+1)
        } else {            // transposed conv: the tap that read p + d now scatters to p - d
          BW_TAP(0, a0, 1)
          BW_TAP(1, a0, 0)
          BW_TAP(2, a1, 2)
          BW_TAP(3, a1, 1)
          BW_TAP(4, a1, 0)
        }
        aAp += plane;
        aBp += plane;
        wrow += IAF_NTAPS * ncolb;
      }
    }
  }
  // ---- epilogue through shared memory: the register tile (8 px x 8 channels per thread) would store 4 bytes per lane
  // 32 bytes apart; transposing it through smem lets consecutive lanes touch consecutive pixels of one channel, so the
  // output stores and the context / activation loads of the epilogue are fully coalesced
  const int NCS = ncolb + 4;  // tile row stride: [pixel][channel], 16-byte aligned rows
  __syncthreads();            // every thread is done reading the staged chunk
  if (active) {
#pragma unroll
    for (int j = 0; j < BW_PX; ++j) {
      const int x = seg * BW_PX + j;
      if (x >= W) continue;
      float* tp = sm + (size_t)(yl * W + x) * NCS + ctl * BW_CT;
      *reinterpret_cast<float4*>(tp) = make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]);
      *reinterpret_cast<float4*>(tp + 4) = make_float4(acc[j][4], acc[j][5], acc[j][6], acc[j][7]);
    }
  }
  __syncthreads();
  const int npix = R * W;
  const BwDiv dNpix = bw_mkdiv(npix);
  for (int i = tid; i < ncolb * npix; i += BW_THREADS) {
    const int cl = bw_div(i, dNpix), pos = i - cl * npix;
    const int co = cblk * ncolb + cl;
    if (co >= p.nout) continue;
    const int ylp = bw_div(pos, dW), x = pos - ylp * W;
    const int y = r0 + ylp;
    const bool byH = (y == H - 1), bx0 = (x == 0), bxW = (x == W - 1);
    const int pix = y * W + x;
    const int gp = p.flip ? HW - 1 - pix : pix;
    float v = sm[(size_t)pos * NCS + cl];
    const size_t o = ((size_t)n * p.out_planes + co) * HW + gp;
    if (p.epi == EPI_FWD_HIDDEN || p.epi == EPI_FWD_HEADS) {
      v += __ldg(p.bias + co);
      if (p.padw) {  // pad channel = 1 where the tap falls outside the image (conv.py:77-83)
        if (bxW) v += __ldg(p.padw + co);
        if (byH || bx0) v += __ldg(p.padw + p.ncol + co);
        if (byH) v += __ldg(p.padw + 2 * p.ncol + co);
        if (byH || bxW) v += __ldg(p.padw + 3 * p.ncol + co);
      }
      if (p.epi == EPI_FWD_HIDDEN) {
        if (p.ctx) v += __ldg(p.ctx + o);  // out_planes == nout for hidden layers
        v = bw_apply_nl(v, p.nl);
      }
      p.out[o] = v;
    } else if (p.epi == EPI_BWD_HIDDEN) {
      p.out[o] = v * bw_nl_grad(__ldg(p.hprev + o), p.nl);
    } else {  // EPI_BWD_Z: the direct term exp(-arw_logsd) * g_z' is already there
      p.out[o] = p.out[o] + v;
    }
  }
}

// ------------------------------------------------------------------------------------------
// wT[t][k][ci] = w[t][ci][k]  (k < kin, ci < cin; zero padded to cin_pad columns)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BW_THREADS) iaf_bwd_transpose_kernel(const float* w, float* wT, int cin, int ncol, int kin,
                                                                         int cin_pad) {
  const int total = IAF_NTAPS * kin * cin_pad;
  for (int i = blockIdx.x * BW_THREADS + threadIdx.x; i < total; i += gridDim.x * BW_THREADS) {
    const int ci = i % cin_pad;
    const int k = (i / cin_pad) % kin;
    const int t = i / (cin_pad * kin);
    wT[i] = (ci < cin && k < ncol) ? w[((size_t)t * cin + ci) * ncol + k] : 0.f;
  }
}

// ------------------------------------------------------------------------------------------
// heads: packed column of (head k, channel c).  Two heads are interleaved in groups of 4 (iaf_pack.cu).
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ int bw_head_col(int n_heads, int k, int c) { return n_heads == 2 ? ((c >> 2) * 8 + 4 * k + (c & 3)) : c; }

// step: hb holds the raw heads (m, s) on entry and (g_m, g_s) on exit; g_z receives the direct term
struct IafAffineBwdParams {
  const float* z; const float* g_zout; const float* g_logsd; const float* g_logdet;
  const float* z_out; const float* logsd;  // kept by the training forward; when given, hb is write-only
  float* hb; float* g_z;
  int B, C, HW, cp, head_pad;
  float scale;
};
__global__ void __launch_bounds__(BW_THREADS) iaf_bwd_affine_kernel(const __grid_constant__ IafAffineBwdParams p) {
  const size_t total = (size_t)p.B * p.head_pad * p.HW;
  for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < total; i += (size_t)gridDim.x * BW_THREADS) {
    const int gp = (int)(i % p.HW);
    const int c = (int)((i / p.HW) % p.head_pad);
    const int n = (int)(i / ((size_t)p.HW * p.head_pad));
    const int mcol = (c >> 2) * 8 + (c & 3), scol = mcol + 4;
    const size_t om = ((size_t)n * p.cp + mcol) * p.HW + gp, os = ((size_t)n * p.cp + scol) * p.HW + gp;
    if (c >= p.C) {  // padding columns of the packed heads carry no gradient
      p.hb[om] = 0.f;
      p.hb[os] = 0.f;
      continue;
    }
    const size_t e = ((size_t)n * p.C + c) * p.HW + gp;
    // z' = (z - scale*m) * exp(-scale*s); arw_logsd = scale*s; logdet = -sum(arw_logsd)   (models.py:282-285)
    float ex, zn;
    if (p.z_out) {
      ex = expf(-__ldg(p.logsd + e));
      zn = __ldg(p.z_out + e);
    } else {
      const float m = p.hb[om], s = p.hb[os];
      ex = expf(-p.scale * s);
      zn = (__ldg(p.z + e) - p.scale * m) * ex;
    }
    const float gzo = __ldg(p.g_zout + e);
    float gs = -p.scale * zn * gzo;
    if (p.g_logsd) gs += p.scale * __ldg(p.g_logsd + e);
    if (p.g_logdet) gs -= p.scale * __ldg(p.g_logdet + n);
    p.hb[om] = -p.scale * ex * gzo;
    p.hb[os] = gs;
    p.g_z[e] = ex * gzo;
  }
}

// fused layer (tf_train.py:56-85 / models.py:273-298), elementwise parts of its backward:
//   pre:    z0 = post_mean + exp(post_logsd) * eps                                  (the sample the stack sees)
//   affine: gkl = g_kl + g_kl_bc[b,c] + g_kl_cost[b];  d = z' - prior_mean;  E = exp(-2 prior_logsd)
//           G_z' = g_z' + gkl d E,  G_logsd = gkl  ->  g_m, g_s, direct g_z0 as in the step;
//           g_prior_mean = -gkl d E,  g_prior_logsd = gkl (1 - d^2 E)
//   post:   g_post_mean = g_z0;  g_post_logsd = g_z0 exp(post_logsd) eps - gkl;  g_eps = g_z0 exp(post_logsd) - gkl eps
struct IafLayerBwdParams {
  const float* eps; const float* post_mean; const float* post_logsd; const float* prior_mean; const float* prior_logsd;
  const float* g_zout; const float* g_kl; const float* g_kl_bc; const float* g_kl_cost;
  float* z0; float* hb; float* g_z0;
  float* g_post_mean; float* g_post_logsd; float* g_prior_mean; float* g_prior_logsd; float* g_eps;
  int B, C, HW, cp, head_pad;
  float scale;
};
__device__ __forceinline__ float bw_gkl(const IafLayerBwdParams& p, size_t e, int n, int c) {
  float g = 0.f;
  if (p.g_kl) g += __ldg(p.g_kl + e);
  if (p.g_kl_bc) g += __ldg(p.g_kl_bc + (size_t)n * p.C + c);
  if (p.g_kl_cost) g += __ldg(p.g_kl_cost + n);
  return g;
}
__global__ void __launch_bounds__(BW_THREADS) iaf_bwd_layer_pre_kernel(const __grid_constant__ IafLayerBwdParams p) {
  const size_t total = (size_t)p.B * p.C * p.HW;
  for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < total; i += (size_t)gridDim.x * BW_THREADS)
    p.z0[i] = fmaf(expf(__ldg(p.post_logsd + i)), __ldg(p.eps + i), __ldg(p.post_mean + i));
}
__global__ void __launch_bounds__(BW_THREADS) iaf_bwd_layer_affine_kernel(const __grid_constant__ IafLayerBwdParams p) {
  const size_t total = (size_t)p.B * p.head_pad * p.HW;
  for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < total; i += (size_t)gridDim.x * BW_THREADS) {
    const int gp = (int)(i % p.HW);
    const int c = (int)((i / p.HW) % p.head_pad);
    const int n = (int)(i / ((size_t)p.HW * p.head_pad));
    const int mcol = (c >> 2) * 8 + (c & 3), scol = mcol + 4;
    const size_t om = ((size_t)n * p.cp + mcol) * p.HW + gp, os = ((size_t)n * p.cp + scol) * p.HW + gp;
    if (c >= p.C) {
      p.hb[om] = 0.f;
      p.hb[os] = 0.f;
      continue;
    }
    const size_t e = ((size_t)n * p.C + c) * p.HW + gp;
    const float m = p.hb[om], s = p.hb[os];
    const float ex = expf(-p.scale * s);
    const float zn = (p.z0[e] - p.scale * m) * ex;
    const float gkl = bw_gkl(p, e, n, c);
    const float d = zn - __ldg(p.prior_mean + e);
    const float E = expf(-2.0f * __ldg(p.prior_logsd + e));
    float gzo = gkl * d * E;
    if (p.g_zout) gzo += __ldg(p.g_zout + e);
    p.g_prior_mean[e] = -gkl * d * E;
    p.g_prior_logsd[e] = gkl * (1.0f - d * d * E);
    p.hb[om] = -p.scale * ex * gzo;
    p.hb[os] = -p.scale * zn * gzo + p.scale * gkl;
    p.g_z0[e] = ex * gzo;
  }
}
__global__ void __launch_bounds__(BW_THREADS) iaf_bwd_layer_post_kernel(const __grid_constant__ IafLayerBwdParams p) {
  const size_t total = (size_t)p.B * p.C * p.HW;
  for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < total; i += (size_t)gridDim.x * BW_THREADS) {
    const int c = (int)((i / p.HW) % p.C);
    const int n = (int)(i / ((size_t)p.HW * p.C));
    const float gkl = bw_gkl(p, i, n, c);
    const float gz = p.g_z0[i];
    const float sd = expf(__ldg(p.post_logsd + i)), ep = __ldg(p.eps + i);
    p.g_post_mean[i] = gz;
    p.g_post_logsd[i] = gz * sd * ep - gkl;
    if (p.g_eps) p.g_eps[i] = gz * sd - gkl * ep;
  }
}

// multiconv: the caller's head gradients -> packed column order; g_z starts at zero
struct IafScatterParams {
  const float* g0; const float* g1;
  float* hb; float* g_z;
  int B, C, HW, cp, head_pad, n_heads, n_z;
};
__global__ void __launch_bounds__(BW_THREADS) iaf_bwd_scatter_kernel(const __grid_constant__ IafScatterParams p) {
  const size_t total = (size_t)p.B * p.cp * p.HW;
  for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < total; i += (size_t)gridDim.x * BW_THREADS) {
    const int gp = (int)(i % p.HW);
    const int col = (int)((i / p.HW) % p.cp);
    const int n = (int)(i / ((size_t)p.HW * p.cp));
    int k = 0, c = col;
    if (p.n_heads == 2) { k = (col >> 2) & 1; c = (col >> 3) * 4 + (col & 3); }
    float v = 0.f;
    if (c < p.C) v = __ldg((k ? p.g1 : p.g0) + ((size_t)n * p.C + c) * p.HW + gp);
    p.hb[i] = v;
  }
  const size_t tz = (size_t)p.B * p.n_z * p.HW;
  for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < tz; i += (size_t)gridDim.x * BW_THREADS) p.g_z[i] = 0.f;
}

// ------------------------------------------------------------------------------------------
// weight gradient: part[g][t][ci][col] = sum over this CTA's (sample, band) units of x[ci, p + d_t] * G[col, p],
// plus the bias and pad-channel column sums.  CTA tile 64 ci x 64 col, thread tile 4 x 4 x 5 taps.
// ------------------------------------------------------------------------------------------
#define WG_T 64
#define WG_S 68  // smem row stride (floats): 16-byte aligned float4 reads, 4-way conflicts only on the staging stores
struct IafWgradParams {
  const float* x;   // [B][x_planes][HW]  layer input
  const float* g;   // [B][g_planes][HW]  gradient at the layer's pre-activation output
  float* part;      // [NG][5*cin*ncol + 5*ncol]
  int B, H, W, cin, x_planes, ncol, g_planes;
  int flip, RB, n_bands, NG, n_cib, n_colb, PW;
};
__global__ void __launch_bounds__(BW_THREADS, 2) iaf_bwd_wgrad_kernel(const __grid_constant__ IafWgradParams p) {
  IAF_DYN_SMEM(float, sm);
  const int tid = threadIdx.x;
  const int H = p.H, W = p.W, HW = H * W, PW = p.PW;
  const int xpos = (p.RB + 1) * PW;  // staged x positions: rows r0 .. r0+RB, cols -1 .. W
  const int gpos = p.RB * W;
  const size_t buf_floats = (size_t)(xpos + gpos) * WG_S;  // one stage: Xs [xpos][WG_S] then Gs [gpos][WG_S]
  const BwDiv dPW = bw_mkdiv(PW), dWg = bw_mkdiv(W);
  int bid = blockIdx.x;
  const int colb = bid % p.n_colb; bid /= p.n_colb;
  const int cib = bid % p.n_cib;
  const int g = bid / p.n_cib;
  const int ti = tid >> 4, tj = tid & 15;
  const bool side = (cib == 0 && ti == 0);  // these threads also own the bias / pad-channel sums of their 4 columns

  float acc[IAF_NTAPS][4][4];
#pragma unroll
  for (int t = 0; t < IAF_NTAPS; ++t)
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) acc[t][a][b] = 0.f;
  float sb[5][4];
#pragma unroll
  for (int t = 0; t < 5; ++t)
#pragma unroll
    for (int b = 0; b < 4; ++b) sb[t][b] = 0.f;

  // Asynchronous, double-buffered staging (cp.async, 4 bytes per element because the copy transposes [channel][pixel] ->
  // [pixel][channel]): unit u+NG lands while unit u is being contracted.  Lane mapping inside a warp: 4 channels x 8
  // consecutive pixels, i.e. four 32-byte global segments per warp-copy and 32 distinct shared-memory banks (row stride
  // WG_S = 68 = 4 mod 32).  The first version staged with load -> store loops and spent about half its time waiting
  // (ncu: FMA pipe 35-38 % busy, 1.1 M staging bank conflicts).
  auto stage = [&](int u, float* buf) {
    const int n = u / p.n_bands, band = u % p.n_bands;
    const int r0 = band * p.RB;
    const int R = min(p.RB, H - r0);
    float* Xs = buf;
    float* Gs = buf + (size_t)xpos * WG_S;
    const int nx = ((xpos + 7) >> 3) * (WG_T / 4) * 32;
    for (int i = tid; i < nx; i += BW_THREADS) {
      const int c_lo = i & 3, p_lo = (i >> 2) & 7, rest = i >> 5;
      const int c = (rest % (WG_T / 4)) * 4 + c_lo, pos = (rest / (WG_T / 4)) * 8 + p_lo;
      if (pos >= xpos) continue;
      const int l = bw_div(pos, dPW), col = pos - l * PW;
      const int y = r0 + l, x = col - 1;
      const int ci = cib * WG_T + c;
      const bool valid = ci < p.cin && l <= R && y < H && x >= 0 && x < W;
      const int pix = valid ? y * W + x : 0;
      const float* src = valid ? p.x + ((size_t)n * p.x_planes + ci) * HW + (p.flip ? HW - 1 - pix : pix) : p.x;
      iaf_cp_async4(Xs + (size_t)pos * WG_S + c, src, valid);
    }
    const int ng = ((gpos + 7) >> 3) * (WG_T / 4) * 32;
    for (int i = tid; i < ng; i += BW_THREADS) {
      const int c_lo = i & 3, p_lo = (i >> 2) & 7, rest = i >> 5;
      const int c = (rest % (WG_T / 4)) * 4 + c_lo, pos = (rest / (WG_T / 4)) * 8 + p_lo;
      if (pos >= gpos) continue;
      const int l = bw_div(pos, dWg), x = pos - l * W;
      const int col = colb * WG_T + c;
      const bool valid = col < p.g_planes && l < R;
      const int pix = valid ? (r0 + l) * W + x : 0;
      const float* src = valid ? p.g + ((size_t)n * p.g_planes + col) * HW + (p.flip ? HW - 1 - pix : pix) : p.g;
      iaf_cp_async4(Gs + (size_t)pos * WG_S + c, src, valid);
    }
    iaf_cp_async_commit();
  };

  const int units = p.B * p.n_bands;
  if (g < units) stage(g, sm);
  int it = 0;
  for (int u = g; u < units; u += p.NG, ++it) {
    const int un = u + p.NG;
    if (un < units) {
      stage(un, sm + (size_t)((it + 1) & 1) * buf_floats);
      iaf_cp_async_wait<1>();  // everything but the newest group: unit u has landed
    } else {
      iaf_cp_async_wait<0>();
    }
    __syncthreads();
    const float* Xs = sm + (size_t)(it & 1) * buf_floats;
    const float* Gs = Xs + (size_t)xpos * WG_S;
    const int r0 = (u % p.n_bands) * p.RB;
    const int R = min(p.RB, H - r0);
    for (int l = 0; l < R; ++l) {
      const bool byH = (r0 + l == H - 1);
      for (int x = 0; x < W; ++x) {
        const float4 gv = *reinterpret_cast<const float4*>(Gs + (l * W + x) * WG_S + tj * 4);
        const float* xa = Xs + (l * PW + x + 1) * WG_S + ti * 4;         // (y, x)
        const float* xb = Xs + ((l + 1) * PW + x) * WG_S + ti * 4;       // (y+1, x-1)
        const float4 x0 = *reinterpret_cast<const float4*>(xa);
        const float4 x1 = *reinterpret_cast<const float4*>(xa + WG_S);
        const float4 x2 = *reinterpret_cast<const float4*>(xb);
        const float4 x3 = *reinterpret_cast<const float4*>(xb + WG_S);
        const float4 x4 = *reinterpret_cast<const float4*>(xb + 2 * WG_S);
        const float gg[4] = {gv.x, gv.y, gv.z, gv.w};
        const float xx[IAF_NTAPS][4] = {{x0.x, x0.y, x0.z, x0.w}, {x1.x, x1.y, x1.z, x1.w}, {x2.x, x2.y, x2.z, x2.w},
                                        {x3.x, x3.y, x3.z, x3.w}, {x4.x, x4.y, x4.z, x4.w}};
#pragma unroll
        for (int t = 0; t < IAF_NTAPS; ++t)
#pragma unroll
          for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int b = 0; b < 4; ++b) acc[t][a][b] = fmaf(xx[t][a], gg[b], acc[t][a][b]);
        if (side) {
          const bool bx0 = (x == 0), bxW = (x == W - 1);
          const float f1 = bxW ? 1.f : 0.f, f2 = (byH || bx0) ? 1.f : 0.f, f3 = byH ? 1.f : 0.f, f4 = (byH || bxW) ? 1.f : 0.f;
#pragma unroll
          for (int b = 0; b < 4; ++b) {
            sb[0][b] += gg[b];
            sb[1][b] = fmaf(f1, gg[b], sb[1][b]);
            sb[2][b] = fmaf(f2, gg[b], sb[2][b]);
            sb[3][b] = fmaf(f3, gg[b], sb[3][b]);
            sb[4][b] = fmaf(f4, gg[b], sb[4][b]);
          }
        }
      }
    }
    __syncthreads();  // this buffer is refilled by the stage issued in the next iteration
  }

  const size_t nw = (size_t)IAF_NTAPS * p.cin * p.ncol;
  float* out = p.part + (size_t)g * (nw + 5 * (size_t)p.ncol);
#pragma unroll
  for (int t = 0; t < IAF_NTAPS; ++t)
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int ci = cib * WG_T + ti * 4 + a;
      if (ci >= p.cin) continue;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int col = colb * WG_T + tj * 4 + b;
        if (col < p.ncol) out[((size_t)t * p.cin + ci) * p.ncol + col] = acc[t][a][b];
      }
    }
  if (side) {
#pragma unroll
    for (int t = 0; t < 5; ++t)
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int col = colb * WG_T + tj * 4 + b;
        if (col < p.ncol) out[nw + (size_t)t * p.ncol + col] = sb[t][b];
      }
  }
}

#define BW_RED_SEG (BW_THREADS / 32)
__global__ void __launch_bounds__(BW_THREADS) iaf_bwd_reduce_kernel(const float* part, float* out, int n, int NG, int stride) {
  // One block per 32 outputs, one warp per SEGMENT of the NG split-K partials: warp w sums partials w, w + 8, w + 16, ...
  // (four interleaved chains, fixed order), then a fixed tree over the 8 segments.  Deterministic; NG / 32 dependent
  // round trips per thread instead of NG / 8 (C2a's 64x64 layers have NG = 296: 40 us -> a few us per layer).
  __shared__ float seg_sum[BW_RED_SEG][32];
  const int lane = threadIdx.x & 31, seg = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + lane;
  float s[4] = {0.f, 0.f, 0.f, 0.f};
  if (i < n) {
    int g = seg;
    for (; g + 3 * BW_RED_SEG < NG; g += 4 * BW_RED_SEG) {
#pragma unroll
      for (int k = 0; k < 4; ++k) s[k] += part[(size_t)(g + k * BW_RED_SEG) * stride + i];
    }
    for (int k = 0; g < NG; g += BW_RED_SEG, ++k) s[k] += part[(size_t)g * stride + i];
  }
  seg_sum[seg][lane] = (s[0] + s[1]) + (s[2] + s[3]);
  __syncthreads();
  if (seg == 0 && i < n) {
    float t[BW_RED_SEG];
#pragma unroll
    for (int k = 0; k < BW_RED_SEG; ++k) t[k] = seg_sum[k][lane];
    out[i] = ((t[0] + t[1]) + (t[2] + t[3])) + ((t[4] + t[5]) + (t[6] + t[7]));
  }
}

// ------------------------------------------------------------------------------------------
// Bias and pad-channel gradients of one layer when the weight gradient runs on the tensor cores (iaf_wg_kernel does the
// [5][cin][ncol] part only): out[t][col] = sum over samples and pixels of g * {1, [x = W-1], [y = H-1 or x = 0], [y = H-1],
// [y = H-1 or x = W-1]} -- the same five sums iaf_bwd_wgrad_kernel's `side` threads form.  One block per column, fixed order.
// ------------------------------------------------------------------------------------------
#define BW_BIAS_SEG 16
#ifndef IAF_EMU  // tensor-core path only (never taken under host emulation): warp shuffles
template <bool PADW>
__global__ void __launch_bounds__(BW_THREADS) iaf_bwd_bias_kernel(const float* g, float* bpart, int B, int planes, int ncol, int H,
                                                                  int W, int flip) {
  // block (column, batch segment): partial sums of its samples -> bpart[segment][5][ncol]; iaf_bwd_reduce_kernel adds the
  // segments.  Fixed order: per-thread strided sums, xor-shuffle tree inside a warp, the 8 warps in index order.
  // PADW = false (TF numerics): only the plain sum is needed, the pad-channel rows are written as zeros.
  constexpr int NS = PADW ? 5 : 1;
  __shared__ float red[BW_THREADS / 32][5];
  const int col = blockIdx.x % ncol, seg = blockIdx.x / ncol, tid = threadIdx.x, HW = H * W;
  const int n0 = (int)((long long)B * seg / BW_BIAS_SEG), n1 = (int)((long long)B * (seg + 1) / BW_BIAS_SEG);
  float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  const BwDiv dHW = bw_mkdiv(HW), dW = bw_mkdiv(W);
  const int total = (n1 - n0) * HW;
  for (int i0 = 0; i0 < total; i0 += 8 * BW_THREADS) {
    float v[8];
    int px[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {  // eight loads in flight per thread
      const int i = i0 + k * BW_THREADS + tid;
      v[k] = 0.f; px[k] = 0;
      if (i < total) {
        const int nl = bw_div(i, dHW), pix = i - nl * HW;
        px[k] = pix;
        v[k] = g[((size_t)(n0 + nl) * planes + col) * HW + (flip ? HW - 1 - pix : pix)];
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      s[0] += v[k];
      if (PADW) {
        const int y = bw_div(px[k], dW), x = px[k] - y * W;
        const bool byH = (y == H - 1), bx0 = (x == 0), bxW = (x == W - 1);
        s[1] += bxW ? v[k] : 0.f;
        s[2] += (byH || bx0) ? v[k] : 0.f;
        s[3] += byH ? v[k] : 0.f;
        s[4] += (byH || bxW) ? v[k] : 0.f;
      }
    }
  }
#pragma unroll
  for (int t = 0; t < NS; ++t)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[t] += __shfl_xor_sync(0xffffffffu, s[t], o);
  if ((tid & 31) == 0)
#pragma unroll
    for (int t = 0; t < 5; ++t) red[tid >> 5][t] = s[t];
  __syncthreads();
  if (tid < 5) {
    float r = 0.f;
    for (int w = 0; w < BW_THREADS / 32; ++w) r += red[w][tid];
    bpart[((size_t)seg * 5 + tid) * ncol + col] = r;
  }
}
#endif

// ------------------------------------------------------------------------------------------
// dW (packed) -> raw-parameter gradients through the mask and the weight normalisation.  One block per
// (output channel, layer), mirroring iaf_pack_kernel.
//   TF     (layers.py:53-60):  W = exp(g) * v / sqrt(max(ss, 1e-12)),   v = mask*V, ss = sum v^2
//   Theano (ar.py:267-281,312-317): W = exp(3s) * v / (sqrt(ss) + 1e-8)   (pad channel included in v)
// ------------------------------------------------------------------------------------------
struct IafWnormLayer {
  const float* w; const float* scale;  // raw parameters
  const float* dwp;                    // packed gradient: [5*cin*ncol] dW, [ncol] db, [4*ncol] dpadw
  float* g_w; float* g_scale; float* g_bias;
  int cin, cout, ncol, zerodiag, n_heads, head;  // n_heads == 0: hidden layer
};
struct IafWnormParams {
  IafWnormLayer layer[IAF_MAX_HIDDEN + IAF_MAX_HEADS];
  int n_layers, variant;
};

__device__ __forceinline__ bool bw_centre_visible(int ci, int co, int cin, int cout, int zd) {
  if (cout >= cin) {
    const int k = cout / cin, i = co / k;
    return zd ? (ci < i) : (ci <= i);
  }
  const int k = cin / cout;
  return zd ? (ci < co * k) : (ci < (co + 1) * k);
}
__device__ __forceinline__ size_t bw_raw_index(const IafWnormLayer& L, int variant, int ky, int kx, int ci, int co) {
  if (variant == IAF_VARIANT_TF) return ((size_t)(ky * 3 + kx) * L.cin + ci) * L.cout + co;
  return (((size_t)co * (L.cin + 1) + ci) * 3 + ky) * 3 + kx;
}
// live tap index of kernel position (ky,kx), or -1 (layers.py:134-141)
__device__ __forceinline__ int bw_tap_of(int ky, int kx) {
  if (ky == 1) return kx == 1 ? 0 : (kx == 2 ? 1 : -1);
  if (ky == 2) return 2 + kx;
  return -1;
}

__global__ void __launch_bounds__(128) iaf_bwd_wnorm_kernel(const __grid_constant__ IafWnormParams p) {
  const IafWnormLayer& L = p.layer[blockIdx.y];
  const int co = blockIdx.x;
  if (co >= L.cout) return;
  const int tid = threadIdx.x;
  const int col = L.n_heads ? bw_head_col(L.n_heads, L.head, co) : co;
  const int cin_all = L.cin + (p.variant == IAF_VARIANT_THEANO ? 1 : 0);
  const int n_ent = 9 * cin_all;
  const size_t nw = (size_t)IAF_NTAPS * L.cin * L.ncol;

  // pass 1: ss = sum v^2, dot = sum dW * v over the live entries of this output channel
  float ss = 0.f, dot = 0.f;
  for (int e = tid; e < n_ent; e += 128) {
    const int ci = e / 9, ky = (e % 9) / 3, kx = e % 3;
    const int t = bw_tap_of(ky, kx);
    if (t < 0) continue;
    float dv;
    if (ci < L.cin) {
      if (t == 0 && !bw_centre_visible(ci, co, L.cin, L.cout, L.zerodiag)) continue;
      dv = L.dwp[((size_t)t * L.cin + ci) * L.ncol + col];
    } else {
      if (t == 0) continue;  // pad channel: centre tap masked (ar.py:249-262)
      dv = L.dwp[nw + (size_t)t * L.ncol + col];
    }
    const float v = L.w[bw_raw_index(L, p.variant, ky, kx, ci, co)];
    ss = fmaf(v, v, ss);
    dot = fmaf(dv, v, dot);
  }
  __shared__ float r1[128];
  __shared__ float r2[128];
  r1[tid] = ss;
  r2[tid] = dot;
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1) {
    if (tid < s) { r1[tid] += r1[tid + s]; r2[tid] += r2[tid + s]; }
    __syncthreads();
  }
  ss = r1[0];
  dot = r2[0];

  float f, k;  // dV = f * dW - k * v
  if (p.variant == IAF_VARIANT_TF) {
    const float n2 = fmaxf(ss, 1e-12f);
    f = expf(L.scale[co]) / sqrtf(n2);
    k = ss > 1e-12f ? f * dot / n2 : 0.f;
    if (tid == 0 && L.g_scale) L.g_scale[co] = f * dot;          // dL/dg = sum dW * W
  } else {
    const float r = sqrtf(ss), nn = r + 1e-8f, E = expf(3.0f * L.scale[co]);
    f = E / nn;
    k = r > 0.f ? E * dot / (nn * nn * r) : 0.f;
    if (tid == 0 && L.g_scale) L.g_scale[co] = 3.0f * f * dot;   // logscale_scale = 3 (ar.py:316)
  }
  if (tid == 0 && L.g_bias) L.g_bias[co] = L.dwp[nw + col];
  if (!L.g_w) return;
  // pass 2: every raw entry of this output channel; masked entries get exactly zero
  for (int e = tid; e < n_ent; e += 128) {
    const int ci = e / 9, ky = (e % 9) / 3, kx = e % 3;
    const int t = bw_tap_of(ky, kx);
    const size_t ri = bw_raw_index(L, p.variant, ky, kx, ci, co);
    float out = 0.f;
    bool live = t >= 0;
    if (live && ci < L.cin && t == 0 && !bw_centre_visible(ci, co, L.cin, L.cout, L.zerodiag)) live = false;
    if (live && ci >= L.cin && t == 0) live = false;
    if (live) {
      const float dv = ci < L.cin ? L.dwp[((size_t)t * L.cin + ci) * L.ncol + col] : L.dwp[nw + (size_t)t * L.ncol + col];
      out = f * dv - k * L.w[ri];
    }
    L.g_w[ri] = out;
  }
}

// ------------------------------------------------------------------------------------------
// data-dependent initialisation (TF layers.py:38-51 with init_scale = 1, Theano ar.py:331-353): per-channel mean and
// population variance of one stage's pre-activation, the layer's new parameters, and its normalised output.  Values
// are fp32, accumulation is in double, reductions are fixed-order shared-memory trees (no shuffles, no float
// atomics): reruns are bit-identical.
// ------------------------------------------------------------------------------------------
#define IN_THREADS 256

// sum over the CTA in a fixed order; every thread gets the result
__device__ __forceinline__ double in_block_sum(double v, double* red) {
  const int tid = threadIdx.x;
  red[tid] = v;
  __syncthreads();
  for (int s = IN_THREADS / 2; s > 0; s >>= 1) {
    if (tid < s) red[tid] += red[tid + s];
    __syncthreads();
  }
  const double r = red[0];
  __syncthreads();  // red is reused by the next call
  return r;
}

struct IafInitStatsParams {
  const float* x;  // [B][planes][HW]
  double* part;    // [channel][nseg][3]: count, mean, sum of squared deviations of each segment
  int planes, HW, nseg;
  long long N;     // B * HW values per channel
};

// grid (nseg, channels): segment s of a channel's N values (sample-major), two passes over it (mean, then squared
// deviations from that mean) so a constant channel gives exactly zero
__global__ void __launch_bounds__(IN_THREADS) iaf_init_stats_kernel(const __grid_constant__ IafInitStatsParams p) {
  __shared__ double red[IN_THREADS];
  const int c = blockIdx.y, s = blockIdx.x, tid = threadIdx.x;
  const long long e0 = p.N * s / p.nseg, e1 = p.N * (s + 1) / p.nseg;
  const float* xc = p.x + (size_t)c * p.HW;
  const size_t bstride = (size_t)p.planes * p.HW;
  double acc = 0.0;
  for (long long e = e0 + tid; e < e1; e += IN_THREADS) {
    const long long b = e / p.HW;
    acc += (double)__ldg(xc + b * bstride + (e - b * p.HW));
  }
  const double n = (double)(e1 - e0);
  const double mean = n > 0.0 ? in_block_sum(acc, red) / n : 0.0;
  acc = 0.0;
  for (long long e = e0 + tid; e < e1; e += IN_THREADS) {
    const long long b = e / p.HW;
    const double d = (double)__ldg(xc + b * bstride + (e - b * p.HW)) - mean;
    acc += d * d;
  }
  const double m2 = in_block_sum(acc, red);
  if (tid == 0) {
    double* q = p.part + ((size_t)c * p.nseg + s) * 3;
    q[0] = n; q[1] = mean; q[2] = m2;
  }
}

struct IafInitLayer {
  const float* scale_in;  // Theano: kept by a skipped layer
  const float* bias_in;
  float* scale_out;
  float* bias_out;
  int cout, col0, pairs;  // column of channel co in the stage's output: pairs ? (co/4)*8 + col0 + co%4 : co (iaf_pack.cu)
};

struct IafInitFinalParams {
  IafInitLayer layer[IAF_MAX_HEADS];  // one CTA per layer of the stage: the heads stage has one per head
  const double* part;
  double* coef;                       // [column][2]: the apply kernel's map out = (x - coef[0]) * coef[1]
  int* skipped;                       // entry of the stage's first layer, or nullptr
  int nseg, variant;
};

__device__ __forceinline__ int in_col(const IafInitLayer& L, int co) { return L.pairs ? (co >> 2) * 8 + L.col0 + (co & 3) : co; }

__global__ void __launch_bounds__(IN_THREADS) iaf_init_finalize_kernel(const __grid_constant__ IafInitFinalParams p) {
  __shared__ double red[IN_THREADS];
  const IafInitLayer& L = p.layer[blockIdx.x];
  const int tid = threadIdx.x;
  const bool tf = p.variant == IAF_VARIANT_TF;
  double nzero = 0.0;
  for (int co = tid; co < L.cout; co += IN_THREADS) {
    const int col = in_col(L, co);
    // the segments' (count, mean, M2) merged in order (Chan, Golub & LeVeque's pairwise update)
    double n = 0.0, mean = 0.0, m2 = 0.0;
    for (int s = 0; s < p.nseg; ++s) {
      const double* q = p.part + ((size_t)col * p.nseg + s) * 3;
      if (q[0] == 0.0) continue;
      const double nn = n + q[0], dl = q[1] - mean;
      mean += dl * (q[0] / nn);
      m2 += q[2] + dl * dl * (n * q[0] / nn);
      n = nn;
    }
    const double var = m2 / n;  // population variance: tf.nn.moments, Theano std (ddof 0)
    if (!tf && var == 0.0) nzero += 1.0;
    p.coef[2 * col] = mean;
    p.coef[2 * col + 1] = 1.0 / sqrt(tf ? var + 1e-10 : var);  // layers.py:46 | ar.py:333 (inf when std = 0: skipped below)
  }
  // Theano: a layer with any zero-std channel keeps its parameters and returns h unchanged (ar.py:334-336)
  const double nzero_all = in_block_sum(nzero, red);
  const bool skip = nzero_all > 0.0;
  for (int co = tid; co < L.cout; co += IN_THREADS) {
    const int col = in_col(L, co);
    double* k = p.coef + 2 * col;
    if (skip) {
      L.scale_out[co] = L.scale_in[co];
      L.bias_out[co] = L.bias_in[co];
      k[0] = 0.0;
      k[1] = 1.0;
    } else {
      // TF: g = log(scale) / 3, b = -m * scale (layers.py:47-48); Theano: s = -log(std) / 3, b = -mean(h / std)
      // (ar.py:339,348-350)
      L.scale_out[co] = (float)(log(k[1]) / 3.0);
      L.bias_out[co] = (float)(-k[0] * k[1]);
    }
  }
  if (tid == 0 && p.skipped) p.skipped[blockIdx.x] = (int)nzero_all;
}

struct IafInitApplyParams {
  const float* pre;     // [B][planes][HW]: the stage's pre-activation
  const double* coef;
  const float* ctx;     // first hidden layer: [B][cout][HW], else nullptr
  float* out[IAF_MAX_HEADS];  // hidden stage: out[0] = the next stage's input; heads: one per head (nullptr: not wanted)
  int n_out, cout, pairs, planes, B, HW;
  int nl;               // hidden stage: the nonlinearity; heads: IAF_NL_NONE
};

// out = nl((pre - mean) / std (+ context)) on hidden layers (layers.py:161-166, ar.py:400-409); heads: no context, no nl
__global__ void __launch_bounds__(IN_THREADS) iaf_init_apply_kernel(const __grid_constant__ IafInitApplyParams p) {
  const size_t per = (size_t)p.B * p.cout * p.HW;
  const size_t total = per * p.n_out;
  for (size_t i = (size_t)blockIdx.x * IN_THREADS + threadIdx.x; i < total; i += (size_t)gridDim.x * IN_THREADS) {
    const int k = (int)(i / per);
    const size_t r = i - k * per;
    float* out = p.out[k];
    if (!out) continue;
    const int b = (int)(r / ((size_t)p.cout * p.HW));
    const size_t r2 = r - (size_t)b * p.cout * p.HW;
    const int co = (int)(r2 / p.HW), px = (int)(r2 - (size_t)co * p.HW);
    const int col = p.pairs ? (co >> 2) * 8 + 4 * k + (co & 3) : co;
    const float x = __ldg(p.pre + ((size_t)b * p.planes + col) * p.HW + px);
    float v = (float)(((double)x - p.coef[2 * col]) * p.coef[2 * col + 1]);
    if (p.ctx) v += __ldg(p.ctx + r);
    out[r] = bw_apply_nl(v, p.nl);
  }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int bw_round_up(int a, int b) { return (a + b - 1) / b * b; }

struct IafBwdPlan {
  iaf_desc_t d;
  int n_stages;
  int cin[IAF_MAX_STAGES], cout[IAF_MAX_STAGES], ncol[IAF_MAX_STAGES];
  int head_pad;
  // lconv geometry (shared by every layer: depends on H, W only, nctb per layer)
  int nseg, P;
  // scratch (grows with B)
  int scratch_B;
  float* h[IAF_MAX_STAGES];   // h[j] = input of stage j (j >= 1): [B][cout[j-1]][HW]
  float* hb;                  // heads raw / gradient: [B][ncol[last]][HW]
  float* z0; float* gz0;      // fused-layer mode: the posterior sample and its gradient, [B][n_z][HW] (allocated on first use)
  int z0_B;
  float* G[2];                // ping-pong gradient buffers of the hidden layers
  float* wT;                  // transposed weights of the current layer
  float* part;                // wgrad partials
  float* dwp[IAF_MAX_STAGES]; // reduced packed gradients per stage
  int NG[IAF_MAX_STAGES];      // weight-gradient CTAs per (ci block, column block) tile of each stage
  int num_sms;
  size_t wg_smem; int wg_RB;
  size_t lc_smem_max;
  IafDgPlan* dg;               // data gradient on the tensor cores (nullptr: exact-fp32 SIMT lconv kernels)
  int wg_tc;                   // weight gradient on the tensor cores too (IAF_BWD_WG_TC=0: the SIMT kernel)
  float* bpart;                // [BW_BIAS_SEG][5][max ncol]: bias / pad-channel partial sums of that path
  double* ini_part;            // data-dependent init: per-segment statistics [max ncol][nseg][3] (allocated on first use)
  size_t ini_part_n;
  double* ini_coef;            // [max ncol][2]
};

static void bw_free_scratch(IafBwdPlan* pl) {
  for (int j = 0; j < IAF_MAX_STAGES; ++j) {
    if (pl->h[j]) cudaFree(pl->h[j]);
    pl->h[j] = nullptr;
  }
  if (pl->hb) cudaFree(pl->hb);
  if (pl->z0) cudaFree(pl->z0);
  if (pl->gz0) cudaFree(pl->gz0);
  pl->z0 = pl->gz0 = nullptr; pl->z0_B = 0;
  if (pl->G[0]) cudaFree(pl->G[0]);
  if (pl->G[1]) cudaFree(pl->G[1]);
  if (pl->part) cudaFree(pl->part);
  pl->hb = pl->G[0] = pl->G[1] = pl->part = nullptr;
  pl->scratch_B = 0;
}

int iaf_bwd_plan_uses_tc(const IafBwdPlan* p) { return !p || !p->dg ? 0 : (p->wg_tc ? 2 : 1); }

int iaf_bwd_plan_create(IafBwdPlan** out, const iaf_desc_t* d, const int* cin, const int* cout, const int* cout_pad,
                        int head_pad, int allow_tc) {
  IafBwdPlan* pl = new (std::nothrow) IafBwdPlan();
  if (!pl) return IAF_ERR_BAD_ARG;
  memset(pl, 0, sizeof(*pl));
  pl->d = *d;
  pl->n_stages = d->n_hidden + 1;
  pl->head_pad = head_pad;
  size_t wt_max = 0;
  for (int j = 0; j < pl->n_stages; ++j) {
    pl->cin[j] = cin[j]; pl->cout[j] = cout[j]; pl->ncol[j] = cout_pad[j];
    const size_t n = (size_t)IAF_NTAPS * cin[j] * cout_pad[j] + 5 * (size_t)cout_pad[j];
    if (cudaMalloc(&pl->dwp[j], sizeof(float) * n) != cudaSuccess) { iaf_bwd_plan_destroy(pl); return IAF_ERR_CUDA; }
    wt_max = std::max(wt_max, (size_t)IAF_NTAPS * cout_pad[j] * bw_round_up(cin[j], 8));
  }
  if (cudaMalloc(&pl->wT, sizeof(float) * wt_max) != cudaSuccess) { iaf_bwd_plan_destroy(pl); return IAF_ERR_CUDA; }
  {
    int dev = 0;
    cudaDeviceProp prop;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaGetDeviceProperties(&prop, dev) != cudaSuccess) { iaf_bwd_plan_destroy(pl); return IAF_ERR_CUDA; }
    pl->num_sms = prop.multiProcessorCount;
  }
  pl->nseg = (d->W + BW_PX - 1) / BW_PX;
  pl->P = BW_PX * pl->nseg + 2;
  if (pl->nseg > BW_THREADS) { iaf_bwd_plan_destroy(pl); return IAF_ERR_UNSUPPORTED; }
  // wgrad band: the largest band of rows whose TWO staging buffers fit 100 KB (two CTAs per SM), at least one row within 200 KB
  const int PW = d->W + 2;
  int rb = 0;
  for (int r = d->H; r >= 1; --r) {
    const size_t s = 2 * sizeof(float) * WG_S * ((size_t)(r + 1) * PW + (size_t)r * d->W);
    if (s <= 100 * 1024 || (r == 1 && s <= 200 * 1024)) { rb = r; pl->wg_smem = s; break; }
  }
  if (!rb) { iaf_bwd_plan_destroy(pl); return IAF_ERR_UNSUPPORTED; }
  {  // even bands: the same number of bands, all (but possibly the last) of equal height (16 rows: 4 x 4, not 5+5+5+1)
    const int nb = (d->H + rb - 1) / rb;
    rb = (d->H + nb - 1) / nb;
    pl->wg_smem = 2 * sizeof(float) * WG_S * ((size_t)(rb + 1) * PW + (size_t)rb * d->W);
  }
  pl->wg_RB = rb;
  if (iaf_smem_optin(iaf_bwd_wgrad_kernel) != cudaSuccess || iaf_smem_optin(iaf_lconv_kernel<false>) != cudaSuccess ||
      iaf_smem_optin(iaf_lconv_kernel<true>) != cudaSuccess) {
    iaf_bwd_plan_destroy(pl);
    return IAF_ERR_CUDA;
  }
  // data gradient on the tensor cores when every layer fits the layered kernel's stage (channels in multiples of 16,
  // packed columns == the next layer's input channels); otherwise, and with IAF_BWD_TC=0, the SIMT kernels below
  pl->dg = nullptr;
  {
    bool ok = allow_tc != 0;
    for (int j = 0; j + 1 < pl->n_stages; ++j) ok = ok && pl->ncol[j] == pl->cin[j + 1];
    if (ok && iaf_dg_plan_create(&pl->dg, d, pl->cin, pl->ncol, pl->n_stages) != IAF_OK) pl->dg = nullptr;
    cudaGetLastError();
    const char* we = getenv("IAF_BWD_WG_TC");
    pl->wg_tc = (pl->dg && !(we && we[0] == '0')) ? 1 : 0;
    if (pl->wg_tc) {
      int mc = 0;
      for (int j = 0; j < pl->n_stages; ++j) mc = std::max(mc, pl->ncol[j]);
      if (cudaMalloc(&pl->bpart, sizeof(float) * BW_BIAS_SEG * 5 * mc) != cudaSuccess) { pl->bpart = nullptr; pl->wg_tc = 0; cudaGetLastError(); }
    }
  }
  *out = pl;
  return IAF_OK;
}

void iaf_bwd_plan_destroy(IafBwdPlan* pl) {
  if (!pl) return;
  if (pl->dg) iaf_dg_plan_destroy(pl->dg);
  if (pl->bpart) cudaFree(pl->bpart);
  if (pl->ini_part) cudaFree(pl->ini_part);
  if (pl->ini_coef) cudaFree(pl->ini_coef);
  bw_free_scratch(pl);
  for (int j = 0; j < IAF_MAX_STAGES; ++j)
    if (pl->dwp[j]) cudaFree(pl->dwp[j]);
  if (pl->wT) cudaFree(pl->wT);
  delete pl;
}

static int bw_ensure_scratch(IafBwdPlan* pl, int B) {
  if (B <= pl->scratch_B) return IAF_OK;
  bw_free_scratch(pl);
  const size_t hw = (size_t)pl->d.H * pl->d.W;
  int maxh = 0;
  for (int j = 1; j < pl->n_stages; ++j) {
    if (cudaMalloc(&pl->h[j], sizeof(float) * B * pl->cout[j - 1] * hw) != cudaSuccess) return IAF_ERR_CUDA;
    maxh = std::max(maxh, pl->cout[j - 1]);
  }
  const int last = pl->n_stages - 1;
  if (cudaMalloc(&pl->hb, sizeof(float) * B * pl->ncol[last] * hw) != cudaSuccess) return IAF_ERR_CUDA;
  for (int a = 0; a < 2 && maxh; ++a)
    if (cudaMalloc(&pl->G[a], sizeof(float) * B * maxh * hw) != cudaSuccess) return IAF_ERR_CUDA;
  // weight gradient: enough CTAs per tile to fill the machine twice over (the first version used a flat 32 and left
  // C2a's 64x64 layers on 32 of 148 SMs: 1.76 ms; measured after: see DESIGN.md), never more than there are units
  const int n_bands = (pl->d.H + pl->wg_RB - 1) / pl->wg_RB;
  size_t pmax = 0;
  for (int j = 0; j < pl->n_stages; ++j) {
    const int tiles = ((pl->cin[j] + WG_T - 1) / WG_T) * ((pl->ncol[j] + WG_T - 1) / WG_T);
    pl->NG[j] = std::max(1, std::min(std::min(B * n_bands, 512), (2 * pl->num_sms + tiles - 1) / tiles));
    pmax = std::max(pmax, ((size_t)IAF_NTAPS * pl->cin[j] * pl->ncol[j] + 5 * (size_t)pl->ncol[j]) * pl->NG[j]);
  }
  if (cudaMalloc(&pl->part, sizeof(float) * pmax) != cudaSuccess) return IAF_ERR_CUDA;
  pl->scratch_B = B;
  return IAF_OK;
}

// geometry of one lconv launch for `ncol` weight columns
static void bw_lconv_geom(const IafBwdPlan* pl, IafLconvParams* q, size_t* smem) {
  const int H = pl->d.H;
  q->nseg = pl->nseg; q->P = pl->P;
  const int nct = q->ncol / BW_CT;
  int nctb = std::min(nct, 8);
  while (q->nseg * nctb > BW_THREADS) nctb /= 2;
  q->nctb = nctb;
  q->n_cblk = (nct + nctb - 1) / nctb;
  q->RB = std::max(1, std::min(H, BW_THREADS / (q->nseg * nctb)));
  q->n_bands = (H + q->RB - 1) / q->RB;
  // per staged input channel: one activation plane and 5 x (column block) weights; up to ~80 KB so that two CTAs fit an SM
  const size_t per_c = sizeof(float) * ((size_t)(q->RB + 1) * q->P + (size_t)IAF_NTAPS * nctb * BW_CT);
  int ck = (int)std::min<size_t>(32, (80 * 1024) / per_c);
  q->CK = std::max(1, ck);
  // keep the weight region 16-byte aligned: CK * plane floats must be a multiple of 4
  while (q->CK > 1 && ((size_t)q->CK * (q->RB + 1) * q->P) % 4 != 0) --q->CK;
  *smem = std::max(per_c * q->CK, sizeof(float) * (size_t)q->RB * pl->d.W * (nctb * BW_CT + 4));  // staging | output tile
}

static int bw_lconv(const IafBwdPlan* pl, IafLconvParams& q, cudaStream_t stream) {
  size_t smem = 0;
  bw_lconv_geom(pl, &q, &smem);
  if (smem > 100 * 1024 || ((size_t)q.CK * (q.RB + 1) * q.P) % 4 != 0) return IAF_ERR_UNSUPPORTED;
  const int grid = q.B * q.n_bands * q.n_cblk;
  if (q.bwd) IAF_LAUNCH(iaf_lconv_kernel<true>, grid, BW_THREADS, smem, stream, q);
  else IAF_LAUNCH(iaf_lconv_kernel<false>, grid, BW_THREADS, smem, stream, q);
  return cudaGetLastError() == cudaSuccess ? IAF_OK : IAF_ERR_CUDA;
}

int iaf_bwd_run(IafBwdPlan* pl, const IafBwdArgs* a, cudaStream_t stream, int* n_launches) {
  const iaf_desc_t& d = pl->d;
  const int B = a->B, H = d.H, W = d.W, HW = H * W;
  const int nst = pl->n_stages, last = nst - 1;
  const int flip = d.variant == IAF_VARIANT_THEANO ? 1 : 0;
  int st = bw_ensure_scratch(pl, B);
  if (st != IAF_OK) return st;
  int nl_ = 0;
  // elementwise kernels: grid-stride, at most 4 CTAs per SM on 148 SMs
  auto ew_grid = [](size_t total) { return (int)std::min<size_t>(592, (total + BW_THREADS - 1) / BW_THREADS); };

  // activations: recomputed below, or the ones the training forward kept
  const bool saved = a->have_saved != 0;  // step: z', arw_logsd and the hidden activations; multiconv: the hidden activations
  const float* hcur[IAF_MAX_STAGES];
  for (int j = 1; j < nst; ++j) hcur[j] = saved ? a->h_saved[j - 1] : pl->h[j];
  hcur[0] = a->z;

  // fused-layer mode: the stack's input is the posterior sample z0 = post_mean + exp(post_logsd) * eps (a->z is eps), and
  // the gradient of z0 is a workspace from which the gradients of the posterior statistics are formed at the end
  const bool layer = a->mode == IAF_MODE_LAYER;
  float* g_zin = a->g_z;
  IafLayerBwdParams lq;
  memset(&lq, 0, sizeof(lq));
  if (layer) {
    if (B > pl->z0_B) {
      if (pl->z0) cudaFree(pl->z0);
      if (pl->gz0) cudaFree(pl->gz0);
      pl->z0 = pl->gz0 = nullptr; pl->z0_B = 0;
      if (cudaMalloc(&pl->z0, sizeof(float) * B * d.n_z * HW) != cudaSuccess ||
          cudaMalloc(&pl->gz0, sizeof(float) * B * d.n_z * HW) != cudaSuccess) return IAF_ERR_CUDA;
      pl->z0_B = B;
    }
    lq.eps = a->z; lq.post_mean = a->post_mean; lq.post_logsd = a->post_logsd;
    lq.prior_mean = a->prior_mean; lq.prior_logsd = a->prior_logsd;
    lq.g_zout = a->g_zout; lq.g_kl = a->g_kl; lq.g_kl_bc = a->g_kl_bc; lq.g_kl_cost = a->g_kl_cost;
    lq.z0 = pl->z0; lq.hb = pl->hb; lq.g_z0 = pl->gz0;
    lq.g_post_mean = a->g_post_mean; lq.g_post_logsd = a->g_post_logsd;
    lq.g_prior_mean = a->g_prior_mean; lq.g_prior_logsd = a->g_prior_logsd; lq.g_eps = a->g_eps;
    lq.B = B; lq.C = d.n_z; lq.HW = HW; lq.cp = pl->ncol[last]; lq.head_pad = pl->head_pad; lq.scale = 0.1f;
    IAF_LAUNCH(iaf_bwd_layer_pre_kernel, ew_grid((size_t)B * d.n_z * HW), BW_THREADS, 0, stream, lq);
    if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
    ++nl_;
    hcur[0] = pl->z0;
    g_zin = pl->gz0;
  }

  // ---- 1. forward recompute, layer at a time ----
  for (int j = 0; j < nst && !saved; ++j) {
    IafLconvParams q;
    memset(&q, 0, sizeof(q));
    q.in = hcur[j];
    q.w = a->w_packed[j]; q.bias = a->bias_packed[j];
    q.padw = flip ? a->padw_packed[j] : nullptr;
    q.ctx = (j == 0 && j != last) ? a->ctx : nullptr;
    q.out = j == last ? pl->hb : pl->h[j + 1];
    q.B = B; q.H = H; q.W = W; q.cin = pl->cin[j]; q.in_planes = pl->cin[j];
    q.ncol = pl->ncol[j];
    q.nout = j == last ? pl->ncol[j] : pl->cout[j];
    q.out_planes = j == last ? pl->ncol[j] : pl->cout[j];
    q.bwd = 0; q.epi = j == last ? EPI_FWD_HEADS : EPI_FWD_HIDDEN; q.nl = d.nl; q.flip = flip;
    if ((st = bw_lconv(pl, q, stream)) != IAF_OK) return st;
    ++nl_;
  }

  // ---- 2. gradient at the heads ----
  const bool fused_step = pl->dg && pl->wg_tc && a->mode == IAF_MODE_STEP && saved && iaf_dg_step_supported(pl->dg);
  const float* step_bias = nullptr;
  if (layer) {
    IAF_LAUNCH(iaf_bwd_layer_affine_kernel, ew_grid((size_t)B * pl->head_pad * HW), BW_THREADS, 0, stream, lq);
  } else if (a->mode == IAF_MODE_STEP && fused_step) {
    // tensor-core backward with kept activations: affine backward, per-sample scale, heads' bias sums and gradient image in
    // one launch (iaf_dg_step_kernel); the fp32 heads gradient is not needed by anything downstream
    if ((st = iaf_dg_begin_step(pl->dg, a->z_out_saved, a->logsd_saved, a->g_zout, a->g_logsd, a->g_logdet, a->g_z, nullptr,
                                pl->head_pad, B, stream, &step_bias)) != IAF_OK)
      return st;
  } else if (a->mode == IAF_MODE_STEP) {
    IafAffineBwdParams q;
    memset(&q, 0, sizeof(q));
    q.z = a->z; q.g_zout = a->g_zout; q.g_logsd = a->g_logsd; q.g_logdet = a->g_logdet;
    q.z_out = saved ? a->z_out_saved : nullptr; q.logsd = saved ? a->logsd_saved : nullptr;
    q.hb = pl->hb; q.g_z = a->g_z;
    q.B = B; q.C = d.n_z; q.HW = HW; q.cp = pl->ncol[last]; q.head_pad = pl->head_pad; q.scale = 0.1f;
    IAF_LAUNCH(iaf_bwd_affine_kernel, ew_grid((size_t)B * pl->head_pad * HW), BW_THREADS, 0, stream, q);
  } else {
    IafScatterParams q;
    memset(&q, 0, sizeof(q));
    q.g0 = a->g_heads[0]; q.g1 = d.n_heads == 2 ? a->g_heads[1] : nullptr;
    q.hb = pl->hb; q.g_z = a->g_z;
    q.B = B; q.C = d.head[0]; q.HW = HW; q.cp = pl->ncol[last]; q.head_pad = pl->head_pad; q.n_heads = d.n_heads;
    q.n_z = d.n_z;
    IAF_LAUNCH(iaf_bwd_scatter_kernel, ew_grid((size_t)B * std::max(pl->ncol[last], d.n_z) * HW), BW_THREADS, 0, stream, q);
  }
  if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
  ++nl_;

  // ---- 3. layers, top down ----
  const bool want_params = a->g_w || a->g_scale || a->g_bias;
  const float* Gcur = pl->hb;
  int g_planes = pl->ncol[last];
  for (int j = last; j >= 0; --j) {
    const float* xin = hcur[j];
    if (pl->dg && j == last && !fused_step) {
      if ((st = iaf_dg_begin(pl->dg, Gcur, B, stream)) != IAF_OK) return st;
      ++nl_;
    }
    if (want_params && pl->dg && pl->wg_tc) {
      // tensor cores: X^T G per tap over the slot stream as K (iaf_wg.cuh); bias / pad-channel sums separately
      const int nw = IAF_NTAPS * pl->cin[j] * pl->ncol[j];
      const int n = nw + 5 * pl->ncol[j];
      int ng = 1;
      if ((st = iaf_wg_run(pl->dg, j, xin, (last - j) & 1, pl->part, n, pl->NG[j], B, stream, &ng)) != IAF_OK) return st;
      IAF_LAUNCH(iaf_bwd_reduce_kernel, (nw + 31) / 32, BW_THREADS, 0, stream, (const float*)pl->part, pl->dwp[j], nw, ng, n);
      if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
      if (fused_step && j == last) {  // the prologue left per-sample sums: [B][5][ncol]
        IAF_LAUNCH(iaf_bwd_reduce_kernel, (5 * pl->ncol[j] + 31) / 32, BW_THREADS, 0, stream, step_bias, pl->dwp[j] + nw,
                   5 * pl->ncol[j], B, 5 * pl->ncol[j]);
        if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
        nl_ += 4;
      } else {
#ifndef IAF_EMU
        if (flip) iaf_bwd_bias_kernel<true><<<pl->ncol[j] * BW_BIAS_SEG, BW_THREADS, 0, stream>>>(Gcur, pl->bpart, B, g_planes, pl->ncol[j], H, W, flip);
        else iaf_bwd_bias_kernel<false><<<pl->ncol[j] * BW_BIAS_SEG, BW_THREADS, 0, stream>>>(Gcur, pl->bpart, B, g_planes, pl->ncol[j], H, W, flip);
#endif
        if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
        IAF_LAUNCH(iaf_bwd_reduce_kernel, (5 * pl->ncol[j] + 31) / 32, BW_THREADS, 0, stream, (const float*)pl->bpart,
                   pl->dwp[j] + nw, 5 * pl->ncol[j], BW_BIAS_SEG, 5 * pl->ncol[j]);
        if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
        nl_ += 5;
      }
    } else if (want_params) {
      IafWgradParams q;
      memset(&q, 0, sizeof(q));
      q.x = xin; q.g = Gcur; q.part = pl->part;
      q.B = B; q.H = H; q.W = W; q.cin = pl->cin[j]; q.x_planes = pl->cin[j]; q.ncol = pl->ncol[j]; q.g_planes = g_planes;
      q.flip = flip; q.RB = pl->wg_RB; q.n_bands = (H + pl->wg_RB - 1) / pl->wg_RB; q.NG = pl->NG[j];
      q.n_cib = (pl->cin[j] + WG_T - 1) / WG_T; q.n_colb = (pl->ncol[j] + WG_T - 1) / WG_T; q.PW = W + 2;
      IAF_LAUNCH(iaf_bwd_wgrad_kernel, q.n_cib * q.n_colb * q.NG, BW_THREADS, pl->wg_smem, stream, q);
      if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
      const int n = IAF_NTAPS * pl->cin[j] * pl->ncol[j] + 5 * pl->ncol[j];
      IAF_LAUNCH(iaf_bwd_reduce_kernel, (n + 31) / 32, BW_THREADS, 0, stream,
                 (const float*)pl->part, pl->dwp[j], n, pl->NG[j], n);
      if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
      nl_ += 2;
    }
    // data gradient
    if (pl->dg) {
      // tensor cores: the layered kernel's hidden stage on the point-reflected stream with transposed weights (iaf_tc.cu)
      float* Gnext = nullptr;
      float* outp = g_zin;
      if (j > 0) {
        Gnext = (j == 1 && a->g_ctx) ? a->g_ctx : pl->G[j & 1];  // the gradient at a_0 IS the context gradient
        outp = Gnext;
      }
      if ((st = iaf_dg_stage(pl->dg, j, a->w_packed[j], (last - j) & 1, j > 0 ? hcur[j] : nullptr, outp, j > 0 ? 1 : 0, B,
                             stream)) != IAF_OK)
        return st;
      nl_ += 2;
      Gcur = Gnext;
      g_planes = pl->cin[j];
      continue;
    }
    const int cin_pad = bw_round_up(pl->cin[j], 8);
    {
      const int total = IAF_NTAPS * g_planes * cin_pad;
      IAF_LAUNCH(iaf_bwd_transpose_kernel, ew_grid((size_t)total), BW_THREADS, 0, stream,
                 a->w_packed[j], pl->wT, pl->cin[j], pl->ncol[j], g_planes, cin_pad);
      if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
      ++nl_;
    }
    IafLconvParams q;
    memset(&q, 0, sizeof(q));
    q.in = Gcur; q.w = pl->wT;
    q.B = B; q.H = H; q.W = W; q.cin = g_planes; q.in_planes = g_planes;
    q.ncol = cin_pad; q.nout = pl->cin[j]; q.out_planes = pl->cin[j];
    q.bwd = 1; q.nl = d.nl; q.flip = flip;
    float* Gnext = nullptr;
    if (j == 0) {
      q.epi = EPI_BWD_Z; q.out = g_zin;
    } else {
      q.epi = EPI_BWD_HIDDEN; q.hprev = hcur[j];
      Gnext = (j == 1 && a->g_ctx) ? a->g_ctx : pl->G[j & 1];  // the gradient at a_0 IS the context gradient
      q.out = Gnext;
    }
    if ((st = bw_lconv(pl, q, stream)) != IAF_OK) return st;
    ++nl_;
    Gcur = Gnext;
    g_planes = pl->cin[j];
  }

  if (layer) {
    IAF_LAUNCH(iaf_bwd_layer_post_kernel, ew_grid((size_t)B * d.n_z * HW), BW_THREADS, 0, stream, lq);
    if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
    ++nl_;
  }

  // ---- 4. raw-parameter gradients ----
  if (want_params) {
    IafWnormParams q;
    memset(&q, 0, sizeof(q));
    q.n_layers = d.n_hidden + d.n_heads;
    q.variant = d.variant;
    int max_cout = 0;
    for (int i = 0; i < q.n_layers; ++i) {
      IafWnormLayer& L = q.layer[i];
      const bool is_head = i >= d.n_hidden;
      const int j = is_head ? d.n_hidden : i;
      L.w = a->w_raw[i]; L.scale = a->scale_raw[i];
      L.dwp = pl->dwp[j];
      L.g_w = a->g_w ? a->g_w[i] : nullptr;
      L.g_scale = a->g_scale ? a->g_scale[i] : nullptr;
      L.g_bias = a->g_bias ? a->g_bias[i] : nullptr;
      L.cin = pl->cin[j];
      L.cout = is_head ? d.head[i - d.n_hidden] : d.hidden[i];
      L.ncol = pl->ncol[j];
      L.zerodiag = is_head ? 1 : 0;
      L.n_heads = is_head ? d.n_heads : 0;
      L.head = is_head ? i - d.n_hidden : 0;
      max_cout = std::max(max_cout, L.cout);
    }
    IAF_LAUNCH(iaf_bwd_wnorm_kernel, dim3(max_cout, q.n_layers), 128, 0, stream, q);
    if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
    ++nl_;
  }
  if (n_launches) *n_launches = nl_;
  return IAF_OK;
}

// Data-dependent initialisation, one stage at a time: conv (pre-activation epilogue), statistics, parameters, output.
// It runs on these exact-fp32 kernels for every plan, tensor-core plans included: it runs once per training run, on one
// batch, and its statistics become the model's parameters.
int iaf_init_run(IafBwdPlan* pl, const IafInitArgs* a, cudaStream_t stream, int* n_launches) {
  const iaf_desc_t& d = pl->d;
  const int B = a->B, HW = d.H * d.W;
  const int nst = pl->n_stages, last = nst - 1;
  const int flip = d.variant == IAF_VARIANT_THEANO ? 1 : 0;
  int st = bw_ensure_scratch(pl, B);
  if (st != IAF_OK) return st;
  // statistics segments of about 4096 values, at most 64 per channel (a function of the shape only: the merge order,
  // and so every bit of the result, is the same on every run)
  const long long N = (long long)B * HW;
  const int nseg = (int)std::min<long long>(64, std::max<long long>(1, N / 4096));
  int maxcol = 0;
  for (int j = 0; j < nst; ++j) maxcol = std::max(maxcol, pl->ncol[j]);
  const size_t npart = (size_t)maxcol * nseg * 3;
  if (npart > pl->ini_part_n) {
    if (pl->ini_part) cudaFree(pl->ini_part);
    pl->ini_part = nullptr;
    pl->ini_part_n = 0;
    if (cudaMalloc(&pl->ini_part, sizeof(double) * npart) != cudaSuccess) return IAF_ERR_CUDA;
    pl->ini_part_n = npart;
  }
  if (!pl->ini_coef && cudaMalloc(&pl->ini_coef, sizeof(double) * 2 * maxcol) != cudaSuccess) {
    pl->ini_coef = nullptr;
    return IAF_ERR_CUDA;
  }
  int nl_ = 0;
  const float* xin = a->z;
  for (int j = 0; j < nst; ++j) {
    const bool heads = j == last;
    const int planes = heads ? pl->ncol[j] : pl->cout[j];  // heads keep the packed (interleaved) column order
    float* pre = heads ? pl->hb : pl->G[0];
    {  // the heads' epilogue writes the pre-activation: bias and pad channel, no context, no nl
      IafLconvParams q;
      memset(&q, 0, sizeof(q));
      q.in = xin;
      q.w = a->w_packed[j]; q.bias = a->bias_packed[j];
      q.padw = flip ? a->padw_packed[j] : nullptr;
      q.out = pre;
      q.B = B; q.H = d.H; q.W = d.W; q.cin = pl->cin[j]; q.in_planes = pl->cin[j];
      q.ncol = pl->ncol[j]; q.nout = planes; q.out_planes = planes;
      q.bwd = 0; q.epi = EPI_FWD_HEADS; q.nl = d.nl; q.flip = flip;
      if ((st = bw_lconv(pl, q, stream)) != IAF_OK) return st;
    }
    IafInitStatsParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.x = pre; sp.part = pl->ini_part; sp.planes = planes; sp.HW = HW; sp.nseg = nseg; sp.N = N;
    IAF_LAUNCH(iaf_init_stats_kernel, dim3(nseg, planes), IN_THREADS, 0, stream, sp);
    if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;

    const int nlay = heads ? d.n_heads : 1;
    const int i0 = heads ? d.n_hidden : j;  // index of the stage's first layer in the parameter arrays
    IafInitFinalParams fp;
    memset(&fp, 0, sizeof(fp));
    for (int k = 0; k < nlay; ++k) {
      IafInitLayer& L = fp.layer[k];
      L.scale_in = flip ? a->scale_in[i0 + k] : nullptr;
      L.bias_in = flip ? a->bias_in[i0 + k] : nullptr;
      L.scale_out = a->scale_out[i0 + k];
      L.bias_out = a->bias_out[i0 + k];
      L.cout = heads ? d.head[k] : d.hidden[j];
      L.pairs = heads && d.n_heads == 2;
      L.col0 = 4 * k;
    }
    fp.part = pl->ini_part; fp.coef = pl->ini_coef;
    fp.skipped = a->skipped ? a->skipped + i0 : nullptr;
    fp.nseg = nseg; fp.variant = d.variant;
    IAF_LAUNCH(iaf_init_finalize_kernel, nlay, IN_THREADS, 0, stream, fp);
    if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
    nl_ += 3;

    if (heads && !a->outs) break;
    IafInitApplyParams ap;
    memset(&ap, 0, sizeof(ap));
    ap.pre = pre; ap.coef = pl->ini_coef;
    ap.planes = planes; ap.B = B; ap.HW = HW;
    if (heads) {
      for (int k = 0; k < d.n_heads; ++k) ap.out[k] = a->outs[k];
      ap.n_out = d.n_heads; ap.cout = d.head[0]; ap.pairs = d.n_heads == 2; ap.nl = IAF_NL_NONE;
    } else {
      ap.ctx = j == 0 ? a->ctx : nullptr;
      ap.out[0] = pl->h[j + 1];
      ap.n_out = 1; ap.cout = d.hidden[j]; ap.nl = d.nl;
    }
    const size_t total = (size_t)ap.n_out * B * ap.cout * HW;
    IAF_LAUNCH(iaf_init_apply_kernel, (int)std::min<size_t>(592, (total + IN_THREADS - 1) / IN_THREADS), IN_THREADS, 0,
               stream, ap);
    if (cudaGetLastError() != cudaSuccess) return IAF_ERR_CUDA;
    ++nl_;
    xin = pl->h[j + 1];
  }
  if (n_launches) *n_launches = nl_;
  return IAF_OK;
}
