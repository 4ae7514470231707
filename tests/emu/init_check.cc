// Sanitizer pass over the data-dependent initialisation kernels (TEST INFRASTRUCTURE ONLY): iaf_multiconv_init under
// the host emulation of CUDA.  Built and run by tests/test_data_init.py::test_init_kernels_under_sanitizers:
//   g++ -std=c++20 -O1 -g -fsanitize=thread|address,undefined -DIAF_EMU -I tests/emu -I iaf_b200/csrc -x c++ <sources> init_check.cc
// Runs weight packing, the layer conv with the pre-activation epilogue, the statistics, finalize and apply kernels on a
// Theano stack with a skipped head (pad channel, flip), a TF stack large enough for several statistics segments, and
// a Theano stack without hidden layers; then checks that the plan refuses a forward until it is packed again.
#include <cstdio>
#include <vector>

#include "../../include/iaf_b200.h"

static std::vector<float> rnd(size_t n, float s, unsigned seed) {
  std::vector<float> v(n);
  unsigned x = seed * 2654435761u + 12345u;
  for (auto& e : v) {
    x = x * 1664525u + 1013904223u;
    e = s * ((float)((x >> 8) & 0xFFFF) / 32768.0f - 1.0f);
  }
  return v;
}

static int run(int variant, int n_z, int n_hidden, int nh, int H, int W, int B, bool zero_head_channel) {
  iaf_desc_t d = {};
  d.variant = variant; d.n_z = n_z; d.n_hidden = n_hidden; d.hidden[0] = nh; d.n_heads = 2; d.head[0] = d.head[1] = n_z;
  d.H = H; d.W = W; d.nl = IAF_NL_ELU; d.path = IAF_PATH_SIMT;
  iaf_plan_t* pl = nullptr;
  if (iaf_plan_create(&pl, &d) != IAF_OK) return 1;
  const int n = n_hidden + 2;
  std::vector<int> cin(n), cout(n);
  for (int i = 0; i < n; ++i) {
    cin[i] = i == 0 ? n_z : (n_hidden ? nh : n_z);
    cout[i] = i < n_hidden ? nh : n_z;
  }
  std::vector<std::vector<float>> w(n), s(n), b(n), so(n), bo(n);
  std::vector<const float*> wp(n), sp(n), bp(n);
  std::vector<float*> sop(n), bop(n);
  for (int i = 0; i < n; ++i) {
    const size_t nw = variant == IAF_VARIANT_TF ? (size_t)9 * cin[i] * cout[i] : (size_t)cout[i] * (cin[i] + 1) * 9;
    w[i] = rnd(nw, 0.05f, 10 + i); s[i] = rnd(cout[i], 0.3f, 20 + i); b[i] = rnd(cout[i], 0.1f, 30 + i);
    so[i].assign(cout[i], 0.f); bo[i].assign(cout[i], 0.f);
    wp[i] = w[i].data(); sp[i] = s[i].data(); bp[i] = b[i].data(); sop[i] = so[i].data(); bop[i] = bo[i].data();
  }
  if (zero_head_channel)  // Theano layout [Cout][Cin+1][3][3]: channel 1 of the last head becomes the constant b[1]
    for (size_t e = 0; e < (size_t)(cin[n - 1] + 1) * 9; ++e) w[n - 1][(size_t)1 * (cin[n - 1] + 1) * 9 + e] = 0.f;
  const size_t nzv = (size_t)B * n_z * H * W, ncv = (size_t)B * (n_hidden ? nh : 1) * H * W;
  auto z = rnd(nzv, 1.f, 1), ctx = rnd(ncv, 0.1f, 2);
  std::vector<float> o0(nzv), o1(nzv);
  float* outs[2] = {o0.data(), o1.data()};
  std::vector<int> skipped(n, -1);
  if (iaf_multiconv_init(pl, z.data(), ctx.data(), wp.data(), sp.data(), bp.data(), sop.data(), bop.data(), outs,
                         skipped.data(), B, nullptr) != IAF_OK) return 2;
  if (zero_head_channel && skipped[n - 1] != 1) return 3;
  if (iaf_multiconv_fwd(pl, z.data(), ctx.data(), outs, B, nullptr) != IAF_ERR_NOT_PACKED) return 4;
  if (iaf_pack_weights(pl, wp.data(), sop.data(), bop.data(), nullptr) != IAF_OK) return 5;
  if (iaf_multiconv_fwd(pl, z.data(), ctx.data(), outs, B, nullptr) != IAF_OK) return 6;
  iaf_plan_destroy(pl);
  return 0;
}

int main() {
  int rc = run(IAF_VARIANT_THEANO, 4, 1, 8, 5, 9, 3, true);
  if (rc) { printf("theano run failed at step %d\n", rc); return rc; }
  rc = run(IAF_VARIANT_TF, 4, 1, 8, 8, 8, 128, false);  // 8192 values per channel: two statistics segments
  if (rc) { printf("tf run failed at step %d\n", rc); return 10 + rc; }
  rc = run(IAF_VARIANT_THEANO, 4, 0, 0, 4, 4, 2, false);
  if (rc) { printf("depth-0 run failed at step %d\n", rc); return 20 + rc; }
  printf("init_check ok\n");
  return 0;
}
